// compound.cu - path 2, compound heatwaves: the percentile x definition sweep over the days on which TWO measures of one grid (e.g.
// tmax and tmin: hot days and hot nights) both exceed their own thresholds (the contract is stated in include/hdp_b200.h).
//
//   k_hot_pair   the hot-word kernel of the compound pass.  It reads the word plan of k_hot_words (metric.cu) and writes the same
//                u32 [P, K, C] word planes, so k_scan and k_intensity run on them unchanged.  A CTA owns 32 cells, one 32-day
//                day-of-year block and one slice of whole percentile groups (gridDim.z): it keeps BOTH measures' threshold tiles
//                in shared memory, each rounded as k_hot_words rounds its own (down for heat, up for cold), puts the samples of
//                both measures in flight and sets a day's bit only where both compare true (setp + setp.and: one predicated OR per
//                day and percentile).  Each sample, threshold and output word crosses HBM once; when the two tiles of all
//                percentiles do not fit one CTA's shared memory (P 32) the slices re-read the samples.
#include <algorithm>

#include "metric.cuh"

namespace hdp {

constexpr int kPairDays = 8;                // days of each of kHotYears words whose samples (of both measures) are in flight together
constexpr size_t kPairSmemMax = 227 * 1024; // shared memory of one CTA on sm_100

// m |= bit where va > ta and vb > tb (false when any side is NaN)
__device__ __forceinline__ void or_if_both_gt(uint32_t &m, float va, float ta, float vb, float tb, uint32_t bit)
{
    asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, %2;\n\tsetp.gt.and.f32 p, %3, %4, p;\n\t@p or.b32 %0, %0, %5;\n\t}"
        : "+r"(m) : "f"(va), "f"(ta), "f"(vb), "f"(tb), "r"(bit));
}

// the same with va < ta and vb < tb: cold days and cold nights
__device__ __forceinline__ void or_if_both_lt(uint32_t &m, float va, float ta, float vb, float tb, uint32_t bit)
{
    asm("{\n\t.reg .pred p;\n\tsetp.lt.f32 p, %1, %2;\n\tsetp.lt.and.f32 p, %3, %4, p;\n\t@p or.b32 %0, %0, %5;\n\t}"
        : "+r"(m) : "f"(va), "f"(ta), "f"(vb), "f"(tb), "r"(bit));
}

// One threshold tile: percentile groups [g0, g0 + n_g) of 32 cells x nd days of year from thr [C, n_doy, P] into
// tile [n_g][32 doy][PG][kTilePad], rounded as k_hot_words rounds (see there); what it leaves alone holds the padding.
template <int PG, bool COLD>
__device__ __forceinline__ void fill_pair_tile(float *tile, const double *__restrict__ thr, int64_t C, int64_t c0, int n_doy, int db, int nd,
                                               int P, int g0, int n_g)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_el = nd * P;
    const float inv_p = 1.0f / (float)P;                   // exact enough: see k_hot_words
    for (int e0 = 0; e0 < n_el; e0 += 32 * kFillLoads) {
        int dst[kFillLoads];
#pragma unroll
        for (int i = 0; i < kFillLoads; i++) {
            const int e = e0 + 32 * i + lane;
            const int j = __float2int_rz(((float)e + 0.5f) * inv_p), p = e - j * P, g = p / PG - g0, q = p - (g + g0) * PG;
            dst[i] = e < n_el && g >= 0 && g < n_g ? ((g * kTileDoy + j) * PG + q) * kTilePad : -1;
        }
        for (int cell = warp; cell < kTileCells; cell += 8) {
            if (c0 + cell >= C) break;
            const double *src = thr + ((c0 + cell) * n_doy + (int64_t)db * kTileDoy) * P + e0 + lane;
            double v[kFillLoads];
#pragma unroll
            for (int i = 0; i < kFillLoads; i++) v[i] = dst[i] >= 0 ? __ldg(src + 32 * i) : 0.0;
#pragma unroll
            for (int i = 0; i < kFillLoads; i++)
                if (dst[i] >= 0) tile[dst[i] + cell] = COLD ? __double2float_ru(v[i]) : __double2float_rd(v[i]);
        }
    }
}

// kPairDays days (from J0 on) of kHotYears words of both measures against one percentile group of both tiles
template <int PG, int J0, int UNIT, bool COLD>
__device__ __forceinline__ void pair_days(uint32_t (&m)[kHotYears][PG], const float *const (&xa)[kHotYears], const float *const (&xb)[kHotYears],
                                          const int (&jo)[kHotYears], const int (&nb)[kHotYears], int64_t ld_a, int64_t ld_b,
                                          const float *ta, const float *tb)
{
    float va[kHotYears][kPairDays], vb[kHotYears][kPairDays];
#pragma unroll
    for (int y = 0; y < kHotYears; y++)
#pragma unroll
        for (int j = 0; j < kPairDays; j++) {              // NaN = never hot: days outside the word
            const bool in = (unsigned)(J0 + j - jo[y]) < (unsigned)nb[y];
            va[y][j] = in ? __ldg(xa[y] + (int64_t)(J0 + j) * ld_a) : __int_as_float(0x7fc00000);
            vb[y][j] = in ? __ldg(xb[y] + (int64_t)(J0 + j) * ld_b) : __int_as_float(0x7fc00000);
        }
    if (UNIT != 0) {
#pragma unroll
        for (int y = 0; y < kHotYears; y++)
#pragma unroll
            for (int j = 0; j < kPairDays; j++) { va[y][j] = to_celsius_f(va[y][j], UNIT); vb[y][j] = to_celsius_f(vb[y][j], UNIT); }
    }
#pragma unroll
    for (int j = 0; j < kPairDays; j++) {
        float sa[PG], sb[PG];
#pragma unroll
        for (int q = 0; q < PG; q++) { sa[q] = ta[((J0 + j) * PG + q) * kTilePad]; sb[q] = tb[((J0 + j) * PG + q) * kTilePad]; }
#pragma unroll
        for (int y = 0; y < kHotYears; y++)
#pragma unroll
            for (int q = 0; q < PG; q++) {
                if (COLD) or_if_both_lt(m[y][q], va[y][j], sa[q], vb[y][j], sb[q], 1u << (J0 + j));
                else or_if_both_gt(m[y][q], va[y][j], sa[q], vb[y][j], sb[q], 1u << (J0 + j));
            }
    }
}

// Both measures are cell-contiguous (metric_pass normalised any other layout): day t of cell c is x[t * ld_t + c].
// Shared memory: tile A then tile B, each [groups_per_slice][32 doy][PG][kTilePad].
template <int PG, int UNIT, bool COLD>
__global__ void __launch_bounds__(256, PG <= 10 ? 2 : 1)
k_hot_pair(const float *__restrict__ xa, int64_t ld_a, const float *__restrict__ xb, int64_t ld_b, int64_t C,
           const double *__restrict__ thr_a, const double *__restrict__ thr_b, int n_doy, int P, int groups_per_slice,
           const int4 *__restrict__ words, const int *__restrict__ blk_start, const int *__restrict__ blk_words,
           int K, uint32_t *__restrict__ hot)
{
    extern __shared__ float pair_s[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int db = blockIdx.y;
    const int64_t c0 = (int64_t)blockIdx.x * kTileCells;
    const int g0 = blockIdx.z * groups_per_slice;
    const int n_g = min(groups_per_slice, (P + PG - 1) / PG - g0);
    const int nd = min(kTileDoy, n_doy - db * kTileDoy);
    const int tile_floats = groups_per_slice * kTileDoy * PG * kTilePad;
    float *tile_a = pair_s, *tile_b = pair_s + tile_floats;

    if (nd < kTileDoy || (g0 + n_g) * PG > P)              // padding days / percentiles: never hot (cold)
        for (int i = tid; i < 2 * tile_floats; i += 256) pair_s[i] = __int_as_float(COLD ? 0xff800000 : 0x7f800000);
    __syncthreads();
    fill_pair_tile<PG, COLD>(tile_a, thr_a, C, c0, n_doy, db, nd, P, g0, n_g);
    fill_pair_tile<PG, COLD>(tile_b, thr_b, C, c0, n_doy, db, nd, P, g0, n_g);
    __syncthreads();

    const int64_t c = c0 + lane;
    if (c >= C) return;
    // as in k_hot_words: a warp takes kHotYears words at a time; kPairDays days of each of both measures are in flight together
    const int w_begin = blk_start[db], w_end = blk_start[db + 1];
    const int64_t plane_words = (int64_t)K * C;
    for (int i0 = w_begin + warp * kHotYears; i0 < w_end; i0 += 8 * kHotYears) {
        int kk[kHotYears], jo[kHotYears], nb[kHotYears];
        const float *pa[kHotYears], *pb[kHotYears];
        int j_hi = 0;
#pragma unroll
        for (int y = 0; y < kHotYears; y++) {
            const bool live = i0 + y < w_end;
            kk[y] = blk_words[live ? i0 + y : i0];
            const int4 w = words[kk[y]];                   // {t0, nbits, doy of bit 0, -}
            jo[y] = w.z & (kTileDoy - 1);
            nb[y] = live ? w.y : 0;
            pa[y] = xa + ((int64_t)w.x - jo[y]) * ld_a + c;
            pb[y] = xb + ((int64_t)w.x - jo[y]) * ld_b + c;
            if (live) j_hi = max(j_hi, jo[y] + nb[y]);
        }
        for (int g = 0; g < n_g; g++) {
            const int pg = (g0 + g) * PG;
            uint32_t m[kHotYears][PG];
#pragma unroll
            for (int y = 0; y < kHotYears; y++)
#pragma unroll
                for (int q = 0; q < PG; q++) m[y][q] = 0u;
            const float *ta = tile_a + (size_t)g * (kTileDoy * PG * kTilePad) + lane;
            const float *tb = tile_b + (size_t)g * (kTileDoy * PG * kTilePad) + lane;
            pair_days<PG, 0, UNIT, COLD>(m, pa, pb, jo, nb, ld_a, ld_b, ta, tb);
            if (j_hi > kPairDays) pair_days<PG, kPairDays, UNIT, COLD>(m, pa, pb, jo, nb, ld_a, ld_b, ta, tb);      // warp-uniform
            if (j_hi > 2 * kPairDays) pair_days<PG, 2 * kPairDays, UNIT, COLD>(m, pa, pb, jo, nb, ld_a, ld_b, ta, tb);
            if (j_hi > 3 * kPairDays) pair_days<PG, 3 * kPairDays, UNIT, COLD>(m, pa, pb, jo, nb, ld_a, ld_b, ta, tb);
#pragma unroll
            for (int y = 0; y < kHotYears; y++) {
                uint32_t *hp = hot + ((int64_t)pg * K + kk[y]) * C + c;     // percentile planes are K * C words apart
#pragma unroll
                for (int q = 0; q < PG; q++)
                    if (nb[y] > 0 && pg + q < P) hp[(int64_t)q * plane_words] = m[y][q] >> jo[y];
            }
        }
    }
}

static_assert(kTileDoy == 4 * kPairDays, "k_hot_pair walks a 32-day block in four steps");

bool hot_pair_plan(int P, int &pg, int &slices, int &groups_per_slice, size_t &smem)
{
    if (P <= 0 || P > HDP_B200_MAX_PERCENTILES) return false;
    pg = pick_pg(P);
    const int groups = (P + pg - 1) / pg;
    const size_t group_bytes = (size_t)2 * kTileDoy * pg * kTilePad * sizeof(float);     // both measures' tiles
    const int fit = (int)std::max<size_t>(1, kPairSmemMax / group_bytes);
    slices = (groups + fit - 1) / fit;
    groups_per_slice = (groups + slices - 1) / slices;
    smem = groups_per_slice * group_bytes;
    return true;
}

int run_hot_pair(const Layout &L, const WordPlan &plan, int64_t C, int P, cudaStream_t st, int unit, bool cold)
{
    const int K = (int)plan.words.size();
    int pg, slices, gps;
    size_t smem;
    if (!hot_pair_plan(P, pg, slices, gps, smem)) return HDP_B200_ERR_UNSUPPORTED;
    dim3 grid((unsigned)((C + kTileCells - 1) / kTileCells), (unsigned)plan.n_blk, (unsigned)slices);
    const auto kernel = hot_kernel(pg, unit, cold, [](auto PG, auto U, auto CO) {
        return k_hot_pair<decltype(PG)::value, decltype(U)::value, decltype(CO)::value>;
    });
    KernelTimer timer(kHotPair, st);
    HDP_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, 256, smem, st>>>(L.x[0], L.ld_t[0], L.x[1], L.ld_t[1], C, L.thr[0], L.thr[1], L.n_doy, P, gps, L.words, L.blk_start,
                                    L.blk_words, K, L.hot);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace hdp

using namespace hdp;

extern "C" {

size_t hdp_b200_compound_workspace_bytes(int64_t C, int64_t T, int64_t ld_c_a, int64_t ld_c_b, int n_doy, int P, int D, int Y,
                                         const int32_t *h_doy_map)
{
    (void)D;
    const int64_t ld_c[2] = {ld_c_a, ld_c_b};
    return metric_pass_workspace_bytes(C, T, ld_c, 2, n_doy, P, Y, h_doy_map, true);
}

int hdp_b200_compound(const float *d_a, int64_t ld_t_a, int64_t ld_c_a, const float *d_b, int64_t ld_t_b, int64_t ld_c_b,
                      int64_t C, int64_t T, const double *d_thr_a, const double *d_thr_b, int n_doy, int P,
                      const int32_t *h_doy_map, const int32_t *h_defs, int D,
                      const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                      const uint8_t *d_is_south, uint16_t *d_out, float *d_int,
                      void *d_workspace, size_t workspace_bytes, void *stream, int input_unit)
{
    if (C > 0 && Y > 0 && !d_out && !d_int) return HDP_B200_ERR_INVALID;
    const Measure ms[2] = {{d_a, ld_t_a, ld_c_a, d_thr_a}, {d_b, ld_t_b, ld_c_b, d_thr_b}};
    return metric_pass(ms, 2, C, T, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y, d_is_south, d_out, d_int,
                       d_workspace, workspace_bytes, stream, C, false, input_unit);
}

int hdp_b200_compound_plan(int P, int *info)
{
    if (!info || P <= 0) return HDP_B200_ERR_INVALID;
    int pg, slices, gps;
    size_t smem;
    if (!hot_pair_plan(P, pg, slices, gps, smem)) return HDP_B200_ERR_UNSUPPORTED;
    info[0] = pg; info[1] = slices; info[2] = (int)smem;
    return HDP_B200_OK;
}

}  // extern "C"
