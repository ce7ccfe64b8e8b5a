// intensity.cu - path 2, intensity: how hot the heatwaves of every season were (HWC cumulative, HWI mean, HWP peak
// exceedance of the threshold over the heatwave days; the contract is stated in intensity.h).
//
// Runs on the hot-day words k_hot_words (metric.cu) leaves in the workspace, so one call can produce the integer metrics
// (k_scan) and the intensity metrics (k_intensity) from a single pass over the samples for the hot-day bits.
//
//   k_intensity  one warp per (32 neighbouring cells, percentile), one lane per cell; the P percentile warps of a cell group sit
//                next to each other (same CTA where they fit) so that the sample sectors a run reads are shared through L1 / L2.
//                The lanes read word k of their cells together (one coalesced load per word), pop the word's hot runs and feed
//                each run to every definition's index_heatwaves state machine (hdp::index_run, seams.h - the function the
//                building-block kernel and its host replay use).  A run that some definition labels and that overlaps the lane's
//                open season then reads its in-season samples and thresholds once (lane-divergent, scattered reads) for its
//                partial sum and maximum, which go to the season accumulators of the definitions that label it.  State machines
//                and accumulators live in shared memory, [definition][lane] per warp; a season is flushed as float32 when it
//                closes.  One open season per lane: the season tables of a hemisphere must be disjoint (intensity.h).
#include <algorithm>
#include <vector>

#include "intensity.h"
#include "metric.cuh"

namespace hdp {

struct IntensityDefs {
    int v[3 * HDP_B200_MAX_DEFINITIONS];    // {min_duration, max_break, max_subs} per definition
};

constexpr int kIntWarpsMax = 8;
constexpr size_t kIntSmemMax = 200 * 1024;
constexpr int kIntBatch = 4;                 // days of a block whose sample and threshold loads are in flight together

// bytes of shared memory one warp keeps: state machine + accumulator per (definition, lane)
static size_t int_warp_bytes(int D) { return (size_t)D * 32 * (sizeof(IndexState) + sizeof(IntensityAcc)); }

__global__ void __launch_bounds__(kIntWarpsMax * 32)
k_intensity(const uint32_t *__restrict__ hot, const float *__restrict__ x, int64_t ld_t, const double *__restrict__ thr, int n_doy,
            int64_t C, int K, int T, const int4 *__restrict__ words, int P, int D, const __grid_constant__ IntensityDefs defs,
            const int4 *__restrict__ seasons_north, int n_north, const int4 *__restrict__ seasons_south, int n_south, int Y,
            const uint8_t *__restrict__ is_south, int unit, int warps_per_cta, float *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem_int[];
    int2 *word_s = (int2 *)smem_int;                                 // [K] {t0, doy of the first day}
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < K; i += blockDim.x) { const int4 w = words[i]; word_s[i] = make_int2(w.x, w.z); }
    __syncthreads();

    // warp -> (cell group, percentile), percentile-minor
    const int64_t n_cg = (C + 31) / 32;
    const int64_t wg = (int64_t)blockIdx.x * warps_per_cta + warp;
    const int64_t cg = wg / P;
    const int p = (int)(wg - cg * P);
    if (cg >= n_cg) return;                                          // warp-uniform
    const bool alive = cg * 32 + lane < C;
    const int64_t c = alive ? cg * 32 + lane : C - 1;               // lanes past the last cell shadow it and write nothing

    unsigned char *wbase = smem_int + (((size_t)K * sizeof(int2) + 15) & ~(size_t)15) + (size_t)warp * D * 32 * (sizeof(IndexState) + sizeof(IntensityAcc));
    IndexState *ist = (IndexState *)wbase;                           // [D][32]
    IntensityAcc *acc = (IntensityAcc *)(wbase + (size_t)D * 32 * sizeof(IndexState));   // [D][32]
    for (int d = 0; d < D; d++) { ist[d * 32 + lane] = IndexState(); acc[d * 32 + lane] = IntensityAcc(); }

    const bool south = is_south != nullptr && is_south[c] != 0;
    IntensityLane L;
    L.start((const int32_t *)(south ? seasons_south : seasons_north), south ? n_south : n_north);

    const int64_t plane = (int64_t)P * D * Y * C;
    auto flush = [&]() {
        for (int d = 0; d < D; d++) {
            IntensityAcc &a = acc[d * 32 + lane];
            if (alive) {
                float hwc, hwi, hwp;
                intensity_values(a, hwc, hwi, hwp);
                const int64_t o = (((int64_t)p * D + d) * Y + L.row) * C + c;
                out[o] = hwc;
                out[o + plane] = hwi;
                out[o + 2 * plane] = hwp;
            }
            a = IntensityAcc();
        }
    };
    const double *thr_c = thr + (int64_t)c * n_doy * P + p;          // thr[c, doy, p] = thr_c[doy * P]
    const float *x_c = x + c;
    int kw = 0;                                                      // word of the day being read (blocks only move forward)
    auto block = [&](int64_t lo, int64_t hi, double &r, double &m) {
        for (int64_t t0 = lo; t0 < hi; t0 += kIntBatch) {
            float v[kIntBatch];
            double th[kIntBatch];
#pragma unroll
            for (int j = 0; j < kIntBatch; j++) {
                const int t = (int)(t0 + j);
                if (t < hi) {
                    while (kw + 1 < K && word_s[kw + 1].x <= t) kw++;
                    const int2 w = word_s[kw];
                    v[j] = __ldg(x_c + (int64_t)t * ld_t);
                    th[j] = __ldg(thr_c + (int64_t)(w.y + (t - w.x)) * P);
                }
            }
#pragma unroll
            for (int j = 0; j < kIntBatch; j++)
                if (t0 + j < hi) intensity_day(r, m, intensity_excess(to_celsius_f(v[j], unit), th[j]));
        }
    };

    const uint32_t *hp = hot + (int64_t)p * K * C + c;
    HotRuns runs{&word_s[0].x, 2, K, T};
    for (int k = 0; k <= K; k++) {
        if (!__any_sync(0xffffffffu, L.open())) break;
        const uint32_t w = k < K ? __ldg(hp + (int64_t)k * C) : 0u;
        if (!L.open()) continue;
        runs.word(k, w);
        int s, e;
        while (runs.pop(s, e, kw)) intensity_run(L, s, e, label_run(ist + lane, 32, defs.v, D, s, e), acc + lane, 32, block, flush);
    }
    while (L.open()) { flush(); L.next(); }
}

int run_intensity(const Layout &L, const WordPlan &plan, const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                  const double *d_thr, int n_doy, int P, const int32_t *h_defs, int D, const std::vector<int32_t> &seasons, int Y,
                  const uint8_t *d_is_south, float *d_int, cudaStream_t st, bool tables_resident, int input_unit)
{
    const int K = (int)plan.words.size();
    const size_t words_bytes = ((size_t)K * sizeof(int2) + 15) & ~(size_t)15;
    const size_t per_warp = int_warp_bytes(D);
    if (words_bytes + per_warp > kIntSmemMax) return HDP_B200_ERR_UNSUPPORTED;
    const int wpc = (int)std::min<size_t>(kIntWarpsMax, (kIntSmemMax - words_bytes) / per_warp);
    const size_t smem = words_bytes + (size_t)wpc * per_warp;
    IntensityDefs defs;
    for (int i = 0; i < 3 * HDP_B200_MAX_DEFINITIONS; i++) defs.v[i] = i < 3 * D ? h_defs[i] : 0;
    if (!tables_resident)
        HDP_CUDA_TRY(cudaMemcpyAsync(L.int_seasons, seasons.data(), sizeof(int32_t) * seasons.size(), cudaMemcpyHostToDevice, st));
    const float *x = ld_c != 1 ? L.xn : d_measure;                  // run_hot_words normalised other layouts into L.xn
    const int64_t x_ld_t = ld_c != 1 ? C : ld_t;
    const int64_t n_warps = ((C + 31) / 32) * P;
    const unsigned grid = (unsigned)((n_warps + wpc - 1) / wpc);
    KernelTimer timer(kIntensity, st);
    HDP_CUDA_TRY(cudaFuncSetAttribute(k_intensity, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_intensity<<<grid, wpc * 32, smem, st>>>(L.hot, x, x_ld_t, d_thr, n_doy, C, K, (int)T, L.words, P, D, defs,
                                              L.int_seasons, Y, L.int_seasons + (Y + 1), Y, Y, d_is_south, input_unit, wpc, d_int);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace hdp

using namespace hdp;

extern "C" {

size_t hdp_b200_intensity_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                          int n_doy, int P, int D, int Y, const int32_t *h_doy_map)
{
    (void)ld_t; (void)D;
    return metric_pass_workspace_bytes(C, T, ld_c, n_doy, P, Y, h_doy_map, true);
}

int hdp_b200_intensity(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                       const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                       const int32_t *h_defs, int D,
                       const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                       const uint8_t *d_is_south, float *d_int, uint16_t *d_out,
                       void *d_workspace, size_t workspace_bytes, void *stream, int input_unit)
{
    if (C > 0 && Y > 0 && !d_int) return HDP_B200_ERR_INVALID;
    return metric_pass(d_measure, C, T, ld_t, ld_c, d_thr, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y,
                       d_is_south, d_out, d_int, d_workspace, workspace_bytes, stream, C, false, input_unit);
}

}  // extern "C"
