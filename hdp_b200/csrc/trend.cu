// trend.cu - trend statistics of [rows, Y, C] season series (hdp_b200_trend): Theil-Sen slope, Sen (1968) confidence interval and
// the Mann-Kendall test per (row, cell), with the rules of trend.h.
//
// k_trend<T>: one CTA per row and 32 cells.  The CTA loads the [Y, 32] tile with coalesced loads into shared memory; each of its 8
// warps then takes 4 of the 32 series, one at a time.  A warp compacts the valid values of its series (f64) and their season indices,
// walks the n x n value pairs once for S, the tie counts and the two middle values of y, and selects the four order statistics of the
// N slopes by a radix select over their 64-bit keys: 8 passes of one 8-bit digit, each recomputing every slope from the n values (so
// shared memory holds Y values per warp, not N slopes) into a 256-bin histogram per group of targets.  A warp aggregates equal bins
// with match.any before its shared-memory atomic: the high digits of most slopes are equal.
#include "common.cuh"
#include "trend.h"

namespace hdp {

namespace {

constexpr int kTrendWarps = 8;
constexpr unsigned kFull = 0xffffffffu;

template <typename T> __device__ __forceinline__ bool trend_valid(T v, int missing);
template <> __device__ __forceinline__ bool trend_valid<uint16_t>(uint16_t v, int missing) { return (int)v != missing; }
template <> __device__ __forceinline__ bool trend_valid<float>(float v, int) { return isfinite(v); }

// the value of rank r (< m) among m keys: the lanes whose key has exactly r smaller ones below and covers r write it
__device__ __forceinline__ void trend_pick(const TrendPoint &p, int64_t r, double v, double *slot)
{
    if (p.below <= r && r < p.below + p.same) *slot = v;
}

// bytes of dynamic shared memory of one CTA for Y seasons of T
template <typename T>
size_t trend_smem(int Y)
{
    return (size_t)Y * 32 * sizeof(T)                                                    // the raw tile [Y][32]
           + (size_t)kTrendWarps * ((size_t)Y * 8 + (size_t)kTrendTargets * kTrendBins * 4 + ((size_t)Y * 2 + 15) / 16 * 16)
           + (size_t)kTrendPlanes * 32 * 8 + (size_t)kTrendWarps * 2 * 8;
}

template <typename T>
__global__ void __launch_bounds__(kTrendWarps * 32) k_trend(const T *__restrict__ x, int64_t rows, int Y, int64_t C, int missing,
                                                             double zq, double *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int64_t groups = (C + 31) / 32;
    const int64_t row = (int64_t)blockIdx.x / groups, c0 = ((int64_t)blockIdx.x - row * groups) * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // layout: res [8][32] f64 | mids [warps][2] f64 | per warp: ys [Y] f64, hist [4][256] u32, xs [Y] u16 | tile [Y][32] T
    double *res = (double *)smem;
    double *mids = res + kTrendPlanes * 32;
    const size_t per_warp = (size_t)Y * 8 + kTrendTargets * kTrendBins * 4 + ((size_t)Y * 2 + 15) / 16 * 16;
    unsigned char *wbase = (unsigned char *)(mids + kTrendWarps * 2) + warp * per_warp;
    double *ys = (double *)wbase;
    uint32_t *hist = (uint32_t *)(wbase + (size_t)Y * 8);
    uint16_t *xs = (uint16_t *)(hist + kTrendTargets * kTrendBins);
    T *tile = (T *)((unsigned char *)(mids + kTrendWarps * 2) + kTrendWarps * per_warp);
    double *mid = mids + warp * 2;

    const T *src = x + row * (int64_t)Y * C + c0;
    const int width = C - c0 < 32 ? (int)(C - c0) : 32;
    for (int k = threadIdx.x; k < Y * 32; k += kTrendWarps * 32) {
        const int y = k >> 5, c = k & 31;
        if (c < width) tile[k] = src[(int64_t)y * C + c];
    }
    __syncthreads();

    for (int c = warp; c < width; c += kTrendWarps) {
        // compaction: valid values in season order
        int n = 0;
        for (int y0 = 0; y0 < Y; y0 += 32) {
            const int y = y0 + lane;
            const T v = y < Y ? tile[y * 32 + c] : T(0);
            const bool ok = y < Y && trend_valid<T>(v, missing);
            const unsigned m = __ballot_sync(kFull, ok);
            if (ok) {
                const int at = n + __popc(m & ((1u << lane) - 1u));
                ys[at] = (double)v;
                xs[at] = (uint16_t)y;
            }
            n += __popc(m);
        }
        __syncwarp();

        // one walk over the value pairs: S, the tie counts, the middle values of y
        const int64_t ylo = trend_mid_lo(n), yhi = n / 2;
        int64_t S = 0, tie_sum = 0;
        for (int i = lane; i < n; i += 32) {
            TrendPoint p;
            const double yi = ys[i];
            const uint64_t ki = trend_key(yi);
            for (int k = 0; k < n; k++) trend_point(p, yi, ki, ys[k], k > i);
            S += p.S;
            tie_sum += trend_tie_term(p.ties);
            trend_pick(p, ylo, yi, mid);
            trend_pick(p, yhi, yi, mid + 1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            S += __shfl_xor_sync(kFull, S, o);
            tie_sum += __shfl_xor_sync(kFull, tie_sum, o);
        }
        __syncwarp();
        const double var = trend_mk_var(n, tie_sum);
        const int64_t N = (int64_t)n * (n - 1) / 2;

        // radix select of the four order statistics of the N slopes
        double a[kTrendTargets] = {0.0, 0.0, 0.0, 0.0};
        if (N > 0) {
            int64_t r[kTrendTargets];
            trend_ranks(N, var, zq, r);
            TrendSelect sel;
            sel.start(r);
            const int iters = (int)((N + 31) / 32);
            for (int shift = 56; shift >= 0; shift -= 8) {
                sel.groups();
                for (int b = lane; b < sel.ng * kTrendBins; b += 32) hist[b] = 0u;
                __syncwarp();
                int i = 0, j = 1;
                trend_pair_advance(i, j, lane, n);
                for (int it = 0; it < iters; it++) {
                    int b = -1;
                    if (i < n - 1) {
                        b = sel.bin(trend_key(trend_slope(ys[i], ys[j], xs[i], xs[j])), shift);
                        trend_pair_advance(i, j, 32, n);
                    }
                    const unsigned same = __match_any_sync(kFull, b);
                    if (b >= 0 && lane == __ffs(same) - 1) atomicAdd(&hist[b], (uint32_t)__popc(same));
                }
                __syncwarp();
                // per target: the digit its rank falls on (each lane scans 8 bins, then a warp scan over the lanes)
#pragma unroll
                for (int t = 0; t < kTrendTargets; t++) {
                    const uint32_t *h = hist + sel.gid[t] * kTrendBins + lane * 8;
                    uint32_t own = 0;
#pragma unroll
                    for (int q = 0; q < 8; q++) own += h[q];
                    uint32_t incl = own;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t v = __shfl_up_sync(kFull, incl, o);
                        if (lane >= o) incl += v;
                    }
                    const int64_t rt = sel.rank[t];
                    const bool mine = (int64_t)(incl - own) <= rt && rt < (int64_t)incl;
                    const int src_lane = __ffs(__ballot_sync(kFull, mine)) - 1;
                    int d = 0;
                    int64_t before = 0;
                    if (mine) {
                        int64_t inner = 0;
                        d = lane * 8 + trend_digit(h, 8, rt - (int64_t)(incl - own), inner);
                        before = (int64_t)(incl - own) + inner;
                    }
                    d = __shfl_sync(kFull, d, src_lane);
                    before = __shfl_sync(kFull, before, src_lane);
                    sel.take(t, d, before, shift);
                }
                __syncwarp();
            }
#pragma unroll
            for (int t = 0; t < kTrendTargets; t++) a[t] = trend_unkey(sel.pre[t]);
        }

        if (lane == 0) {
            const double xmed = n > 0 ? trend_mid(n, (double)xs[ylo], (double)xs[yhi]) : 0.0;
            const double ymed = n > 0 ? trend_mid(n, mid[0], mid[1]) : 0.0;
            double o[kTrendPlanes];
            trend_finish(n, S, var, ymed, xmed, a, o);
#pragma unroll
            for (int q = 0; q < kTrendPlanes; q++) res[q * 32 + c] = o[q];
        }
        __syncwarp();
    }
    __syncthreads();
    const int64_t plane = rows * C;
    for (int k = threadIdx.x; k < kTrendPlanes * 32; k += kTrendWarps * 32) {
        const int q = k >> 5, c = k & 31;
        if (c < width) out[q * plane + row * C + c0 + c] = res[k];
    }
}

template <typename T>
int trend_launch(const T *x, int64_t rows, int Y, int64_t C, int missing, double zq, double *out, cudaStream_t st)
{
    const int64_t blocks = rows * ((C + 31) / 32);
    if (blocks > 0x7fffffffLL) return HDP_B200_ERR_UNSUPPORTED;
    const size_t smem = trend_smem<T>(Y);
    HDP_CUDA_TRY(cudaFuncSetAttribute(k_trend<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    KernelTimer timer(kTrend, st);
    k_trend<T><<<(unsigned)blocks, kTrendWarps * 32, smem, st>>>(x, rows, Y, C, missing, zq, out);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace

}  // namespace hdp

extern "C" int hdp_b200_trend(const void *d_x, int dtype, int64_t rows, int Y, int64_t C, int64_t missing, double zq, double *d_out,
                              void *stream)
{
    using namespace hdp;
    if (rows < 0 || Y < 0 || C < 0 || !(zq < 0.0) || !isfinite(zq)) return HDP_B200_ERR_INVALID;
    if (dtype != HDP_B200_DTYPE_U16 && dtype != HDP_B200_DTYPE_F32) return HDP_B200_ERR_INVALID;
    if (dtype == HDP_B200_DTYPE_U16 && (missing < -1 || missing > 0xffff)) return HDP_B200_ERR_INVALID;
    if (Y > kTrendMaxY) return HDP_B200_ERR_UNSUPPORTED;
    if (rows == 0 || C == 0) return HDP_B200_OK;
    if (!d_out || (Y > 0 && !d_x)) return HDP_B200_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == HDP_B200_DTYPE_U16) return trend_launch((const uint16_t *)d_x, rows, Y, C, (int)missing, zq, d_out, st);
    return trend_launch((const float *)d_x, rows, Y, C, -1, zq, d_out, st);
}
