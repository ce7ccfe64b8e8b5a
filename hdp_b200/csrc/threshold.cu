// threshold.cu - path 1: per cell and day of year, percentiles over the pooled day-of-year window.
//
// Replaces (reference = AgentOxygen/HDP v1.0.2):
//   compute_percentiles gufunc        hdp/threshold.py:52-78
//   compute_percentiles_wrapper       hdp/threshold.py:81-93   (the loop over cells)
//   np.quantile as compiled by Numba  numba/np/arraymath.py:1655-1704, 1754-1768
//
// The quantile arithmetic is reproduced operation by operation in double precision with explicitly
// rounded intrinsics (__dmul_rn/__dadd_rn/...), so nvcc cannot contract the interpolation into an FMA:
//     rank = 1 + (n-1) * ((q*100)/100);  f = floor(rank);  m = rank - f
//     val  = sorted[f-1] * (1-m) + sorted[f] * m
// which is bit-identical to the reference (tests/test_gpu_parity.py compares at 0 ulp).
//
// Kernels, fastest first (hdp_b200_thresholds picks by what the window tables and the quantiles allow):
//   k_thr_cand     high quantiles, finite samples: a segment of days shares one ordering of the few samples that can be
//                  among any window's largest (candidate filter); register-light, 24 warps per SM
//   k_thr_seg      any quantiles, any samples: the same segment scheme over all samples (with the candidate filter when the
//                  quantiles allow); also works through the segments k_thr_cand hands over
//   k_thr_ranked   windows that do not fit a segment (31-day windows): one ordering per cell, sliding rank bitmaps
//   k_thr_generic  any table (rows pooled any number of times, windows of up to 32 768 samples): gather + bitonic sort
#include <math.h>
#include <stdlib.h>
#include <vector>
#include <algorithm>
#include <memory>
#include <mutex>

#include "common.cuh"
#include "thr_net.cuh"

namespace hdp {

struct QTable {
    double q[HDP_B200_MAX_PERCENTILES];
};

// One output value from an ascending-sorted window (sorted[i], i < n, NaN-free: NaNs are counted separately).
// n_nan / n_pinf / n_ninf: how many NaN, +inf, -inf samples the window holds.
__device__ __forceinline__ double quantile_from_sorted(const float *sorted, int n, double q, int n_nan, int n_pinf, int n_ninf)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    // _can_collect_percentiles, arraymath.py:1707-1721
    if (n_nan > 0 || n == 0) return nan;
    if (n == 1) return (n_pinf + n_ninf) ? nan : (double)sorted[0];           // arraymath.py:1661-1663 / :1719
    const double pct = __dmul_rn(q, 100.0);                                   // arraymath.py:1757
    const bool all_finite = (n_pinf + n_ninf) == 0;
    if (pct == 100.0) {                                                       // arraymath.py:1669-1675
        const double v = (double)sorted[n - 1];
        return (!all_finite && isinf(v)) ? nan : v;
    }
    if (pct == 0.0) {                                                         // arraymath.py:1678-1695
        double v = (double)sorted[0];
        if (!all_finite) {
            const int n_fin = n - (n_pinf + n_ninf);
            if (n_fin == 0) v = nan;
            if (n_pinf == 1 && n == 2) v = nan;
            if (n_ninf > 1) v = nan;
            if (n_fin == 1 && n_pinf > 1 && n_ninf != 1) v = nan;
        }
        return v;
    }
    // arraymath.py:1697-1701
    const double rank = __dadd_rn(1.0, __dmul_rn((double)(n - 1), __ddiv_rn(pct, 100.0)));
    const double f = floor(rank);
    const double m = __dsub_rn(rank, f);
    int k = (int)f - 1;
    double lower, upper;
    if (k >= n - 1) { lower = upper = (double)sorted[n - 1]; }                // rank == n: q rounded up to the maximum
    else { if (k < 0) k = 0; lower = (double)sorted[k]; upper = (double)sorted[k + 1]; }
    return __dadd_rn(__dmul_rn(lower, __dsub_rn(1.0, m)), __dmul_rn(upper, m));
}

// ----------------------------------------------------------------------------------------------------
// k_thr_generic: gather + bitonic sort per (cell, day of year).  Handles every table the reference can
// produce (mirrored upper wrap, -1 pads, duplicated rows, any window size up to 32768 samples).
// A CTA sorts NC cells' windows for one day of year side by side.
// ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_thr_generic(const float *__restrict__ temps, int64_t C, int64_t T_b, int64_t ld_t,
              const int *__restrict__ time_index, const int *__restrict__ win_rows, int n_doy, int n_y, int W,
              const __grid_constant__ QTable qt, int P, int NC, int b_pad_log2, double *__restrict__ out)
{
    extern __shared__ float keys[];                       // [NC][b_pad], then int counts[NC][3]
    const int b = W * n_y, b_pad = 1 << b_pad_log2;
    int *counts = (int *)(keys + (size_t)NC * b_pad);
    const int tid = threadIdx.x;
    const int d = blockIdx.y;
    const int64_t c0 = (int64_t)blockIdx.x * NC;

    for (int i = tid; i < NC * 3; i += 256) counts[i] = 0;
    __syncthreads();

    // gather: consecutive threads -> consecutive cells of the same sample (one 32-byte sector for 8 cells)
    const float pinf = __int_as_float(0x7f800000);
    for (int idx = tid; idx < NC * b_pad; idx += 256) {
        const int cell = idx % NC, i = idx / NC;
        float v = pinf;                                   // padding sorts to the end
        if (i < b && c0 + cell < C) {
            const int row = win_rows[d * W + i / n_y];
            int64_t t = time_index[row * n_y + i % n_y];
            if (t < 0) t += T_b;                          // -1 pads read the LAST sample (threshold.py:35,77)
            v = temps[t * ld_t + (c0 + cell)];
            if (v != v) { atomicAdd(&counts[cell * 3 + 0], 1); v = pinf; }
            else if (v == pinf) atomicAdd(&counts[cell * 3 + 1], 1);
            else if (v == -pinf) atomicAdd(&counts[cell * 3 + 2], 1);
        }
        keys[(size_t)cell * b_pad + i] = v;
    }
    __syncthreads();

    // bitonic sort, ascending, all NC arrays in lock step
    const int half = b_pad >> 1;
    for (int k = 2; k <= b_pad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int pi = tid; pi < NC * half; pi += 256) {
                const int arr = pi >> (b_pad_log2 - 1), l = pi & (half - 1);
                const int i = ((l & ~(j - 1)) << 1) | (l & (j - 1));
                float *a = keys + (size_t)arr * b_pad;
                const float x = a[i], y = a[i | j];
                const bool up = (i & k) == 0;
                if ((x > y) == up) { a[i] = y; a[i | j] = x; }
            }
            __syncthreads();
        }
    }

    for (int idx = tid; idx < NC * P; idx += 256) {
        const int cell = idx / P, p = idx - cell * P;
        if (c0 + cell >= C) continue;
        const int *cn = counts + cell * 3;
        out[((c0 + cell) * n_doy + d) * (int64_t)P + p] =
            quantile_from_sorted(keys + (size_t)cell * b_pad, b, qt.q[p], cn[0], cn[1], cn[2]);
    }
}

// ----------------------------------------------------------------------------------------------------
// k_thr_ranked: one CTA per cell, full radix sort + sliding rank bitmaps.  The single-kernel path for shapes k_thr_seg
// does not cover (windows wider than its segments, E <= 65535).
//
//   1. gather the cell's E = n_doy * n_y window elements (every slot of the reference's time_index table,
//      -1 pads included: they are ordinary elements holding the last sample) into shared memory;
//   2. order them ONCE with a stable LSD radix sort (4-bit digits, per-thread private counters) on the
//      order-preserving integer image of the f32 samples, and record rank_of[element];
//   3. every warp owns a contiguous range of days of year and keeps that window as a bitmap over RANKS
//      (plane A: row present, plane B: row present twice - the reference's mirrored year-end wrap pools
//      some rows twice).  Moving to the next day of year flips the bits of the rows that leave / enter;
//   4. every requested percentile is read from that single ordering: the k-th and (k+1)-th window members
//      are found by a popcount prefix scan across lanes and an in-word select, and interpolated in double.
// ----------------------------------------------------------------------------------------------------
constexpr int kRankedThreads = 1024;
constexpr int kRankedWarps = kRankedThreads / 32;
constexpr int kRadixBits = 4, kRadixBins = 1 << kRadixBits, kRadixPasses = 32 / kRadixBits;

enum SelMode { kSelInterp = 0, kSelMax = 1, kSelMin = 2 };

struct SelTable {                    // per percentile, identical for every cell and day of year (n is fixed)
    int pos_lo[HDP_B200_MAX_PERCENTILES];     // 0-based positions in the sorted window
    int pos_hi[HDP_B200_MAX_PERCENTILES];
    int mode[HDP_B200_MAX_PERCENTILES];
    double w_lo[HDP_B200_MAX_PERCENTILES];    // 1 - m
    double w_hi[HDP_B200_MAX_PERCENTILES];    // m
    int8_t b_slot[64];                        // per warp: index of its plane B (rows pooled twice), -1 = none needed
};

__device__ __forceinline__ uint32_t f32_to_key(float v)
{
    const uint32_t u = __float_as_uint(v);
    if (v != v) return 0xffffffffu;                               // every NaN sorts last
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float key_to_f32(uint32_t k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// position (0..31) of the n-th (0-based) member of the multiset {bit i of a} + {bit i of b} in rank order
template <bool kTwoPlanes>
__device__ __forceinline__ int select_in_word(uint32_t a, uint32_t b, int n)
{
    int pos = 0;
#pragma unroll
    for (int width = 16; width >= 1; width >>= 1) {
        const uint32_t mask = (1u << width) - 1u;
        int c = __popc(a & mask);
        if (kTwoPlanes) c += __popc(b & mask);
        if (n >= c) { n -= c; pos += width; a >>= width; if (kTwoPlanes) b >>= width; }
    }
    return pos;
}

// members of the window whose rank lies in [lo, hi) (warp-cooperative; non-finite bookkeeping only)
__device__ __forceinline__ int range_count(const uint32_t *A, const uint32_t *B, bool dup, int wpl, int lane, int lo, int hi)
{
    int c = 0;
    for (int i = 0; i < wpl; i++) {
        const int w = lane * wpl + i, r0 = w * 32;
        if (r0 + 32 <= lo || r0 >= hi) continue;
        uint32_t m = 0xffffffffu;
        if (lo > r0) m &= 0xffffffffu << (lo - r0);
        if (hi < r0 + 32) m &= (1u << (hi - r0)) - 1u;
        c += __popc(A[w] & m) + (dup ? __popc(B[w] & m) : 0);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    return c;
}

__global__ void __launch_bounds__(kRankedThreads, 1)
k_thr_ranked(const float *__restrict__ temps, int64_t T_b, int64_t ld_t,
             const int *__restrict__ time_index, int E, int n_y, int n_doy, int n,
             const int *__restrict__ op_off, const int *__restrict__ ops, const uint8_t *__restrict__ doy_dup,
             int dpw, int ept, int nwords_pad, const __grid_constant__ SelTable sel, int P, double *__restrict__ out,
             const int *__restrict__ cell_count, const int *__restrict__ cell_list)
{
    constexpr int NT = kRankedThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Epad = (E + 63) & ~63;
    uint32_t *keyA = (uint32_t *)smem_raw;                        // sorted keys after the last pass
    uint16_t *rank_of = (uint16_t *)(keyA + Epad);                // also the second index buffer of the sort
    uint32_t *keyB = (uint32_t *)(rank_of + Epad);
    uint16_t *idxA = (uint16_t *)(keyB + Epad);
    uint16_t *cnt = idxA + Epad;                                  // [16][NT] private digit counters
    uint32_t *planes = keyB;                                      // after the sort: [warp][2][nwords_pad] (over keyB, idxA, cnt)
    __shared__ int s_nonfinite[3];                                // NaN, +inf, -inf elements of this cell
    __shared__ int s_warp_tot[kRankedWarps];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // cells: blockIdx.x itself, or (as the hand-over target of k_thr_cell) the entries of a device-side list
    const int n_cells = cell_list ? *cell_count : (int)gridDim.x;
    for (int ci = blockIdx.x; ci < n_cells; ci += gridDim.x) {
    const int64_t c = cell_list ? cell_list[ci] : ci;

    __syncthreads();
    if (tid < 3) s_nonfinite[tid] = 0;
    __syncthreads();

    // ---- 1. gather ----
    const float pinf = __int_as_float(0x7f800000);
    for (int e = tid; e < E; e += NT) {
        int64_t t = time_index[e];
        if (t < 0) t += T_b;                                      // -1 pads read the LAST sample (threshold.py:35,77)
        const float v = temps[t * ld_t + c];
        if (v != v) atomicAdd(&s_nonfinite[0], 1);
        else if (v == pinf) atomicAdd(&s_nonfinite[1], 1);
        else if (v == -pinf) atomicAdd(&s_nonfinite[2], 1);
        keyA[e] = f32_to_key(v);
        idxA[e] = (uint16_t)e;
    }
    __syncthreads();

    // ---- 2. stable LSD radix sort of (key, element) ----
    {
        uint32_t *sk = keyA, *dk = keyB;
        uint16_t *si = idxA, *di = rank_of;
        const int e0 = min(tid * ept, E), e1 = min(e0 + ept, E);
        for (int pass = 0; pass < kRadixPasses; pass++) {
            const int shift = pass * kRadixBits;
#pragma unroll
            for (int d = 0; d < kRadixBins; d++) cnt[d * NT + tid] = 0;
            for (int e = e0; e < e1; e++) cnt[((sk[e] >> shift) & (kRadixBins - 1)) * NT + tid]++;
            __syncthreads();
            // exclusive scan of the 16*NT counters in (digit, thread) order; thread t owns entries [16t, 16t+16)
            uint16_t *mine = cnt + tid * kRadixBins;
            int local[kRadixBins], tot = 0;
#pragma unroll
            for (int i = 0; i < kRadixBins; i++) { local[i] = tot; tot += mine[i]; }
            int incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            if (lane == 31) s_warp_tot[warp] = incl;
            __syncthreads();
            int base = incl - tot;
            for (int w = 0; w < warp; w++) base += s_warp_tot[w];
#pragma unroll
            for (int i = 0; i < kRadixBins; i++) mine[i] = (uint16_t)(base + local[i]);
            __syncthreads();
            for (int e = e0; e < e1; e++) {
                const uint32_t k = sk[e];
                const int slot = ((k >> shift) & (kRadixBins - 1)) * NT + tid;
                const int pos = cnt[slot];
                cnt[slot] = (uint16_t)(pos + 1);
                dk[pos] = k;
                di[pos] = si[e];
            }
            __syncthreads();
            uint32_t *tk = sk; sk = dk; dk = tk;
            uint16_t *ti = si; si = di; di = ti;
        }
        // an even number of passes: sorted keys are back in keyA, their elements in idxA
    }
    for (int r = tid; r < E; r += NT) rank_of[idxA[r]] = (uint16_t)r;
    __syncthreads();

    // ---- 3./4. sliding rank bitmaps, one day-of-year range per warp ----
    const int wpl = nwords_pad >> 5;                              // bitmap words per lane
    // layout: [warp] plane A | [warp] members-in-front-of-word (u16) | plane B of the few warps that need one
    uint32_t *A = planes + (size_t)warp * nwords_pad;
    uint16_t *pre = (uint16_t *)(planes + (size_t)kRankedWarps * nwords_pad) + (size_t)warp * nwords_pad;
    const bool range_dup = sel.b_slot[warp] >= 0;
    uint32_t *B = planes + (size_t)kRankedWarps * nwords_pad * 3 / 2 + (size_t)(range_dup ? sel.b_slot[warp] : 0) * nwords_pad;
    for (int i = lane; i < nwords_pad; i += 32) { A[i] = 0u; if (range_dup) B[i] = 0u; }
    const int d_begin = warp * dpw, d_end = min(n_doy, d_begin + dpw);
    const int n_nan = s_nonfinite[0], n_pinf = s_nonfinite[1], n_ninf = s_nonfinite[2];
    const bool nonfinite = (n_nan | n_pinf | n_ninf) != 0;
    __syncwarp();

    for (int d = d_begin; d < d_end; d++) {
        // rows leaving / entering the window (multiset difference to the previous day; full build on the first)
        for (int o = op_off[d]; o < op_off[d + 1]; o++) {
            const int op = ops[o], row = op >> 1;
            for (int j = lane; j < n_y; j += 32) {
                const int r = rank_of[row * n_y + j];
                const uint32_t bit = 1u << (r & 31);
                if (op & 1) {
                    const uint32_t old = atomicOr(&A[r >> 5], bit);
                    if (range_dup && (old & bit)) atomicOr(&B[r >> 5], bit);
                } else {
                    if (range_dup && (B[r >> 5] & bit)) atomicAnd(&B[r >> 5], ~bit);
                    else atomicAnd(&A[r >> 5], ~bit);
                }
            }
            __syncwarp();
        }
        const bool dup = doy_dup[d] != 0;

        // members per lane slice (and the running count in front of every word), inclusive scan across lanes
        int s = 0;
        if (!dup) {
#pragma unroll 4
            for (int i = 0; i < wpl; i++) { pre[lane * wpl + i] = (uint16_t)s; s += __popc(A[lane * wpl + i]); }
        } else {
            for (int i = 0; i < wpl; i++) { pre[lane * wpl + i] = (uint16_t)s; s += __popc(A[lane * wpl + i]) + __popc(B[lane * wpl + i]); }
        }
        int incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        __syncwarp();

        int w_nan = 0, w_pinf = 0, w_ninf = 0;
        if (nonfinite) {                                          // rare: count the window's non-finite members by rank range
            w_ninf = range_count(A, B, dup, wpl, lane, 0, n_ninf);
            w_pinf = range_count(A, B, dup, wpl, lane, E - n_nan - n_pinf, E - n_nan);
            w_nan = range_count(A, B, dup, wpl, lane, E - n_nan, E);
        }

        for (int p0 = 0; p0 < P; p0 += 16) {
            // lane 2i -> lower pick of percentile p0+i, lane 2i+1 -> upper pick
            const int p = min(p0 + (lane >> 1), P - 1);
            const int target = (lane & 1) ? sel.pos_hi[p] : sel.pos_lo[p];
            int lo = 0, hi = 31;                                  // first lane whose inclusive count exceeds target
#pragma unroll
            for (int it = 0; it < 5; it++) {
                const int mid = (lo + hi) >> 1;
                const int v = __shfl_sync(0xffffffffu, incl, mid);
                if (v > target) hi = mid; else lo = mid + 1;
            }
            const int owner = lo;
            int rem = target - (__shfl_sync(0xffffffffu, incl, owner) - __shfl_sync(0xffffffffu, s, owner));
            // last word of the owner's slice whose running count is <= rem (binary search over <= 16 words)
            const uint16_t *pw = pre + owner * wpl;
            int wl = 0, wh = wpl - 1;
            while (wl < wh) {
                const int mid = (wl + wh + 1) >> 1;
                if ((int)pw[mid] <= rem) wl = mid; else wh = mid - 1;
            }
            const int w = owner * wpl + wl;
            rem -= pw[wl];
            const uint32_t a = A[w], b = dup ? B[w] : 0u;
            const int bitpos = dup ? select_in_word<true>(a, b, rem) : select_in_word<false>(a, 0u, rem);
            const int r = min(w * 32 + bitpos, E - 1);
            const double val = (double)key_to_f32(keyA[r]);
            const double lower = __shfl_sync(0xffffffffu, val, (lane & 15) * 2);
            const double upper = __shfl_sync(0xffffffffu, val, (lane & 15) * 2 + 1);
            if (lane < 16 && p0 + lane < P) {
                const int pp = p0 + lane, mode = sel.mode[pp];
                const double nan = __longlong_as_double(0x7ff8000000000000LL);
                double v;
                if (mode == kSelInterp) {                         // arraymath.py:1697-1701
                    v = __dadd_rn(__dmul_rn(lower, sel.w_lo[pp]), __dmul_rn(upper, sel.w_hi[pp]));
                } else if (mode == kSelMax) {                     // arraymath.py:1669-1675
                    v = upper;
                    if ((w_pinf | w_ninf) && isinf(v)) v = nan;
                } else {                                          // arraymath.py:1678-1695
                    v = lower;
                    if (w_pinf | w_ninf) {
                        const int n_fin = n - (w_pinf + w_ninf);
                        if (n_fin == 0) v = nan;
                        if (w_pinf == 1 && n == 2) v = nan;
                        if (w_ninf > 1) v = nan;
                        if (n_fin == 1 && w_pinf > 1 && w_ninf != 1) v = nan;
                    }
                }
                if (w_nan > 0) v = nan;                           // _can_collect_percentiles, arraymath.py:1714
                out[(c * n_doy + d) * (int64_t)P + pp] = v;
            }
        }
    }
}   // cells
}

// ----------------------------------------------------------------------------------------------------
// k_thr_seg: the current fast path.  One WARP per (cell, SEGMENT of S consecutive days of year); the warps of a CTA
// own neighbouring cells of the same segment.
//
// The windows of a segment touch R <= S + W - 1 day-of-year rows, i.e. NE = R * n_y <= 1024 samples.
//   G. the CTA gathers the [cells x NE] tile: 8 neighbouring cells of one time step are one 32-byte sector, so every
//      sector that crosses L2 -> SM is used completely (one block-wide barrier; everything after it is warp-private);
//   1. each lane takes 32 of its cell's samples into registers; finite min / max, NaN / +inf / -inf counts;
//   2. counting sort in ONE pass: monotone bucket b = 1 + trunc((v - vmin) * scale) out of 2048 (float subtraction,
//      multiplication and truncation are monotone, so bucket order never contradicts value order; -inf, +inf and NaN
//      have buckets of their own), one shared-memory atomic on a 16-bit counter claims the slot inside the bucket;
//      the lane that draws slot 1 puts the bucket on a work list (it holds more than one sample);
//   3. exclusive scan of the counters (two packed 16-bit sums per add), position = base[bucket] + slot;
//   4. the samples are scattered to their positions together with their local row; buckets on the work list are
//      put in exact order by insertion sort on the float values, long runs by a warp-wide counting rank;
//   5. PB[i] = bitmap over the sorted positions ("local ranks") of the samples in local rows < i, and
//      cum[i][w] = how many of them sit in words < w.  Rows own disjoint bits, so the members of a window of rows
//      [r0, r1) are PB[r1] ^ PB[r0] and cum[r1][w] - cum[r0][w] of them come before word w;
//   6. every (day of year, percentile) query is answered independently by one lane: binary search over the 32
//      words, in-word select, value lookup, interpolation in double.  Rows pooled twice (the reference's mirrored
//      year-end wrap) are a second set of ranges.
// Each ordering serves S days x P percentiles; nothing a query reads changes once built.  Samples never leave the SM.
// ----------------------------------------------------------------------------------------------------
constexpr int kSegWarps = 8;                                      // warps = cells per CTA: 8 x 4 bytes = one sector per time step
constexpr int kSegCap = 1024;                                     // samples per segment: 32 words of 32 sorted positions
constexpr int kSegRounds = kSegCap / 32;
constexpr int kSegNB = 2048, kSegNBHalf = kSegNB / 2;             // buckets; 16-bit counters, bucket b -> word b & 1023, half b >> 10
constexpr int kSegNBF = kSegNB - 4;                               // finite buckets 1 .. NBF; -inf 0, +inf NB-3, NaN NB-2
constexpr int kSegRowsMax = 32;                                   // local rows 0 .. R of the prefix tables: R <= 31
constexpr int kSegPst = 33, kSegCst = 34;                         // words per PB row, u16 per cum row (both odd in words)
constexpr int kSegLongRun = 32;                                   // buckets with more samples are ordered by the whole warp
constexpr int kSegCandTop = 8;                                   // largest per-row rank the candidate filter can ask for
constexpr int kSegRanges = 5;                                     // <= 3 ranges of rows pooled (at least) once + <= 2 pooled twice
// per-warp workspace (bytes)
constexpr int kSegOffSv = 0;                                      // f32 [1024] the gathered tile row, then the sorted values
constexpr int kSegOffCnt = 4096;                                  // u32 [1024 + 32] packed counters / bases (word w at w + (w >> 5)), then PB [32][33]
constexpr int kSegOffRw = kSegOffCnt + 4224;                      // u8 [1024] local row of every sorted position ...
constexpr int kSegOffWl = kSegOffRw + 1024;                       // ... u16 [512] work list (then the row copy of a long run) ...
constexpr int kSegOffLong = kSegOffWl + 1024;                     // ... u32 [32] long runs; the three together: cum u16 [32][34]
constexpr int kSegWarpBytes = kSegOffLong + 128 + 16;             // = 16 (mod 128): the 8 tile rows start in different banks
static_assert(kSegOffLong + 128 - kSegOffRw >= kSegRowsMax * kSegCst * 2, "cum does not fit");
static_assert(kSegRowsMax * kSegPst * 4 <= 4224, "PB does not fit");

struct SegGeom {
    int S, n_seg;                       // days per segment, segments per cell
    int gc, n_groups;                   // cell groups (of kSegWarps cells) per L2-sized chunk, cell groups in all
    int ny_magic;                       // (k * ny_magic) >> 16 == k / n_y for k < 1024
    int n_y;                            // samples per day-of-year row
    int cand_m;                         // candidate filter: keep the samples >= min over rows of the row's cand_m-th largest; 0 = off
    int unit;                           // k_thr_seg behind k_thr_net only: input unit of the samples (to_celsius_f), else 0
};

struct SelShared {                      // SelTable without the k_thr_ranked bookkeeping, in shared memory
    int pos_lo[HDP_B200_MAX_PERCENTILES], pos_hi[HDP_B200_MAX_PERCENTILES], mode[HDP_B200_MAX_PERCENTILES];
    double w_lo[HDP_B200_MAX_PERCENTILES], w_hi[HDP_B200_MAX_PERCENTILES];
};

__device__ __forceinline__ uint32_t lowmask(uint32_t n) { return n >= 32u ? 0xffffffffu : ((1u << n) - 1u); }
__device__ __forceinline__ uint32_t byte_of(const uint4 &v, int i)
{
    const uint32_t w = i < 4 ? v.x : i < 8 ? v.y : i < 12 ? v.z : v.w;
    return (w >> ((i & 3) * 8)) & 0xffu;
}

// A window as row ranges over the segment's local rows: range k covers rows [lo_k, hi_k); ranges < n1 are the rows
// pooled at least once, ranges n1 .. nr-1 the rows pooled twice.  ca/cb: shared addresses of cum rows hi/lo, pa/pb: of PB rows.
// (Plain C++ loads here, not volatile PTX: nothing is written during the query phase, and the compiler is free to
// interleave the independent dependency chains of the two queries a lane works on.)
template <int NR>
struct SegWin {
    const uint16_t *ca[NR], *cb[NR];
    const uint32_t *pa[NR], *pb[NR];
    int n1, nr;
    __device__ __forceinline__ int before(int w) const            // members in words < w
    {
        int cnt = 0;
#pragma unroll
        for (int k = 0; k < NR; k++)
            if (NR == 1 || k < nr) cnt += (int)ca[k][w] - (int)cb[k][w];
        return cnt;
    }
    __device__ __forceinline__ void bits(int w, uint32_t &a, uint32_t &b) const   // a: members of word w, b: members pooled twice
    {
        a = 0u; b = 0u;
#pragma unroll
        for (int k = 0; k < NR; k++)
            if (NR == 1 || k < nr) {
                const uint32_t v = pa[k][w] ^ pb[k][w];
                if (NR == 1 || k < n1) a |= v; else b |= v;
            }
    }
};

// sorted positions of the pos_lo-th and pos_hi-th (0-based, pos_lo <= pos_hi < n) members of the window
template <int NR>
__device__ __forceinline__ void seg_pick(const SegWin<NR> &win, int pos_lo, int pos_hi, int &lr_lo, int &lr_hi)
{
    int w = 0, bw = 0;                                            // bw = members in words < w
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int c = win.before(w + step);
        if (c <= pos_lo) { w += step; bw = c; }
    }
    uint32_t a, b;
    win.bits(w, a, b);
    int rem = pos_lo - bw;
    const int bit = NR == 1 ? select_in_word<false>(a, 0u, rem) : select_in_word<true>(a, b, rem);
    lr_lo = w * 32 + bit;
    lr_hi = lr_lo;
    if (pos_hi != pos_lo) {
        if (NR == 1 && pos_hi == pos_lo + 1) {                    // the next member: the next set bit, here or in a later word
            a &= 0xfffffffeu << bit;
            while (a == 0u && w < 31) { w++; win.bits(w, a, b); }
            lr_hi = w * 32 + __ffs(a) - 1;
            return;
        }
        rem += pos_hi - pos_lo;
        int cw = __popc(a) + __popc(b);
        while (rem >= cw && w < 31) {                             // the upper pick lives in a later word
            rem -= cw;
            w++;
            win.bits(w, a, b);
            cw = __popc(a) + __popc(b);
        }
        lr_hi = w * 32 + (NR == 1 ? select_in_word<false>(a, 0u, rem) : select_in_word<true>(a, b, rem));
    }
}

// The same for TWO single-range windows at once: two independent dependency chains in straight-line code.
__device__ __forceinline__ void seg_pick2(const SegWin<1> &wa, const SegWin<1> &wb, int lo_a, int hi_a, int lo_b, int hi_b,
                                          int &lr_lo_a, int &lr_hi_a, int &lr_lo_b, int &lr_hi_b)
{
    int w_a = 0, bw_a = 0, w_b = 0, bw_b = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int c_a = wa.before(w_a + step), c_b = wb.before(w_b + step);
        if (c_a <= lo_a) { w_a += step; bw_a = c_a; }
        if (c_b <= lo_b) { w_b += step; bw_b = c_b; }
    }
    uint32_t a_a, a_b, unused;
    wa.bits(w_a, a_a, unused);
    wb.bits(w_b, a_b, unused);
    int n_a = lo_a - bw_a, n_b = lo_b - bw_b, bit_a = 0, bit_b = 0;
    uint32_t t_a = a_a, t_b = a_b;
#pragma unroll
    for (int width = 16; width >= 1; width >>= 1) {
        const uint32_t mask = (1u << width) - 1u;
        const int c_a = __popc(t_a & mask), c_b = __popc(t_b & mask);
        if (n_a >= c_a) { n_a -= c_a; bit_a += width; t_a >>= width; }
        if (n_b >= c_b) { n_b -= c_b; bit_b += width; t_b >>= width; }
    }
    lr_lo_a = w_a * 32 + bit_a; lr_hi_a = lr_lo_a;
    lr_lo_b = w_b * 32 + bit_b; lr_hi_b = lr_lo_b;
    if (hi_a != lo_a) {                                           // hi == lo + 1 here: the next set bit, in this word or a later one
        a_a &= 0xfffffffeu << bit_a;
        while (a_a == 0u && w_a < 31) { w_a++; wa.bits(w_a, a_a, unused); }
        lr_hi_a = w_a * 32 + __ffs(a_a) - 1;
    }
    if (hi_b != lo_b) {
        a_b &= 0xfffffffeu << bit_b;
        while (a_b == 0u && w_b < 31) { w_b++; wb.bits(w_b, a_b, unused); }
        lr_hi_b = w_b * 32 + __ffs(a_b) - 1;
    }
}

// members of the window at sorted positions < L
template <int NR>
__device__ __forceinline__ int seg_below(const SegWin<NR> &win, int L, int n)
{
    if (L >= kSegCap) return n;
    uint32_t a, b;
    win.bits(L >> 5, a, b);
    const uint32_t m = lowmask((uint32_t)(L & 31));
    return win.before(L >> 5) + __popc(a & m) + __popc(b & m);
}

// start of bucket b in the sorted order (after the scan)
__device__ __forceinline__ int seg_bucket_base(uint32_t s_cnt, uint32_t b)
{
    const uint32_t w = b & (kSegNBHalf - 1);
    return (int)((lds_u32(s_cnt + 4u * (w + (w >> 5))) >> ((b >> 6) & 16u)) & 0xffffu);
}

// phase 2 for a batch of kSegBatch register rounds: buckets first, then all the atomics of the batch back to back (their
// latencies overlap), then slots; the lanes that draw slot 1 append their bucket to the work list.
// pk = counter byte offset << 9 (word aligned: bits 11..) | half << 10 | slot.
constexpr int kSegBatch = 8;
template <bool kNonFinite>
__device__ __forceinline__ void seg_claim(const float *x, uint32_t *pk, int m0, int nl /* NE - lane */, float vmin, float scale,
                                          uint32_t s_cnt, uint32_t s_wl, int &n_wl, uint32_t lt_mask)
{
    uint32_t bb[kSegBatch], old[kSegBatch];
#pragma unroll
    for (int j = 0; j < kSegBatch; j++) {
        const float v = x[m0 + j];
        const int bi = __float2int_rz((v - vmin) * scale);        // finite: >= 0; NaN -> 0
        uint32_t b = 1u + (uint32_t)min(bi, kSegNBF - 1);
        if (kNonFinite) {
            const float pinf = __int_as_float(0x7f800000);
            b = 1u + (uint32_t)min(max(bi, 0), kSegNBF - 1);
            if (v == pinf) b = (uint32_t)kSegNB - 3u;
            if (v == -pinf) b = 0u;
            if (v != v) b = (uint32_t)kSegNB - 2u;
        }
        bb[j] = b;
    }
#pragma unroll
    for (int j = 0; j < kSegBatch; j++) {
        const uint32_t w = bb[j] & (kSegNBHalf - 1), sh = (bb[j] >> 6) & 16u;
        old[j] = 0u;
        if (nl > 32 * (m0 + j)) old[j] = atoms_add(s_cnt + 4u * (w + (w >> 5)), 1u << sh);
    }
#pragma unroll
    for (int j = 0; j < kSegBatch; j++) {
        const uint32_t b = bb[j], w = b & (kSegNBHalf - 1), half = (b >> 10) & 1u;   // (masked: lanes without a sample hold garbage)
        const uint32_t slot = (old[j] >> (half << 4)) & 0xffffu;
        pk[m0 + j] = ((w + (w >> 5)) << 11) | (half << 10) | slot;
        const bool second = nl > 32 * (m0 + j) && slot == 1u && (!kNonFinite || b - 1u < (uint32_t)kSegNBF);
        const uint32_t hit = __ballot_sync(0xffffffffu, second);
        if (second) sts_u16(s_wl + 2u * (n_wl + __popc(hit & lt_mask)), b);
        n_wl += __popc(hit);
    }
}

// the M-th largest of the n_y samples at shared address a0
template <int M>
__device__ __forceinline__ float seg_row_top(uint32_t a0, int n_y)
{
    float t[M];
#pragma unroll
    for (int i = 0; i < M; i++) t[i] = -__int_as_float(0x7f800000);
#pragma unroll 2
    for (int y = 0; y < n_y; y++) {
        float v = lds_f32(a0 + 4u * y);
#pragma unroll
        for (int i = 0; i < M; i++) { const float hi = fmaxf(t[i], v); v = fminf(t[i], v); t[i] = hi; }
    }
    return t[M - 1];
}

__global__ void __launch_bounds__(kSegWarps * 32, 2)
k_thr_seg(const float *__restrict__ temps, int64_t C, int64_t ld_t,
          const int *__restrict__ seg_time, const int *__restrict__ seg_ne, const uint4 *__restrict__ doy_rng,
          const __grid_constant__ SegGeom geo, const __grid_constant__ SelTable sel, int P, int n, int n_doy,
          double *__restrict__ out, const uint32_t *__restrict__ handed_over, int n_blocks)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ SelShared s_sel;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int i = tid; i < P; i += kSegWarps * 32) {
        s_sel.pos_lo[i] = sel.pos_lo[i]; s_sel.pos_hi[i] = sel.pos_hi[i]; s_sel.mode[i] = sel.mode[i];
        s_sel.w_lo[i] = sel.w_lo[i]; s_sel.w_hi[i] = sel.w_hi[i];
    }
    // Work items.  First (only) launch: one per block of the grid.  Second launch behind k_thr_cand (handed_over != nullptr):
    // the blocks on its hand-over list [count, flags[n_blocks], list[n_blocks]], taken in turns by a small grid; flags[b] = the
    // warps of block b that k_thr_cand left to this kernel.
    const bool from_list = handed_over != nullptr;
    const unsigned n_items = from_list ? handed_over[0] : 1u;
    for (unsigned item = from_list ? blockIdx.x : 0u; item < n_items; item += from_list ? gridDim.x : 1u) {
    const unsigned bid = from_list ? handed_over[1 + n_blocks + item] : blockIdx.x;
    const uint32_t only_mask = from_list ? handed_over[1 + bid] : 0xffffffffu;

    // block -> (chunk of cell groups, segment, cell group): blocks in flight share the segment's time rows, and the
    // halo rows a chunk's neighbouring segments read again are still in L2
    const int per_chunk = geo.n_seg * geo.gc;
    const int chunk = bid / per_chunk, rem_b = bid - chunk * per_chunk;
    const int gcc = min(geo.gc, geo.n_groups - chunk * geo.gc);   // cell groups of this chunk
    const int sg = rem_b / gcc, group = chunk * geo.gc + (rem_b - sg * gcc);
    if (sg >= geo.n_seg) return;                                  // block-uniform (the last chunk is smaller; never on the list), before any barrier
    const int64_t c0 = (int64_t)group * kSegWarps;
    const int NE = seg_ne[sg];

    // ---- G. gather the [cells x NE] tile: lanes 8j .. 8j+7 read the 8 cells of one time step ----
    {
        const int *st = seg_time + (size_t)sg * kSegCap;
        const int cl = tid & (kSegWarps - 1);
        const float *src = temps + min(c0 + cl, C - 1);
        float *dst = (float *)(smem_raw + (size_t)cl * kSegWarpBytes + kSegOffSv);
        const uint32_t s_dst = smem_u32(dst);
#pragma unroll 8
        for (int k = tid / kSegWarps; k < NE; k += 32)            // asynchronous 4-byte copies: every load of the tile is in flight at once
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s_dst + 4u * k), "l"(src + (int64_t)st[k] * ld_t) : "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
        if (geo.unit != 0)                                        // Kelvin / Fahrenheit input: every thread converts what it gathered
            for (int k = tid / kSegWarps; k < NE; k += 32) dst[k] = to_celsius_f(dst[k], geo.unit);
    }
    __syncthreads();                                              // the tile is complete
    [&]() {                                                       // everything below is warp-private: `return` leaves this warp's item
    const int64_t cell = c0 + warp;
    if (cell >= C || !((only_mask >> warp) & 1u)) return;         // warp-uniform

    const uint32_t s_base = smem_u32(smem_raw + (size_t)warp * kSegWarpBytes);
    const uint32_t s_sv = s_base + kSegOffSv, s_cnt = s_base + kSegOffCnt, s_pb = s_cnt, s_rw = s_base + kSegOffRw,
                   s_wl = s_base + kSegOffWl, s_long = s_base + kSegOffLong, s_cum = s_rw;

    // ---- 1. samples into registers; min / max; non-finite census ----
    const float pinf = __int_as_float(0x7f800000);
    float x[kSegRounds];
    float vmin = pinf, vmax = -pinf;
    bool odd = false;                                             // some valid sample is NaN or +-inf
#pragma unroll
    for (int m0 = 0; m0 < kSegRounds; m0 += kSegBatch) {
#pragma unroll
        for (int j = 0; j < kSegBatch; j++) x[m0 + j] = 0.0f;
        if (32 * m0 < NE) {                                       // warp-uniform
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) x[m0 + j] = lds_f32(s_sv + 4u * (32 * (m0 + j) + lane));
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) {
                const float v = x[m0 + j];
                const bool valid = NE - lane > 32 * (m0 + j);
                odd |= valid && !(fabsf(v) < pinf);
                if (valid) { vmin = fminf(vmin, v); vmax = fmaxf(vmax, v); }
            }
        }
    }
    for (int i = lane; i < 1024 + 32; i += 32) sts_u32(s_cnt + 4u * i, 0u);
    int n_nan = 0, n_pinf = 0, n_ninf = 0;
    const bool nonfinite = __any_sync(0xffffffffu, odd);
    if (nonfinite) {                                              // rare: redo min / max over the finite samples only, count the rest
        vmin = pinf; vmax = -pinf;
#pragma unroll
        for (int m = 0; m < kSegRounds; m++) {
            const float v = x[m];
            if (lane < NE - 32 * m) {
                if (v != v) n_nan++;
                else if (v == pinf) n_pinf++;
                else if (v == -pinf) n_ninf++;
                else { vmin = fminf(vmin, v); vmax = fmaxf(vmax, v); }
            }
        }
        n_nan = __reduce_add_sync(0xffffffffu, n_nan);
        n_pinf = __reduce_add_sync(0xffffffffu, n_pinf);
        n_ninf = __reduce_add_sync(0xffffffffu, n_ninf);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
        vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    __syncwarp();

    // ---- 1b. candidate filter (high quantiles only) ----
    // Every requested position is >= kmin, i.e. among the K = n - kmin largest samples of its window.  A window pools W
    // rows; with m = ceil(K / W) and tau = min over the segment's rows of the row's m-th largest sample, every window holds
    // at least m W >= K samples >= tau, so its K largest are all >= tau: only those "candidates" need to be ordered.
    // The window's other members are all smaller than the sample at position kmin, so position pos of the window is
    // position pos - (n - candidates in the window) among its candidates (phase 6).
    int NEc = NE;                                                 // samples that take part in the ordering
    uint32_t rw4[kSegRounds / 4];                                 // local rows of this lane's candidates, four per register
    const bool cand = geo.cand_m > 0 && !nonfinite;               // warp-uniform
    if (cand) {
        const int R0 = (NE * geo.ny_magic) >> 16;
        float tau = pinf;                                         // lane = row: the row's cand_m-th largest sample
        if (lane < R0) {
            const uint32_t a0 = s_sv + 4u * (uint32_t)(lane * geo.n_y);
            switch (geo.cand_m) {                                 // warp-uniform
            case 1: tau = seg_row_top<1>(a0, geo.n_y); break;
            case 2: tau = seg_row_top<2>(a0, geo.n_y); break;
            case 3: tau = seg_row_top<3>(a0, geo.n_y); break;
            case 4: tau = seg_row_top<4>(a0, geo.n_y); break;
            case 5: tau = seg_row_top<5>(a0, geo.n_y); break;
            case 6: tau = seg_row_top<6>(a0, geo.n_y); break;
            case 7: tau = seg_row_top<7>(a0, geo.n_y); break;
            default: tau = seg_row_top<8>(a0, geo.n_y); break;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tau = fminf(tau, __shfl_xor_sync(0xffffffffu, tau, o));
        // every lane packs its own candidates behind those of the lanes before it (the order does not matter)
        int mine = 0;
#pragma unroll
        for (int m = 0; m < kSegRounds; m++) mine += (NE - lane > 32 * m && x[m] >= tau) ? 1 : 0;
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        NEc = __shfl_sync(0xffffffffu, incl, 31);
        __syncwarp();                                             // the tile has been read: its place takes the compacted candidates
        uint32_t pos = (uint32_t)(incl - mine);
#pragma unroll
        for (int m = 0; m < kSegRounds; m++) {
            if (32 * m < NE) {                                    // warp-uniform
                if (NE - lane > 32 * m && x[m] >= tau) {
                    sts_f32(s_sv + 4u * pos, x[m]);
                    sts_u8(s_rw + pos, ((uint32_t)(32 * m + lane) * (uint32_t)geo.ny_magic) >> 16);
                    pos++;
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int m = 0; m < kSegRounds; m++) {
            if ((m & 3) == 0) rw4[m >> 2] = 0u;
            if (32 * m < NEc) {                                   // warp-uniform
                const bool have = NEc - lane > 32 * m;
                x[m] = have ? lds_f32(s_sv + 4u * (32 * m + lane)) : 0.0f;
                rw4[m >> 2] |= (have ? lds_u8(s_rw + 32 * m + lane) : 0u) << (8 * (m & 3));
            }
        }
        vmin = tau;
        __syncwarp();
    }

    // ---- 2. monotone buckets; one atomic claims the slot inside the bucket ----
    const float range = vmax - vmin;
    const float scale = (range > 0.0f && range < pinf) ? (float)(kSegNBF - 1) / range : 0.0f;
    uint32_t pk[kSegRounds];                                      // where the counter is | slot
    int n_wl = 0;                                                 // warp-uniform
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int nl = NEc - lane;                                     // round m holds a sample of this lane iff nl > 32 m
    if (!nonfinite) {
#pragma unroll
        for (int m0 = 0; m0 < kSegRounds; m0 += kSegBatch) {
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) pk[m0 + j] = 0u;
            if (32 * m0 < NEc) seg_claim<false>(x, pk, m0, nl, vmin, scale, s_cnt, s_wl, n_wl, lt_mask);
        }
    } else {
#pragma unroll
        for (int m0 = 0; m0 < kSegRounds; m0 += kSegBatch) {
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) pk[m0 + j] = 0u;
            if (32 * m0 < NEc) seg_claim<true>(x, pk, m0, nl, vmin, scale, s_cnt, s_wl, n_wl, lt_mask);
        }
    }
    __syncwarp();

    // ---- 3. exclusive scan: lane l owns words 32 l .. 32 l + 31 (at 33 l + i); low halves = buckets < 1024 come first ----
    {
        const uint32_t a0 = s_cnt + 4u * (33u * lane);
        uint32_t tot = 0u;
#pragma unroll
        for (int i = 0; i < 32; i++) tot += lds_u32(a0 + 4u * i);     // two 16-bit sums per add: neither can carry (<= 1024)
        uint32_t incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        const uint32_t all = __shfl_sync(0xffffffffu, incl, 31);
        uint32_t carry = (incl - tot) + ((all & 0xffffu) << 16);      // high halves start after every low-half bucket
#pragma unroll
        for (int i = 0; i < 32; i++) {
            const uint32_t wv = lds_u32(a0 + 4u * i);
            sts_u32(a0 + 4u * i, carry);
            carry += wv;
        }
    }
    __syncwarp();

    // ---- 4. scatter (value, local row) to the sorted position; exact order inside the work-list buckets ----
#pragma unroll
    for (int m0 = 0; m0 < kSegRounds; m0 += kSegBatch) {
        if (32 * m0 < NEc) {                                       // warp-uniform
            uint32_t bw[kSegBatch];
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) bw[j] = lds_u32(s_cnt + ((pk[m0 + j] >> 9) & ~3u));   // the batch's base lookups overlap
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) {
                if (nl > 32 * (m0 + j)) {
                    const uint32_t pos = ((bw[j] >> ((pk[m0 + j] >> 6) & 16u)) & 0xffffu) + (pk[m0 + j] & 1023u);
                    sts_f32(s_sv + 4u * pos, x[m0 + j]);
                    const uint32_t row_all = ((uint32_t)(32 * (m0 + j) + lane) * (uint32_t)geo.ny_magic) >> 16;
                    sts_u8(s_rw + pos, cand ? (rw4[(m0 + j) >> 2] >> (8 * ((m0 + j) & 3))) & 0xffu : row_all);
                }
            }
        }
    }
    __syncwarp();
    {
        int n_long = 0;
        for (int q0 = 0; q0 < n_wl; q0 += 32) {
            const int q = q0 + lane;
            bool is_long = false;
            uint32_t desc = 0u;
            if (q < n_wl) {
                const uint32_t b = lds_u16(s_wl + 2u * q);
                const int i0 = seg_bucket_base(s_cnt, b), i1 = seg_bucket_base(s_cnt, b + 1u);
                if (i1 - i0 > kSegLongRun) { is_long = true; desc = (uint32_t)i0 | ((uint32_t)i1 << 16); }
                else if (i1 - i0 == 2) {                          // the common case: one compare, maybe one swap
                    const float v0 = lds_f32(s_sv + 4u * i0), v1 = lds_f32(s_sv + 4u * i0 + 4u);
                    if (v0 > v1) {
                        const uint32_t r0 = lds_u8(s_rw + i0), r1 = lds_u8(s_rw + i0 + 1);
                        sts_f32(s_sv + 4u * i0, v1); sts_f32(s_sv + 4u * i0 + 4u, v0);
                        sts_u8(s_rw + i0, r1); sts_u8(s_rw + i0 + 1, r0);
                    }
                } else {
                    for (int a = i0 + 1; a < i1; a++) {
                        const float ka = lds_f32(s_sv + 4u * a);
                        const uint32_t ra = lds_u8(s_rw + a);
                        int bpos = a;
                        while (bpos > i0) {
                            const float kb = lds_f32(s_sv + 4u * (bpos - 1));
                            if (kb <= ka) break;
                            sts_f32(s_sv + 4u * bpos, kb);
                            sts_u8(s_rw + bpos, lds_u8(s_rw + bpos - 1));
                            bpos--;
                        }
                        sts_f32(s_sv + 4u * bpos, ka);
                        sts_u8(s_rw + bpos, ra);
                    }
                }
            }
            const uint32_t lm = __ballot_sync(0xffffffffu, is_long);
            if (is_long) sts_u32(s_long + 4u * (n_long + __popc(lm & ((1u << lane) - 1u))), desc);   // <= 1024 / 33 = 31 long runs
            n_long += __popc(lm);
        }
        __syncwarp();
        // long runs (ties, fill values, an outlier squeezing the rest into one bucket): nothing to do when already in
        // order, else a warp-wide counting rank through the (now dead) counter and work-list areas
        for (int r = 0; r < n_long; r++) {
            const uint32_t desc = lds_u32(s_long + 4u * r);
            const int i0 = (int)(desc & 0xffffu), i1 = (int)(desc >> 16), L = i1 - i0;
            bool bad = false;
            for (int i = i0 + lane; i + 1 < i1; i += 32) bad |= lds_f32(s_sv + 4u * i) > lds_f32(s_sv + 4u * (i + 1));
            if (!__any_sync(0xffffffffu, bad)) continue;
            for (int i = lane; i < L; i += 32) {
                const float vi = lds_f32(s_sv + 4u * (i0 + i));
                int rank = 0;
                for (int j = 0; j < L; j++) {
                    const float vj = lds_f32(s_sv + 4u * (i0 + j));
                    rank += (vj < vi || (vj == vi && j < i)) ? 1 : 0;
                }
                sts_f32(s_cnt + 4u * rank, vi);
                sts_u8(s_wl + rank, lds_u8(s_rw + i0 + i));
            }
            __syncwarp();
            for (int i = lane; i < L; i += 32) {
                sts_f32(s_sv + 4u * (i0 + i), lds_f32(s_cnt + 4u * i));
                sts_u8(s_rw + i0 + i, lds_u8(s_wl + i));
            }
            __syncwarp();
        }
    }
    __syncwarp();

    // ---- 5. row bitmaps over the sorted positions -> PB (in place, lane = word) and cum (lane = row) ----
    const int R = (NE * geo.ny_magic) >> 16;                      // rows of this segment (NE = R * n_y)
    for (int i = lane; i < kSegRowsMax * kSegPst; i += 32) sts_u32(s_pb + 4u * i, 0u);
    __syncwarp();
#pragma unroll
    for (int m0 = 0; m0 < kSegRounds; m0 += kSegBatch) {
        if (32 * m0 < NEc) {                                       // warp-uniform
            uint32_t rr[kSegBatch];
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) rr[j] = lds_u8(s_rw + 32 * (m0 + j) + lane);
#pragma unroll
            for (int j = 0; j < kSegBatch; j++)
                if (nl > 32 * (m0 + j)) reds_or(s_pb + 4u * (rr[j] * kSegPst + (m0 + j)), 1u << lane);
        }
    }
    __syncwarp();
    {
        uint32_t acc = 0u;
        for (int i = 0; i < R; i++) {
            const uint32_t a = s_pb + 4u * (i * kSegPst + lane), t = lds_u32(a);
            sts_u32(a, acc);
            acc |= t;
        }
        sts_u32(s_pb + 4u * (R * kSegPst + lane), acc);
    }
    __syncwarp();
    if (lane <= R) {
        uint32_t run = 0u;
#pragma unroll 8
        for (int w = 0; w < 32; w++) {
            sts_u16(s_cum + 2u * (lane * kSegCst + w), run);
            run += __popc(lds_u32(s_pb + 4u * (lane * kSegPst + w)));
        }
        sts_u16(s_cum + 2u * (lane * kSegCst + 32), run);          // all of them
    }
    __syncwarp();

    // ---- 6. queries: one (day of the segment, percentile) per lane, two rounds of 32 queries in flight ----
    const int L_ninf = n_ninf, L_fin = NE - n_nan - n_pinf, L_pinf = NE - n_nan;   // where the finite / +inf / NaN samples begin
    const int d0 = sg * geo.S, nd = min(n_doy, d0 + geo.S) - d0;
    const unsigned char *wbase = smem_raw + (size_t)warp * kSegWarpBytes;
    const float *sv_p = (const float *)(wbase + kSegOffSv);
    const uint32_t *pb_p = (const uint32_t *)(wbase + kSegOffCnt);
    const uint16_t *cum_p = (const uint16_t *)(wbase + kSegOffRw);
    double *out_c = out + cell * n_doy * (int64_t)P;

    auto answer = [&](int dl, int p) {
        const int d = d0 + dl;
        const uint4 rg = doy_rng[d];
        const int n1 = (int)byte_of(rg, 0), n2 = (int)byte_of(rg, 1);
        const int pos_lo = s_sel.pos_lo[p], pos_hi = s_sel.pos_hi[p], mode = s_sel.mode[p];
        int lr_lo, lr_hi, w_nan = 0, w_pinf = 0, w_ninf = 0;
        if (n1 == 1 && n2 == 0) {                                 // one contiguous run of rows, each pooled once (almost every day)
            SegWin<1> win;
            const uint32_t r0 = byte_of(rg, 2), r1 = byte_of(rg, 5);
            win.ca[0] = cum_p + r1 * kSegCst; win.cb[0] = cum_p + r0 * kSegCst;
            win.pa[0] = pb_p + r1 * kSegPst; win.pb[0] = pb_p + r0 * kSegPst;
            win.n1 = 1; win.nr = 1;
            const int off = cand ? n - win.before(32) : 0;        // the window's members below tau
            seg_pick<1>(win, pos_lo - off, pos_hi - off, lr_lo, lr_hi);
            if (nonfinite) {
                const int b_pinf = seg_below<1>(win, L_pinf, n);
                w_ninf = seg_below<1>(win, L_ninf, n);
                w_pinf = b_pinf - seg_below<1>(win, L_fin, n);
                w_nan = n - b_pinf;
            }
        } else {
            SegWin<kSegRanges> win;
            win.n1 = n1; win.nr = n1 + n2;
#pragma unroll
            for (int k = 0; k < kSegRanges; k++) {
                // slot k: k < n1 -> bytes 2+k / 5+k, else the (k - n1)-th pooled-twice range -> bytes 8+.. / 10+..
                uint32_t r0 = 0u, r1 = 0u;
#pragma unroll
                for (int j = 0; j < 3; j++) if (k == j && j < n1) { r0 = byte_of(rg, 2 + j); r1 = byte_of(rg, 5 + j); }
#pragma unroll
                for (int j = 0; j < 2; j++) if (k == n1 + j && j < n2) { r0 = byte_of(rg, 8 + j); r1 = byte_of(rg, 10 + j); }
                win.ca[k] = cum_p + r1 * kSegCst; win.cb[k] = cum_p + r0 * kSegCst;
                win.pa[k] = pb_p + r1 * kSegPst; win.pb[k] = pb_p + r0 * kSegPst;
            }
            const int off = cand ? n - win.before(32) : 0;
            seg_pick<kSegRanges>(win, pos_lo - off, pos_hi - off, lr_lo, lr_hi);
            if (nonfinite) {
                const int b_pinf = seg_below<kSegRanges>(win, L_pinf, n);
                w_ninf = seg_below<kSegRanges>(win, L_ninf, n);
                w_pinf = b_pinf - seg_below<kSegRanges>(win, L_fin, n);
                w_nan = n - b_pinf;
            }
        }
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
        const double lower = (double)sv_p[lr_lo], upper = (double)sv_p[lr_hi];
        double v;
        if (mode == kSelInterp) {                                 // arraymath.py:1697-1701
            v = __dadd_rn(__dmul_rn(lower, s_sel.w_lo[p]), __dmul_rn(upper, s_sel.w_hi[p]));
        } else if (mode == kSelMax) {                             // arraymath.py:1669-1675
            v = upper;
            if ((w_pinf | w_ninf) && isinf(v)) v = nan;
        } else {                                                  // arraymath.py:1678-1695
            v = lower;
            if (w_pinf | w_ninf) {
                const int n_fin = n - (w_pinf + w_ninf);
                if (n_fin == 0) v = nan;
                if (w_pinf == 1 && n == 2) v = nan;
                if (w_ninf > 1) v = nan;
                if (n_fin == 1 && w_pinf > 1 && w_ninf != 1) v = nan;
            }
        }
        if (w_nan > 0) v = nan;                                   // _can_collect_percentiles, arraymath.py:1714
        out_c[d * P + p] = v;
    };

    // both queries of a lane on the common path (one run of rows, plain interpolation, finite samples): worked on together
    auto answer2 = [&](int dl_a, int p_a, int dl_b, int p_b) -> bool {
        const uint4 rg_a = doy_rng[d0 + dl_a], rg_b = doy_rng[d0 + dl_b];
        const int lo_a = s_sel.pos_lo[p_a], hi_a = s_sel.pos_hi[p_a], lo_b = s_sel.pos_lo[p_b], hi_b = s_sel.pos_hi[p_b];
        const bool plain = (rg_a.x & 0xffffu) == 1u && (rg_b.x & 0xffffu) == 1u && s_sel.mode[p_a] == kSelInterp && s_sel.mode[p_b] == kSelInterp &&
                           hi_a - lo_a <= 1 && hi_b - lo_b <= 1;
        if (!plain) return false;
        SegWin<1> wa, wb;
        const uint32_t r0a = byte_of(rg_a, 2), r1a = byte_of(rg_a, 5), r0b = byte_of(rg_b, 2), r1b = byte_of(rg_b, 5);
        wa.ca[0] = cum_p + r1a * kSegCst; wa.cb[0] = cum_p + r0a * kSegCst; wa.pa[0] = pb_p + r1a * kSegPst; wa.pb[0] = pb_p + r0a * kSegPst;
        wb.ca[0] = cum_p + r1b * kSegCst; wb.cb[0] = cum_p + r0b * kSegCst; wb.pa[0] = pb_p + r1b * kSegPst; wb.pb[0] = pb_p + r0b * kSegPst;
        wa.n1 = wa.nr = wb.n1 = wb.nr = 1;
        int la, ha, lb, hb;
        const int off_a = cand ? n - wa.before(32) : 0, off_b = cand ? n - wb.before(32) : 0;
        seg_pick2(wa, wb, lo_a - off_a, hi_a - off_a, lo_b - off_b, hi_b - off_b, la, ha, lb, hb);
        out_c[(d0 + dl_a) * P + p_a] = __dadd_rn(__dmul_rn((double)sv_p[la], s_sel.w_lo[p_a]), __dmul_rn((double)sv_p[ha], s_sel.w_hi[p_a]));
        out_c[(d0 + dl_b) * P + p_b] = __dadd_rn(__dmul_rn((double)sv_p[lb], s_sel.w_lo[p_b]), __dmul_rn((double)sv_p[hb], s_sel.w_hi[p_b]));
        return true;
    };

    const int q_dl = 32 / P, q_p = 32 - q_dl * P;                // one round of 32 queries further: q_dl days and q_p percentiles
    int dl = lane / P, p = lane - dl * P;
    const int nq = nd * P;
    for (int qi = lane; qi < nq; qi += 64) {
        int dl2 = dl + q_dl, p2 = p + q_p;
        if (p2 >= P) { p2 -= P; dl2++; }
        const bool two = qi + 32 < nq;
        if (!(two && !nonfinite && answer2(dl, p, dl2, p2))) {
            answer(dl, p);
            if (two) answer(dl2, p2);
        }
        dl = dl2 + q_dl; p = p2 + q_p;
        if (p >= P) { p -= P; dl++; }
    }
    }();
    if (from_list) __syncthreads();                               // the next item's gather overwrites the tiles
    }
}

// ----------------------------------------------------------------------------------------------------
// k_thr_cand: the register- and shared-memory-light variant of k_thr_seg for the candidate path (high quantiles, finite
// samples), 24 warps per SM instead of 16 - k_thr_seg is bound by latency at its occupancy.  Phase 1 streams over the tile
// instead of holding it in 32 registers per lane, the candidates (at most kLCap = 512: 16 rounds) are compacted into their
// own area, and the dead tile then takes the counters.  A warp whose segment has non-finite samples or more candidates
// sets its bit in handed_over[block]; k_thr_seg runs behind this kernel for exactly those warps.
// ----------------------------------------------------------------------------------------------------
constexpr int kLRounds = 24, kLCap = 32 * kLRounds;
constexpr int kLOffTile = 0;                                      // f32 [1024] tile -> u32 [1056] counters -> PB [32][33]
constexpr int kLOffSv = 4224;                                     // f32 [512] candidates, then the sorted values
constexpr int kLOffRw = kLOffSv + 4 * kLCap;                      // u8 [512] rows | u16 [256] work list | u32 [..] long runs; then cum u16 [32][34]
constexpr int kLOffWl = kLOffRw + kLCap;
constexpr int kLOffLong = kLOffWl + kLCap;
constexpr int kLWarpBytes = kLOffRw + kSegRowsMax * kSegCst * 2 + 16;          // = 16 (mod 128)
static_assert(kLOffLong + 64 <= kLOffRw + kSegRowsMax * kSegCst * 2, "work areas do not fit under cum");
static_assert(kLWarpBytes % 128 == 16, "tile rows of the 8 warps must start in different banks");

// seg_row_top plus the row's maximum (into vmax) and whether the row holds a NaN or an infinity (into odd)
template <int M>
__device__ __forceinline__ float seg_row_top_chk(uint32_t a0, int n_y, float &vmax, bool &odd)
{
    const float pinf = __int_as_float(0x7f800000);
    float t[M];
#pragma unroll
    for (int i = 0; i < M; i++) t[i] = -pinf;
#pragma unroll 2
    for (int y = 0; y < n_y; y++) {
        float v = lds_f32(a0 + 4u * y);
        odd |= !(fabsf(v) < pinf);
#pragma unroll
        for (int i = 0; i < M; i++) { const float hi = fmaxf(t[i], v); v = fminf(t[i], v); t[i] = hi; }
    }
    vmax = t[0];
    return t[M - 1];
}

__global__ void __launch_bounds__(kSegWarps * 32, 3)
k_thr_cand(const float *__restrict__ temps, int64_t C, int64_t ld_t,
          const int *__restrict__ seg_time, const int *__restrict__ seg_ne, const uint4 *__restrict__ doy_rng,
          const __grid_constant__ SegGeom geo, const __grid_constant__ SelTable sel, int P, int n, int n_doy,
          double *__restrict__ out, uint32_t *__restrict__ handed_over)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ SelShared s_sel;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // block -> (chunk of cell groups, segment, cell group): blocks in flight share the segment's time rows, and the
    // halo rows a chunk's neighbouring segments read again are still in L2
    const int per_chunk = geo.n_seg * geo.gc;
    const int chunk = blockIdx.x / per_chunk, rem_b = blockIdx.x - chunk * per_chunk;
    const int gcc = min(geo.gc, geo.n_groups - chunk * geo.gc);   // cell groups of this chunk
    const int sg = rem_b / gcc, group = chunk * geo.gc + (rem_b - sg * gcc);
    if (sg >= geo.n_seg) return;                                  // block-uniform (the last chunk is smaller), before any barrier
    const int64_t c0 = (int64_t)group * kSegWarps;
    const int NE = seg_ne[sg];

    for (int i = tid; i < P; i += kSegWarps * 32) {
        s_sel.pos_lo[i] = sel.pos_lo[i]; s_sel.pos_hi[i] = sel.pos_hi[i]; s_sel.mode[i] = sel.mode[i];
        s_sel.w_lo[i] = sel.w_lo[i]; s_sel.w_hi[i] = sel.w_hi[i];
    }
    // ---- G. gather the [cells x NE] tile: lanes 8j .. 8j+7 read the 8 cells of one time step ----
    {
        const int *st = seg_time + (size_t)sg * kSegCap;
        const int cl = tid & (kSegWarps - 1);
        const float *src = temps + min(c0 + cl, C - 1);
        float *dst = (float *)(smem_raw + (size_t)cl * kLWarpBytes + kLOffTile);
        const uint32_t s_dst = smem_u32(dst);
#pragma unroll 8
        for (int k = tid / kSegWarps; k < NE; k += 32)            // asynchronous 4-byte copies: every load of the tile is in flight at once
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s_dst + 4u * k), "l"(src + (int64_t)st[k] * ld_t) : "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
    }
    __syncthreads();                                              // the only block-wide barrier
    const int64_t cell = c0 + warp;
    if (cell >= C) return;                                        // warp-uniform

    const uint32_t s_base = smem_u32(smem_raw + (size_t)warp * kLWarpBytes);
    const uint32_t s_tile = s_base + kLOffTile, s_sv = s_base + kLOffSv, s_cnt = s_tile, s_pb = s_cnt, s_rw = s_base + kLOffRw,
                   s_wl = s_base + kLOffWl, s_long = s_base + kLOffLong, s_cum = s_rw;

    // ---- 1. lanes = rows: the row's cand_m largest samples (tau = the smallest of the rows' cand_m-th largest, the
    //         maximum = the largest of the rows' largest), non-finite census; nothing is kept in registers yet ----
    const float pinf = __int_as_float(0x7f800000);
    const bool nonfinite = false;                                 // (segments with NaN / inf samples are handed over)
    const bool cand = true;
    const int n_nan = 0, n_pinf = 0, n_ninf = 0;
    auto hand_over = [&]() {                                      // [count, flags[n_blocks], list[n_blocks]]
        if (lane == 0 && atomicOr(&handed_over[1 + blockIdx.x], 1u << warp) == 0u)
            handed_over[1 + gridDim.x + atomicAdd(&handed_over[0], 1u)] = blockIdx.x;
    };
    float vmax = -pinf, vmin;
    int NEc;
    float x[kLRounds];
    uint32_t rw4[kLRounds / 4];
    {
        const int R0 = (NE * geo.ny_magic) >> 16;
        float tau = pinf;
        bool odd = false;
        if (lane < R0) {
            const uint32_t a0 = s_tile + 4u * (uint32_t)(lane * geo.n_y);
            switch (geo.cand_m) {                                 // warp-uniform
            case 1: tau = seg_row_top_chk<1>(a0, geo.n_y, vmax, odd); break;
            case 2: tau = seg_row_top_chk<2>(a0, geo.n_y, vmax, odd); break;
            case 3: tau = seg_row_top_chk<3>(a0, geo.n_y, vmax, odd); break;
            case 4: tau = seg_row_top_chk<4>(a0, geo.n_y, vmax, odd); break;
            case 5: tau = seg_row_top_chk<5>(a0, geo.n_y, vmax, odd); break;
            case 6: tau = seg_row_top_chk<6>(a0, geo.n_y, vmax, odd); break;
            case 7: tau = seg_row_top_chk<7>(a0, geo.n_y, vmax, odd); break;
            default: tau = seg_row_top_chk<8>(a0, geo.n_y, vmax, odd); break;
            }
        }
        if (__any_sync(0xffffffffu, odd)) { hand_over(); return; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            tau = fminf(tau, __shfl_xor_sync(0xffffffffu, tau, o));
            vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
        }

        // ---- 1b. candidate filter (see k_thr_seg): the samples >= tau, packed in tile order into their own area ----
        int base = 0;
        const uint32_t lt = (1u << lane) - 1u;
#pragma unroll 4
        for (int m = 0; 32 * m < NE; m++) {
            const float v = lds_f32(s_tile + 4u * (32 * m + lane));
            const bool keep = 32 * m + lane < NE && v >= tau;
            const uint32_t bal = __ballot_sync(0xffffffffu, keep);
            const uint32_t pos = (uint32_t)base + __popc(bal & lt);
            if (keep && pos < (uint32_t)kLCap) {
                sts_f32(s_sv + 4u * pos, v);
                sts_u8(s_rw + pos, ((uint32_t)(32 * m + lane) * (uint32_t)geo.ny_magic) >> 16);
            }
            base += __popc(bal);
        }
        NEc = base;
        if (NEc > kLCap) { hand_over(); return; }                 // warp-uniform: more candidates than this kernel orders
        vmin = tau;
        __syncwarp();                                             // the tile is dead: its place takes the counters
        for (int i = lane; i < 1024 + 32; i += 32) sts_u32(s_cnt + 4u * i, 0u);
#pragma unroll
        for (int m = 0; m < kLRounds; m++) {
            if ((m & 3) == 0) rw4[m >> 2] = 0u;
            const bool have = NEc - lane > 32 * m;
            x[m] = have ? lds_f32(s_sv + 4u * (32 * m + lane)) : 0.0f;
            rw4[m >> 2] |= (have ? lds_u8(s_rw + 32 * m + lane) : 0u) << (8 * (m & 3));
        }
        __syncwarp();
    }

    // ---- 2. monotone buckets; one atomic claims the slot inside the bucket ----
    const float range = vmax - vmin;
    const float scale = (range > 0.0f && range < pinf) ? (float)(kSegNBF - 1) / range : 0.0f;
    uint32_t pk[kLRounds];                                      // where the counter is | slot
    int n_wl = 0;                                                 // warp-uniform
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int nl = NEc - lane;                                     // round m holds a sample of this lane iff nl > 32 m
    if (!nonfinite) {
#pragma unroll
        for (int m0 = 0; m0 < kLRounds; m0 += kSegBatch) {
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) pk[m0 + j] = 0u;
            if (32 * m0 < NEc) seg_claim<false>(x, pk, m0, nl, vmin, scale, s_cnt, s_wl, n_wl, lt_mask);
        }
    } else {
#pragma unroll
        for (int m0 = 0; m0 < kLRounds; m0 += kSegBatch) {
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) pk[m0 + j] = 0u;
            if (32 * m0 < NEc) seg_claim<true>(x, pk, m0, nl, vmin, scale, s_cnt, s_wl, n_wl, lt_mask);
        }
    }
    __syncwarp();

    // ---- 3. exclusive scan: lane l owns words 32 l .. 32 l + 31 (at 33 l + i); low halves = buckets < 1024 come first ----
    {
        const uint32_t a0 = s_cnt + 4u * (33u * lane);
        uint32_t tot = 0u;
#pragma unroll
        for (int i = 0; i < 32; i++) tot += lds_u32(a0 + 4u * i);     // two 16-bit sums per add: neither can carry (<= 1024)
        uint32_t incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        const uint32_t all = __shfl_sync(0xffffffffu, incl, 31);
        uint32_t carry = (incl - tot) + ((all & 0xffffu) << 16);      // high halves start after every low-half bucket
#pragma unroll
        for (int i = 0; i < 32; i++) {
            const uint32_t wv = lds_u32(a0 + 4u * i);
            sts_u32(a0 + 4u * i, carry);
            carry += wv;
        }
    }
    __syncwarp();

    // ---- 4. scatter (value, local row) to the sorted position; exact order inside the work-list buckets ----
#pragma unroll
    for (int m0 = 0; m0 < kLRounds; m0 += kSegBatch) {
        if (32 * m0 < NEc) {                                       // warp-uniform
            uint32_t bw[kSegBatch];
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) bw[j] = lds_u32(s_cnt + ((pk[m0 + j] >> 9) & ~3u));   // the batch's base lookups overlap
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) {
                if (nl > 32 * (m0 + j)) {
                    const uint32_t pos = ((bw[j] >> ((pk[m0 + j] >> 6) & 16u)) & 0xffffu) + (pk[m0 + j] & 1023u);
                    sts_f32(s_sv + 4u * pos, x[m0 + j]);
                    const uint32_t row_all = ((uint32_t)(32 * (m0 + j) + lane) * (uint32_t)geo.ny_magic) >> 16;
                    sts_u8(s_rw + pos, cand ? (rw4[(m0 + j) >> 2] >> (8 * ((m0 + j) & 3))) & 0xffu : row_all);
                }
            }
        }
    }
    __syncwarp();
    {
        int n_long = 0;
        for (int q0 = 0; q0 < n_wl; q0 += 32) {
            const int q = q0 + lane;
            bool is_long = false;
            uint32_t desc = 0u;
            if (q < n_wl) {
                const uint32_t b = lds_u16(s_wl + 2u * q);
                const int i0 = seg_bucket_base(s_cnt, b), i1 = seg_bucket_base(s_cnt, b + 1u);
                if (i1 - i0 > kSegLongRun) { is_long = true; desc = (uint32_t)i0 | ((uint32_t)i1 << 16); }
                else if (i1 - i0 == 2) {                          // the common case: one compare, maybe one swap
                    const float v0 = lds_f32(s_sv + 4u * i0), v1 = lds_f32(s_sv + 4u * i0 + 4u);
                    if (v0 > v1) {
                        const uint32_t r0 = lds_u8(s_rw + i0), r1 = lds_u8(s_rw + i0 + 1);
                        sts_f32(s_sv + 4u * i0, v1); sts_f32(s_sv + 4u * i0 + 4u, v0);
                        sts_u8(s_rw + i0, r1); sts_u8(s_rw + i0 + 1, r0);
                    }
                } else {
                    for (int a = i0 + 1; a < i1; a++) {
                        const float ka = lds_f32(s_sv + 4u * a);
                        const uint32_t ra = lds_u8(s_rw + a);
                        int bpos = a;
                        while (bpos > i0) {
                            const float kb = lds_f32(s_sv + 4u * (bpos - 1));
                            if (kb <= ka) break;
                            sts_f32(s_sv + 4u * bpos, kb);
                            sts_u8(s_rw + bpos, lds_u8(s_rw + bpos - 1));
                            bpos--;
                        }
                        sts_f32(s_sv + 4u * bpos, ka);
                        sts_u8(s_rw + bpos, ra);
                    }
                }
            }
            const uint32_t lm = __ballot_sync(0xffffffffu, is_long);
            if (is_long) sts_u32(s_long + 4u * (n_long + __popc(lm & ((1u << lane) - 1u))), desc);   // <= 1024 / 33 = 31 long runs
            n_long += __popc(lm);
        }
        __syncwarp();
        // long runs (ties, fill values, an outlier squeezing the rest into one bucket): nothing to do when already in
        // order, else a warp-wide counting rank through the (now dead) counter and work-list areas
        for (int r = 0; r < n_long; r++) {
            const uint32_t desc = lds_u32(s_long + 4u * r);
            const int i0 = (int)(desc & 0xffffu), i1 = (int)(desc >> 16), L = i1 - i0;
            bool bad = false;
            for (int i = i0 + lane; i + 1 < i1; i += 32) bad |= lds_f32(s_sv + 4u * i) > lds_f32(s_sv + 4u * (i + 1));
            if (!__any_sync(0xffffffffu, bad)) continue;
            for (int i = lane; i < L; i += 32) {
                const float vi = lds_f32(s_sv + 4u * (i0 + i));
                int rank = 0;
                for (int j = 0; j < L; j++) {
                    const float vj = lds_f32(s_sv + 4u * (i0 + j));
                    rank += (vj < vi || (vj == vi && j < i)) ? 1 : 0;
                }
                sts_f32(s_cnt + 4u * rank, vi);
                sts_u8(s_wl + rank, lds_u8(s_rw + i0 + i));
            }
            __syncwarp();
            for (int i = lane; i < L; i += 32) {
                sts_f32(s_sv + 4u * (i0 + i), lds_f32(s_cnt + 4u * i));
                sts_u8(s_rw + i0 + i, lds_u8(s_wl + i));
            }
            __syncwarp();
        }
    }
    __syncwarp();

    // ---- 5. row bitmaps over the sorted positions -> PB (in place, lane = word) and cum (lane = row) ----
    const int R = (NE * geo.ny_magic) >> 16;                      // rows of this segment (NE = R * n_y)
    for (int i = lane; i < kSegRowsMax * kSegPst; i += 32) sts_u32(s_pb + 4u * i, 0u);
    __syncwarp();
#pragma unroll
    for (int m0 = 0; m0 < kLRounds; m0 += kSegBatch) {
        if (32 * m0 < NEc) {                                       // warp-uniform
            uint32_t rr[kSegBatch];
#pragma unroll
            for (int j = 0; j < kSegBatch; j++) rr[j] = lds_u8(s_rw + 32 * (m0 + j) + lane);
#pragma unroll
            for (int j = 0; j < kSegBatch; j++)
                if (nl > 32 * (m0 + j)) reds_or(s_pb + 4u * (rr[j] * kSegPst + (m0 + j)), 1u << lane);
        }
    }
    __syncwarp();
    {
        uint32_t acc = 0u;
        for (int i = 0; i < R; i++) {
            const uint32_t a = s_pb + 4u * (i * kSegPst + lane), t = lds_u32(a);
            sts_u32(a, acc);
            acc |= t;
        }
        sts_u32(s_pb + 4u * (R * kSegPst + lane), acc);
    }
    __syncwarp();
    if (lane <= R) {
        uint32_t run = 0u;
#pragma unroll 8
        for (int w = 0; w < 32; w++) {
            sts_u16(s_cum + 2u * (lane * kSegCst + w), run);
            run += __popc(lds_u32(s_pb + 4u * (lane * kSegPst + w)));
        }
        sts_u16(s_cum + 2u * (lane * kSegCst + 32), run);          // all of them
    }
    __syncwarp();

    // ---- 6. queries: one (day of the segment, percentile) per lane, two rounds of 32 queries in flight ----
    const int L_ninf = n_ninf, L_fin = NE - n_nan - n_pinf, L_pinf = NE - n_nan;   // where the finite / +inf / NaN samples begin
    const int d0 = sg * geo.S, nd = min(n_doy, d0 + geo.S) - d0;
    const unsigned char *wbase = smem_raw + (size_t)warp * kLWarpBytes;
    const float *sv_p = (const float *)(wbase + kLOffSv);
    const uint32_t *pb_p = (const uint32_t *)(wbase + kLOffTile);
    const uint16_t *cum_p = (const uint16_t *)(wbase + kLOffRw);
    double *out_c = out + cell * n_doy * (int64_t)P;

    auto answer = [&](int dl, int p) {
        const int d = d0 + dl;
        const uint4 rg = doy_rng[d];
        const int n1 = (int)byte_of(rg, 0), n2 = (int)byte_of(rg, 1);
        const int pos_lo = s_sel.pos_lo[p], pos_hi = s_sel.pos_hi[p], mode = s_sel.mode[p];
        int lr_lo, lr_hi, w_nan = 0, w_pinf = 0, w_ninf = 0;
        if (n1 == 1 && n2 == 0) {                                 // one contiguous run of rows, each pooled once (almost every day)
            SegWin<1> win;
            const uint32_t r0 = byte_of(rg, 2), r1 = byte_of(rg, 5);
            win.ca[0] = cum_p + r1 * kSegCst; win.cb[0] = cum_p + r0 * kSegCst;
            win.pa[0] = pb_p + r1 * kSegPst; win.pb[0] = pb_p + r0 * kSegPst;
            win.n1 = 1; win.nr = 1;
            const int off = cand ? n - win.before(32) : 0;        // the window's members below tau
            seg_pick<1>(win, pos_lo - off, pos_hi - off, lr_lo, lr_hi);
            if (nonfinite) {
                const int b_pinf = seg_below<1>(win, L_pinf, n);
                w_ninf = seg_below<1>(win, L_ninf, n);
                w_pinf = b_pinf - seg_below<1>(win, L_fin, n);
                w_nan = n - b_pinf;
            }
        } else {
            SegWin<kSegRanges> win;
            win.n1 = n1; win.nr = n1 + n2;
#pragma unroll
            for (int k = 0; k < kSegRanges; k++) {
                // slot k: k < n1 -> bytes 2+k / 5+k, else the (k - n1)-th pooled-twice range -> bytes 8+.. / 10+..
                uint32_t r0 = 0u, r1 = 0u;
#pragma unroll
                for (int j = 0; j < 3; j++) if (k == j && j < n1) { r0 = byte_of(rg, 2 + j); r1 = byte_of(rg, 5 + j); }
#pragma unroll
                for (int j = 0; j < 2; j++) if (k == n1 + j && j < n2) { r0 = byte_of(rg, 8 + j); r1 = byte_of(rg, 10 + j); }
                win.ca[k] = cum_p + r1 * kSegCst; win.cb[k] = cum_p + r0 * kSegCst;
                win.pa[k] = pb_p + r1 * kSegPst; win.pb[k] = pb_p + r0 * kSegPst;
            }
            const int off = cand ? n - win.before(32) : 0;
            seg_pick<kSegRanges>(win, pos_lo - off, pos_hi - off, lr_lo, lr_hi);
            if (nonfinite) {
                const int b_pinf = seg_below<kSegRanges>(win, L_pinf, n);
                w_ninf = seg_below<kSegRanges>(win, L_ninf, n);
                w_pinf = b_pinf - seg_below<kSegRanges>(win, L_fin, n);
                w_nan = n - b_pinf;
            }
        }
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
        const double lower = (double)sv_p[lr_lo], upper = (double)sv_p[lr_hi];
        double v;
        if (mode == kSelInterp) {                                 // arraymath.py:1697-1701
            v = __dadd_rn(__dmul_rn(lower, s_sel.w_lo[p]), __dmul_rn(upper, s_sel.w_hi[p]));
        } else if (mode == kSelMax) {                             // arraymath.py:1669-1675
            v = upper;
            if ((w_pinf | w_ninf) && isinf(v)) v = nan;
        } else {                                                  // arraymath.py:1678-1695
            v = lower;
            if (w_pinf | w_ninf) {
                const int n_fin = n - (w_pinf + w_ninf);
                if (n_fin == 0) v = nan;
                if (w_pinf == 1 && n == 2) v = nan;
                if (w_ninf > 1) v = nan;
                if (n_fin == 1 && w_pinf > 1 && w_ninf != 1) v = nan;
            }
        }
        if (w_nan > 0) v = nan;                                   // _can_collect_percentiles, arraymath.py:1714
        out_c[d * P + p] = v;
    };

    // both queries of a lane on the common path (one run of rows, plain interpolation, finite samples): worked on together
    auto answer2 = [&](int dl_a, int p_a, int dl_b, int p_b) -> bool {
        const uint4 rg_a = doy_rng[d0 + dl_a], rg_b = doy_rng[d0 + dl_b];
        const int lo_a = s_sel.pos_lo[p_a], hi_a = s_sel.pos_hi[p_a], lo_b = s_sel.pos_lo[p_b], hi_b = s_sel.pos_hi[p_b];
        const bool plain = (rg_a.x & 0xffffu) == 1u && (rg_b.x & 0xffffu) == 1u && s_sel.mode[p_a] == kSelInterp && s_sel.mode[p_b] == kSelInterp &&
                           hi_a - lo_a <= 1 && hi_b - lo_b <= 1;
        if (!plain) return false;
        SegWin<1> wa, wb;
        const uint32_t r0a = byte_of(rg_a, 2), r1a = byte_of(rg_a, 5), r0b = byte_of(rg_b, 2), r1b = byte_of(rg_b, 5);
        wa.ca[0] = cum_p + r1a * kSegCst; wa.cb[0] = cum_p + r0a * kSegCst; wa.pa[0] = pb_p + r1a * kSegPst; wa.pb[0] = pb_p + r0a * kSegPst;
        wb.ca[0] = cum_p + r1b * kSegCst; wb.cb[0] = cum_p + r0b * kSegCst; wb.pa[0] = pb_p + r1b * kSegPst; wb.pb[0] = pb_p + r0b * kSegPst;
        wa.n1 = wa.nr = wb.n1 = wb.nr = 1;
        int la, ha, lb, hb;
        const int off_a = cand ? n - wa.before(32) : 0, off_b = cand ? n - wb.before(32) : 0;
        seg_pick2(wa, wb, lo_a - off_a, hi_a - off_a, lo_b - off_b, hi_b - off_b, la, ha, lb, hb);
        out_c[(d0 + dl_a) * P + p_a] = __dadd_rn(__dmul_rn((double)sv_p[la], s_sel.w_lo[p_a]), __dmul_rn((double)sv_p[ha], s_sel.w_hi[p_a]));
        out_c[(d0 + dl_b) * P + p_b] = __dadd_rn(__dmul_rn((double)sv_p[lb], s_sel.w_lo[p_b]), __dmul_rn((double)sv_p[hb], s_sel.w_hi[p_b]));
        return true;
    };

    const int q_dl = 32 / P, q_p = 32 - q_dl * P;                // one round of 32 queries further: q_dl days and q_p percentiles
    int dl = lane / P, p = lane - dl * P;
    const int nq = nd * P;
    for (int qi = lane; qi < nq; qi += 64) {
        int dl2 = dl + q_dl, p2 = p + q_p;
        if (p2 >= P) { p2 -= P; dl2++; }
        const bool two = qi + 32 < nq;
        if (!(two && !nonfinite && answer2(dl, p, dl2, p2))) {
            answer(dl, p);
            if (two) answer(dl2, p2);
        }
        dl = dl2 + q_dl; p = p2 + q_p;
        if (p >= P) { p -= P; dl++; }
    }
}

static bool bad_dims(int64_t C, int64_t T_b, int n_doy, int n_y, int W, int P)
{
    return C < 0 || T_b < 0 || n_doy <= 0 || n_y <= 0 || W <= 0 || P <= 0 || T_b > 0x3fffffff;
}

// What k_thr_ranked needs besides the reference's two tables.
struct RankedPlan {
    bool usable = false;
    std::vector<int> op_off, ops;       // per day of year: (row << 1 | enter) ops relative to the previous day of the warp's range
    std::vector<uint8_t> doy_dup;       // window pools some row twice
    int dpw = 0, ept = 0, nwords_pad = 0;
    size_t smem = 0;
    SelTable sel;
};

static size_t ranked_smem(int E)
{
    const size_t Epad = ((size_t)E + 63) & ~(size_t)63;
    return Epad * (4 + 2 + 4 + 2) + (size_t)kRadixBins * kRankedThreads * 2;
}

// positions and weights: numba/np/arraymath.py:1655-1704 with n fixed (every window pools W * n_y samples)
static void fill_sel(SelTable &sel, int64_t n, const double *q, int P)
{
    for (int p = 0; p < HDP_B200_MAX_PERCENTILES; p++) {
        sel.pos_lo[p] = sel.pos_hi[p] = 0;
        sel.mode[p] = kSelInterp;
        sel.w_lo[p] = sel.w_hi[p] = 0.0;
        if (p >= P) continue;
        volatile double pct = q[p] * 100.0;
        if (pct == 100.0) { sel.mode[p] = kSelMax; sel.pos_lo[p] = sel.pos_hi[p] = (int)n - 1; continue; }
        if (pct == 0.0) { sel.mode[p] = kSelMin; continue; }
        volatile double frac = pct / 100.0;
        volatile double scaled = (double)(n - 1) * frac;
        volatile double rank = 1.0 + scaled;
        const double f = floor(rank);
        volatile double m = rank - f;
        volatile double w0 = 1.0 - m;
        int64_t k = (int64_t)f - 1;
        if (k < 0) k = 0;
        if (k >= n - 1) { sel.pos_lo[p] = sel.pos_hi[p] = (int)n - 1; }
        else { sel.pos_lo[p] = (int)k; sel.pos_hi[p] = (int)k + 1; }
        sel.w_lo[p] = w0;
        sel.w_hi[p] = m;
    }
    for (int w = 0; w < 64; w++) sel.b_slot[w] = -1;
}

static void plan_ranked(const int32_t *win_rows, int n_doy, int n_y, int W, const double *q, int P, RankedPlan &pl)
{
    const int64_t E = (int64_t)n_doy * n_y, n = (int64_t)W * n_y;
    pl.usable = false;
    if (E > 65535 || n < 2) return;
    pl.smem = ranked_smem((int)E);
    if (pl.smem > 227 * 1024 - 256) return;
    const int nwords = (int)((E + 31) / 32);
    pl.nwords_pad = (nwords + 31) / 32 * 32;
    pl.dpw = (n_doy + kRankedWarps - 1) / kRankedWarps;
    pl.ept = (int)((E + kRankedThreads - 1) / kRankedThreads) | 1;          // odd: conflict-free strided key reads
    pl.doy_dup.assign(n_doy, 0);
    pl.op_off.assign(n_doy + 1, 0);
    pl.ops.clear();
    std::vector<int> cur(n_doy), prev(n_doy);
    for (int d = 0; d < n_doy; d++) {
        std::fill(cur.begin(), cur.end(), 0);
        for (int k = 0; k < W; k++) cur[win_rows[d * W + k]]++;
        for (int r = 0; r < n_doy; r++) {
            if (cur[r] > 2) return;                                         // more than twice: generic kernel
            if (cur[r] == 2) pl.doy_dup[d] = 1;
        }
        const bool first = d % pl.dpw == 0;
        pl.op_off[d] = (int)pl.ops.size();
        for (int r = 0; r < n_doy; r++) {
            const int before = first ? 0 : prev[r];
            for (int i = cur[r]; i < before; i++) pl.ops.push_back(r << 1);        // leaves first ...
        }
        for (int r = 0; r < n_doy; r++) {
            const int before = first ? 0 : prev[r];
            for (int i = before; i < cur[r]; i++) pl.ops.push_back((r << 1) | 1);  // ... then enters
        }
        prev.swap(cur);
    }
    pl.op_off[n_doy] = (int)pl.ops.size();
    fill_sel(pl.sel, n, q, P);
    int n_b = 0;
    for (int w = 0; w < 64; w++) {
        bool need = false;
        for (int d = w * pl.dpw; d < std::min(n_doy, (w + 1) * pl.dpw); d++) need |= pl.doy_dup[d] != 0;
        if (need && w < kRankedWarps) pl.sel.b_slot[w] = (int8_t)n_b++;
    }
    if ((size_t)pl.nwords_pad * (kRankedWarps * 6 + n_b * 4) > pl.smem - (((size_t)E + 63) & ~(size_t)63) * 6) return;
    pl.usable = true;
}

// ---- the segment path (k_thr_seg) ----
struct SegPlan {
    bool usable = false;
    SegGeom geo;
    std::vector<int> seg_time;          // [n_seg][kSegCap] time index of every sample slot (local row major), pads resolved
    std::vector<int> seg_ne;            // [n_seg] samples per segment = rows * n_y
    std::vector<uint8_t> doy_rng;       // [n_doy][16]: n1, n2, lo[3], hi[3], lo2[2], hi2[2] in local rows of the day's segment
};

static bool plan_seg_try(const int32_t *time_index, const int32_t *win_rows, int64_t T_b, int n_doy, int n_y, int W, int S, SegPlan &sp)
{
    const int n_seg = (n_doy + S - 1) / S;
    sp.seg_time.assign((size_t)n_seg * kSegCap, 0);
    sp.seg_ne.assign(n_seg, 0);
    sp.doy_rng.assign((size_t)n_doy * 16, 0);
    std::vector<int> present(n_doy), loc(n_doy), mult;
    for (int sg = 0; sg < n_seg; sg++) {
        const int d0 = sg * S, d1 = std::min(n_doy, d0 + S);
        std::fill(present.begin(), present.end(), 0);
        for (int d = d0; d < d1; d++)
            for (int k = 0; k < W; k++) present[win_rows[d * W + k]] = 1;
        std::vector<int> r;
        for (int i = 0; i < n_doy; i++) if (present[i]) r.push_back(i);
        const int m = (int)r.size();
        if (m + 1 > kSegRowsMax || (int64_t)m * n_y > kSegCap) return false;
        // start the local order after the widest circular gap: a window is then a few runs of consecutive local rows
        int start = 0, best = -1;
        for (int i = 0; i < m; i++) {
            const int gap = m == 1 ? n_doy : (r[(i + 1) % m] - r[i] + n_doy) % n_doy;
            if (gap > best) { best = gap; start = (i + 1) % m; }
        }
        for (int k = 0; k < m; k++) {
            const int row = r[(start + k) % m];
            loc[row] = k;
            for (int j = 0; j < n_y; j++) {
                int64_t t = time_index[(size_t)row * n_y + j];
                if (t < 0) t += T_b;                                        // -1 pads read the LAST sample (threshold.py:35,77)
                sp.seg_time[(size_t)sg * kSegCap + (size_t)k * n_y + j] = (int)t;
            }
        }
        sp.seg_ne[sg] = m * n_y;
        for (int d = d0; d < d1; d++) {
            mult.assign(m + 1, 0);
            for (int k = 0; k < W; k++) mult[loc[win_rows[d * W + k]]]++;
            uint8_t *g = &sp.doy_rng[(size_t)d * 16];
            int n1 = 0, n2 = 0;
            for (int k = 0; k < m; k++) {
                if (mult[k] > 2) return false;                              // pooled more than twice: not this path
                if (mult[k] >= 1 && (k == 0 || mult[k - 1] == 0)) {         // a run of rows pooled at least once starts
                    if (n1 == 3) return false;
                    int e = k;
                    while (e < m && mult[e] >= 1) e++;
                    g[2 + n1] = (uint8_t)k; g[5 + n1] = (uint8_t)e; n1++;
                }
                if (mult[k] == 2 && (k == 0 || mult[k - 1] != 2)) {         // a run of rows pooled twice starts
                    if (n2 == 2) return false;
                    int e = k;
                    while (e < m && mult[e] == 2) e++;
                    g[8 + n2] = (uint8_t)k; g[10 + n2] = (uint8_t)e; n2++;
                }
            }
            g[0] = (uint8_t)n1; g[1] = (uint8_t)n2;
        }
    }
    sp.geo.S = S; sp.geo.n_seg = n_seg;
    return true;
}

static void plan_seg(const int32_t *time_index, const int32_t *win_rows, int64_t T_b, int n_doy, int n_y, int W, SegPlan &sp)
{
    sp.usable = false;
    if ((int64_t)W * n_y < 2 || n_y > kSegCap) return;
    const int magic = (65536 + n_y - 1) / n_y;
    for (int k = 0; k <= kSegCap; k++)
        if (((k * magic) >> 16) != k / n_y) return;                         // the kernel divides sample slots by n_y with one multiply
    // the largest S that fits: the ordering of a segment is shared by S days
    for (int S = std::min(n_doy, kSegRowsMax); S >= 1; S--) {
        if (2 * S < W - 1) return;                                          // more than 3x halo: k_thr_ranked does better
        if (!plan_seg_try(time_index, win_rows, T_b, n_doy, n_y, W, S, sp)) continue;
        sp.geo.ny_magic = magic;
        sp.geo.n_y = n_y;
        sp.geo.cand_m = 0;
        sp.geo.unit = 0;
        sp.usable = true;
        return;
    }
}

static int thr_chunk_groups(int64_t T_b)
{
    // cell groups per chunk: the chunk's slab of the measure array (T_b x 8 cells x 4 bytes per group) should stay in L2, so that
    // the halo rows neighbouring segments read again do not come from HBM twice; HDP_B200_THR_CHUNK_GROUPS overrides
    static int forced = -1;
    if (forced < 0) {
        const char *s = getenv("HDP_B200_THR_CHUNK_GROUPS");
        forced = s ? atoi(s) : 0;
    }
    if (forced > 0) return forced;
    int64_t g = ((int64_t)56 << 20) / std::max<int64_t>(1, T_b * kSegWarps * 4);
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, 1 << 20));
}

struct ThrLayout {
    size_t total = 0;
    float *xn = nullptr;
    int *time_index = nullptr, *win_rows = nullptr, *op_off = nullptr, *ops = nullptr;
    uint8_t *doy_dup = nullptr;
    int *seg_time = nullptr, *seg_ne = nullptr;      // k_thr_seg tables
    uint8_t *doy_rng = nullptr;
    uint32_t *handed_over = nullptr;                 // per k_thr_cand block: the warps left to k_thr_seg
    size_t handed_over_count = 0;
    NetTables net;                                   // k_thr_net tables
};

static ThrLayout carve_thr(void *ws, size_t ws_bytes, int64_t C, int64_t T_b, bool need_copy, int n_doy, int n_y, int W)
{
    ThrLayout L;
    Carver cv(ws, ws_bytes);
    if (need_copy) L.xn = cv.take<float>((size_t)C * T_b);      // transposed and / or converted copy of the samples
    L.time_index = cv.take<int>((size_t)n_doy * n_y);
    L.win_rows = cv.take<int>((size_t)n_doy * W);
    L.op_off = cv.take<int>((size_t)n_doy + 1);
    L.ops = cv.take<int>((size_t)2 * W * (n_doy + kRankedWarps));           // <= 2W changes per day, W per range start
    L.doy_dup = cv.take<uint8_t>((size_t)n_doy);
    L.seg_time = cv.take<int>((size_t)n_doy * kSegCap);                     // <= n_doy segments
    L.seg_ne = cv.take<int>((size_t)n_doy);
    L.doy_rng = cv.take<uint8_t>((size_t)n_doy * 16);
    // >= blocks of the segment kernels: a usable segment has 2 S >= W - 1 days (plan_seg), so there are at most n_doy / S_min
    const int s_min = std::max(1, W / 2);
    L.handed_over_count = (size_t)(C / kSegWarps + 2 + thr_chunk_groups(T_b)) * (size_t)((n_doy + s_min - 1) / s_min);
    L.handed_over = cv.take<uint32_t>(1 + 2 * L.handed_over_count);       // count, flags[blocks], list[blocks]
    L.net.seq_time = cv.take<int>((size_t)(n_doy + W / 2 + 1) * 32);      // k_thr_net: <= 32 samples per row, n_doy + r rows + the pad row
    L.net.win_day = cv.take<int>((size_t)n_doy + W);
    L.net.irr_day = cv.take<int>((size_t)(n_doy / 4 + 1) * W * 4);        // the irregular days' program: <= W steps per day, 4 ints each
    L.net.irr_time = cv.take<int>((size_t)(n_doy / 4 + 1) * W * 32);      // at most a quarter of the days are irregular (net_plan)
    L.net.next_item = cv.take<unsigned long long>(1);
    L.total = cv.off;
    return L;
}

static std::atomic<int> g_force_generic{0};     // 1: k_thr_generic for everything; 2: k_thr_ranked instead of k_thr_seg
static std::atomic<int> g_force_ranked{0};
static std::atomic<int> g_seg_light{1};          // test hook: 0 = the candidate path runs in k_thr_seg itself (no k_thr_cand)
static std::atomic<int> g_seg_candidates{1};     // test hook: 0 = k_thr_seg orders every sample of a segment (no candidate filter)
static std::atomic<int> g_net{1};                // test hook: 0 = no k_thr_net (the lane-per-cell network kernel, thr_net.cu)
static std::atomic<int> g_net_tmem{1};           // test hook: 0 = k_thr_net keeps every list in shared memory (no k_thr_net_tm)

// Everything that depends on the tables and quantiles only, built once per distinct (tables, quantiles) and shared by the
// calls that use them (the lock covers the lookup, not the launches: calls on different devices / streams do not serialise).
struct ThrPlans {
    std::vector<int32_t> rows, ti;
    std::vector<double> q;
    int64_t dims[4] = {0, 0, 0, 0};
    RankedPlan ranked;
    SegPlan seg;
    NetPlan net;
    SelTable sel;
};

// Plans of the (tables, quantiles) pair, built once and shared (host only: no CUDA call).
static std::shared_ptr<ThrPlans> thr_plans(const int32_t *h_time_index, const int32_t *h_win_rows, int64_t T_b, int n_doy, int n_y, int W,
                                           const double *h_q, int P, int64_t C)
{
    static std::mutex plan_mu;
    static std::shared_ptr<ThrPlans> cached;
    std::lock_guard<std::mutex> plan_lock(plan_mu);
    const int64_t b = (int64_t)W * n_y;
    const size_t n_ti = (size_t)n_doy * n_y, n_wr = (size_t)n_doy * W;
    const bool same = cached && cached->dims[0] == n_doy && cached->dims[1] == n_y && cached->dims[2] == W && cached->dims[3] == T_b &&
                      cached->rows.size() == n_wr && std::equal(cached->rows.begin(), cached->rows.end(), h_win_rows) &&
                      cached->ti.size() == n_ti && std::equal(cached->ti.begin(), cached->ti.end(), h_time_index) &&
                      cached->q.size() == (size_t)P && std::equal(cached->q.begin(), cached->q.end(), h_q);
    if (!same) {
        auto fresh = std::make_shared<ThrPlans>();
        plan_ranked(h_win_rows, n_doy, n_y, W, h_q, P, fresh->ranked);
        plan_seg(h_time_index, h_win_rows, T_b, n_doy, n_y, W, fresh->seg);
        fill_sel(fresh->sel, b, h_q, P);
        int is_max[HDP_B200_MAX_PERCENTILES], is_interp[HDP_B200_MAX_PERCENTILES];
        for (int p = 0; p < P; p++) { is_max[p] = fresh->sel.mode[p] == kSelMax; is_interp[p] = fresh->sel.mode[p] == kSelInterp; }
        net_plan(h_time_index, h_win_rows, T_b, n_doy, n_y, W, fresh->sel.pos_lo, fresh->sel.pos_hi, is_max, is_interp,
                 fresh->sel.w_lo, fresh->sel.w_hi, P, C, fresh->net);
        fresh->rows.assign(h_win_rows, h_win_rows + n_wr);
        fresh->ti.assign(h_time_index, h_time_index + n_ti);
        fresh->q.assign(h_q, h_q + P);
        fresh->dims[0] = n_doy; fresh->dims[1] = n_y; fresh->dims[2] = W; fresh->dims[3] = T_b;
        cached = fresh;
    }
    return cached;
}

int thresholds_launch(const float *d_temps, int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                      const int32_t *h_time_index, const int32_t *h_win_rows, int n_doy, int n_y, int W,
                      const double *h_q, int P, double *d_out,
                      void *d_workspace, size_t workspace_bytes, void *stream, int64_t carve_cells, bool tables_resident, int input_unit)
{
    if (bad_dims(C, T_b, n_doy, n_y, W, P) || !h_time_index || !h_win_rows || !h_q) return HDP_B200_ERR_INVALID;
    if (input_unit < 0 || input_unit > 2) return HDP_B200_ERR_INVALID;
    if (C > 0 && (!d_temps || !d_out)) return HDP_B200_ERR_INVALID;
    if (C > 0 && T_b == 0) return HDP_B200_ERR_INVALID;                      // nothing to index into
    if (P > HDP_B200_MAX_PERCENTILES) return HDP_B200_ERR_UNSUPPORTED;
    const int64_t b = (int64_t)W * n_y;
    if (b > HDP_B200_MAX_WINDOW) return HDP_B200_ERR_UNSUPPORTED;
    QTable qt;
    for (int p = 0; p < HDP_B200_MAX_PERCENTILES; p++) {
        qt.q[p] = p < P ? h_q[p] : 0.0;
        if (p < P && !(h_q[p] >= 0.0 && h_q[p] <= 1.0)) return HDP_B200_ERR_INVALID;   // quantile_is_valid, arraymath.py:1747
    }
    for (int64_t i = 0; i < (int64_t)n_doy * n_y; i++)
        if (h_time_index[i] < -T_b || h_time_index[i] >= T_b) return HDP_B200_ERR_INVALID;
    for (int64_t i = 0; i < (int64_t)n_doy * W; i++)
        if (h_win_rows[i] < 0 || h_win_rows[i] >= n_doy) return HDP_B200_ERR_INVALID;
    if (C == 0) return HDP_B200_OK;

    cudaStream_t st = (cudaStream_t)stream;
    const bool need_norm = ld_c != 1;
    ThrLayout L = carve_thr(d_workspace, workspace_bytes, std::max(C, carve_cells), T_b, need_norm || input_unit != 0, n_doy, n_y, W);
    if (!d_workspace || L.total > workspace_bytes) return HDP_B200_ERR_WORKSPACE;
    const float *x = d_temps;
    if (need_norm) {
        int rc = normalize_layout(d_temps, C, T_b, ld_t, ld_c, L.xn, st);
        if (rc != HDP_B200_OK) return rc;
        x = L.xn;
        ld_t = C;
    }
    // Kelvin / Fahrenheit input: k_thr_net converts every sample as it loads it (nothing extra moves); the other kernels work
    // on a converted copy.  `convert_copy` is called on the paths that need it.
    auto convert_copy = [&]() -> int {
        if (input_unit == 0) return HDP_B200_OK;
        if (x != L.xn && ld_t != C) {                                        // rows with a pitch: densify first
            int rc = normalize_layout(x, C, T_b, ld_t, 1, L.xn, st);
            if (rc != HDP_B200_OK) return rc;
            x = L.xn;
            ld_t = C;
        }
        int rc = to_celsius_launch(x, C * T_b, input_unit, L.xn, st);
        x = L.xn;
        input_unit = 0;
        return rc;
    };
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.time_index, h_time_index, sizeof(int) * (size_t)n_doy * n_y, cudaMemcpyHostToDevice, st));

    std::shared_ptr<ThrPlans> plans = thr_plans(h_time_index, h_win_rows, T_b, n_doy, n_y, W, h_q, P, C);
    const RankedPlan &plan = plans->ranked;
    const SegPlan &seg = plans->seg;
    const int E = n_doy * n_y;
    if (seg.usable && !g_force_generic && !g_force_ranked) {
        SelTable sel;
        fill_sel(sel, b, h_q, P);
        if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.seg_time, seg.seg_time.data(), sizeof(int) * seg.seg_time.size(), cudaMemcpyHostToDevice, st));
        if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.seg_ne, seg.seg_ne.data(), sizeof(int) * seg.seg_ne.size(), cudaMemcpyHostToDevice, st));
        if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.doy_rng, seg.doy_rng.data(), seg.doy_rng.size(), cudaMemcpyHostToDevice, st));
        const size_t smem = (size_t)kSegWarps * kSegWarpBytes;
        // per launch, not latched per process: the attribute belongs to the current device's copy of the function
        HDP_CUDA_TRY(cudaFuncSetAttribute(k_thr_seg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SegGeom geo = seg.geo;
        {
            // candidate filter (k_thr_seg phase 1b): every requested position is among the K largest of its window
            int kmin = (int)b - 1;
            for (int p = 0; p < P; p++) kmin = std::min(kmin, sel.pos_lo[p]);
            const int K_top = (int)b - kmin, m = (K_top + W - 1) / W;
            geo.cand_m = (g_seg_candidates && m <= kSegCandTop && 3 * m <= n_y) ? m : 0;      // worth it for the top third only
        }
        geo.n_groups = (int)((C + kSegWarps - 1) / kSegWarps);
        geo.gc = std::min(thr_chunk_groups(T_b), geo.n_groups);
        const int64_t n_chunks = (geo.n_groups + geo.gc - 1) / geo.gc;
        const int64_t blocks = n_chunks * geo.n_seg * geo.gc;
        if (blocks > 0x7fffffffLL) return HDP_B200_ERR_UNSUPPORTED;
        if (input_unit == 2) { const int rc = convert_copy(); if (rc != HDP_B200_OK) return rc; }   // (the division stays out of k_thr_net)
        if (plans->net.usable && g_net && g_seg_light && g_seg_candidates && (size_t)blocks <= L.handed_over_count) {
            // high quantiles, regular windows: the lane-per-cell network kernel; cells with NaN / +-inf samples put all their
            // segments on k_thr_seg's hand-over list, which runs behind it (8 us when the list is empty)
            NetPlan net = plans->net;                                           // (tables are shared; the cell split is per call)
            net_set_cells(net, C);
            net.geo.unit = input_unit;
            if (!tables_resident) {
                HDP_CUDA_TRY(cudaMemcpyAsync(L.net.seq_time, net.seq_time.data(), sizeof(int) * net.seq_time.size(), cudaMemcpyHostToDevice, st));
                HDP_CUDA_TRY(cudaMemcpyAsync(L.net.win_day, net.win_day.data(), sizeof(int) * net.win_day.size(), cudaMemcpyHostToDevice, st));
                if (net.geo.n_irr) {
                    HDP_CUDA_TRY(cudaMemcpyAsync(L.net.irr_day, net.irr_day.data(), sizeof(int) * net.irr_day.size(), cudaMemcpyHostToDevice, st));
                    HDP_CUDA_TRY(cudaMemcpyAsync(L.net.irr_time, net.irr_time.data(), sizeof(int) * net.irr_time.size(), cudaMemcpyHostToDevice, st));
                }
            }
            HDP_CUDA_TRY(cudaMemsetAsync(L.handed_over, 0, sizeof(uint32_t) * (size_t)(1 + blocks), st));
            const NetHandOver hand{L.handed_over, (int)blocks, geo.n_seg, geo.gc, geo.n_groups, kSegWarps};
            {
                KernelTimer timer(kThrNet, st);
                const int rc = net_launch(net, L.net, x, C, ld_t, d_out, hand, st, g_net_tmem != 0);
                if (rc != HDP_B200_OK) return rc;
            }
            KernelTimer timer(kThrSeg, st);
            const unsigned turns = (unsigned)std::min<int64_t>(blocks, 2 * 148 * 4);
            geo.unit = input_unit;                                              // the handed-over cells are converted as they are gathered
            k_thr_seg<<<turns, kSegWarps * 32, smem, st>>>(x, C, ld_t, L.seg_time, L.seg_ne, (const uint4 *)L.doy_rng, geo, sel, P,
                                                           (int)b, n_doy, d_out, L.handed_over, (int)blocks);
            HDP_LAUNCH_CHECK();
            return HDP_B200_OK;
        }
        { const int rc = convert_copy(); if (rc != HDP_B200_OK) return rc; }
        if (geo.cand_m > 0 && g_seg_light && (size_t)blocks <= L.handed_over_count) {
            // high quantiles: the light kernel first, then k_thr_seg for the warps it handed over (non-finite samples,
            // more than kLCap candidates), a small grid taking the blocks on the hand-over list in turns
            const size_t smem_l = (size_t)kSegWarps * kLWarpBytes;
            HDP_CUDA_TRY(cudaFuncSetAttribute(k_thr_cand, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l));
            HDP_CUDA_TRY(cudaMemsetAsync(L.handed_over, 0, sizeof(uint32_t) * (size_t)(1 + blocks), st));
            {
                KernelTimer timer(kThrCand, st);
                k_thr_cand<<<(unsigned)blocks, kSegWarps * 32, smem_l, st>>>(x, C, ld_t, L.seg_time, L.seg_ne, (const uint4 *)L.doy_rng, geo, sel,
                                                                          P, (int)b, n_doy, d_out, L.handed_over);
                HDP_LAUNCH_CHECK();
            }
            KernelTimer timer(kThrSeg, st);
            const unsigned turns = (unsigned)std::min<int64_t>(blocks, 2 * 148 * 4);
            k_thr_seg<<<turns, kSegWarps * 32, smem, st>>>(x, C, ld_t, L.seg_time, L.seg_ne, (const uint4 *)L.doy_rng, geo, sel, P,
                                                           (int)b, n_doy, d_out, L.handed_over, (int)blocks);
            HDP_LAUNCH_CHECK();
            return HDP_B200_OK;
        }
        KernelTimer timer(kThrSeg, st);
        k_thr_seg<<<(unsigned)blocks, kSegWarps * 32, smem, st>>>(x, C, ld_t, L.seg_time, L.seg_ne, (const uint4 *)L.doy_rng, geo, sel, P,
                                                                  (int)b, n_doy, d_out, nullptr, (int)blocks);
        HDP_LAUNCH_CHECK();
        return HDP_B200_OK;
    }
    { const int rc = convert_copy(); if (rc != HDP_B200_OK) return rc; }
    if (plan.usable && !g_force_generic) {
        if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.op_off, plan.op_off.data(), sizeof(int) * plan.op_off.size(), cudaMemcpyHostToDevice, st));
        if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.ops, plan.ops.data(), sizeof(int) * plan.ops.size(), cudaMemcpyHostToDevice, st));
        if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.doy_dup, plan.doy_dup.data(), plan.doy_dup.size(), cudaMemcpyHostToDevice, st));
        HDP_CUDA_TRY(cudaFuncSetAttribute(k_thr_ranked, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
        KernelTimer timer(kThrRanked, st);
        k_thr_ranked<<<(unsigned)C, kRankedThreads, plan.smem, st>>>(x, T_b, ld_t, L.time_index, E, n_y, n_doy, (int)b,
                                                                    L.op_off, L.ops, L.doy_dup, plan.dpw, plan.ept, plan.nwords_pad,
                                                                    plan.sel, P, d_out, nullptr, nullptr);
        HDP_LAUNCH_CHECK();
        return HDP_B200_OK;
    }

    // generic path: any table, any multiplicity
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.win_rows, h_win_rows, sizeof(int) * (size_t)n_doy * W, cudaMemcpyHostToDevice, st));
    int b_pad_log2 = 1;
    while ((1 << b_pad_log2) < b) b_pad_log2++;
    const int b_pad = 1 << b_pad_log2;
    int NC = 16384 / b_pad;                                                  // <= 64 KB of keys per CTA
    if (NC < 1) NC = 1;
    if (NC > 8) NC = 8;
    const size_t smem = (size_t)NC * b_pad * sizeof(float) + (size_t)NC * 3 * sizeof(int);
    HDP_CUDA_TRY(cudaFuncSetAttribute(k_thr_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)((C + NC - 1) / NC), (unsigned)n_doy);
    KernelTimer timer(kThrGeneric, st);
    k_thr_generic<<<grid, 256, smem, st>>>(x, C, T_b, ld_t, L.time_index, L.win_rows, n_doy, n_y, W, qt, P, NC, b_pad_log2, d_out);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace hdp

using namespace hdp;

extern "C" {

void hdp_b200_thresholds_force_generic(int on)
{
    g_force_generic = on == 1; g_force_ranked = on == 2; g_seg_candidates = on != 3; g_seg_light = on != 4; g_net = on != 5;
    g_net_tmem = on != 6;
}

int hdp_b200_thresholds_kernel_choice(const int32_t *h_time_index, const int32_t *h_win_rows, int64_t T_b, int n_doy, int n_y, int W,
                                      const double *h_q, int P, int *info)
{
    if (bad_dims(1, T_b, n_doy, n_y, W, P) || !h_time_index || !h_win_rows || !h_q || !info) return HDP_B200_ERR_INVALID;
    if (P > HDP_B200_MAX_PERCENTILES || (int64_t)W * n_y > HDP_B200_MAX_WINDOW) return HDP_B200_ERR_UNSUPPORTED;
    const auto plans = thr_plans(h_time_index, h_win_rows, T_b, n_doy, n_y, W, h_q, P, 64800);
    const NetGeom &g = plans->net.geo;
    for (int i = 0; i < 8; i++) info[i] = 0;
    if (plans->seg.usable && plans->net.usable) {
        info[0] = 4; info[1] = g.NY; info[2] = g.K; info[3] = g.M; info[4] = g.s; info[5] = g.n_irr; info[6] = g.tm_warps; info[7] = g.tm_lists;
    } else if (plans->seg.usable) {
        int kmin = W * n_y - 1;
        for (int p = 0; p < P; p++) kmin = std::min(kmin, plans->sel.pos_lo[p]);
        const int m = (W * n_y - kmin + W - 1) / W;
        info[0] = (m <= kSegCandTop && 3 * m <= n_y) ? 3 : 2;
        info[4] = plans->seg.geo.S;
    } else if (plans->ranked.usable) info[0] = 1;
    return HDP_B200_OK;
}

size_t hdp_b200_thresholds_workspace_bytes(int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                                           int n_doy, int n_y, int W, int P, int input_unit)
{
    (void)ld_t;
    if (bad_dims(C, T_b, n_doy, n_y, W, P)) return 0;
    return carve_thr(nullptr, 0, C, T_b, ld_c != 1 || input_unit != 0, n_doy, n_y, W).total;
}

int hdp_b200_thresholds(const float *d_temps, int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                        const int32_t *h_time_index, const int32_t *h_win_rows, int n_doy, int n_y, int W,
                        const double *h_q, int P, double *d_out,
                        void *d_workspace, size_t workspace_bytes, void *stream, int input_unit)
{
    return thresholds_launch(d_temps, C, T_b, ld_t, ld_c, h_time_index, h_win_rows, n_doy, n_y, W, h_q, P, d_out,
                             d_workspace, workspace_bytes, stream, C, false, input_unit);
}

}  // extern "C"
