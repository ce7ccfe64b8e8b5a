// metric.cu - path 2: hot-day masks and heatwave metrics for the whole percentile x definition sweep.
//
// Replaces (reference = AgentOxygen/HDP v1.0.2):
//   indicate_hot_days          hdp/metric.py:280-301
//   index_heatwaves            hdp/metric.py:11-60
//   heatwave_frequency/number/duration/average   hdp/metric.py:63-172
//   compute_heatwave_metrics   hdp/metric.py:304-341
//   compute_heatwave_metrics_wrapper (the percentile x definition x cell sweep)   hdp/metric.py:344-369
//
// Two kernels, both HBM-streaming integer/compare work (no tensor cores: nothing here is a contraction):
//
//   k_hot_words  (cells x day-of-year block) tiles.  A CTA owns 32 cells and 32 consecutive days of year,
//                keeps that [32 doy][P][32 cell] threshold tile in shared memory (rounded DOWN to f32, which
//                preserves the reference's double-precision `measure > threshold` exactly) and walks every
//                year of the measure through it, so each threshold is fetched from HBM once and each
//                measure sample once.  Output: one 32-bit word of hot-day bits per (percentile, word, cell).  A cold-spell
//                pass (HDP_B200_COLD) instantiates it with COLD: the tile is rounded UP and the bits mark `measure <
//                threshold`; everything downstream works on the bits and does not know which direction made them.
//   k_scan       one thread per (cell, percentile), lanes = cells (coalesced).  Walks the hot words in
//                time order, pops hot runs with bit tricks and feeds each run to all definitions' state
//                machines held in registers; season accumulators are flushed as u16 when a season closes.
//                The per-day heatwave id array of the reference is never materialised.
#include <limits.h>
#include <vector>
#include <algorithm>

#include "intensity.h"
#include "metric.cuh"

namespace hdp {


// ----------------------------------------------------------------------------------------------------
// k_hot_words
// ----------------------------------------------------------------------------------------------------
constexpr int kHotDays = 16;  // days of each of kHotYears words whose samples are in flight together

template <int PG, int J0, int UNIT, bool COLD>
__device__ __forceinline__ void hot_half(uint32_t (&m)[kHotYears][PG], const float *const (&xp)[kHotYears], const int (&jo)[kHotYears],
                                         const int (&nb)[kHotYears], int64_t ld_t, const float *ts)
{
    float v[kHotYears][kHotDays];
#pragma unroll
    for (int y = 0; y < kHotYears; y++)
#pragma unroll
        for (int j = 0; j < kHotDays; j++)                 // NaN = never hot: days outside the word
            v[y][j] = (unsigned)(J0 + j - jo[y]) < (unsigned)nb[y] ? __ldg(xp[y] + (int64_t)(J0 + j) * ld_t) : __int_as_float(0x7fc00000);
    if (UNIT != 0) {                                       // Kelvin / Fahrenheit input, converted as it is loaded (NaN stays NaN)
#pragma unroll
        for (int y = 0; y < kHotYears; y++)
#pragma unroll
            for (int j = 0; j < kHotDays; j++) v[y][j] = to_celsius_f(v[y][j], UNIT);
    }
#pragma unroll
    for (int j = 0; j < kHotDays; j++) {
        float t[PG];
#pragma unroll
        for (int q = 0; q < PG; q++) t[q] = ts[((J0 + j) * PG + q) * kTilePad];
#pragma unroll
        for (int y = 0; y < kHotYears; y++)
#pragma unroll
            for (int q = 0; q < PG; q++) {
                if (COLD) or_if_lt(m[y][q], v[y][j], t[q], 1u << (J0 + j));
                else or_if_gt(m[y][q], v[y][j], t[q], 1u << (J0 + j));
            }
    }
}

// COLD: the bits mark days with (double)x < thr (cold spells) instead of (double)x > thr.  The tile is then rounded UP
// (__double2float_ru), which keeps the double-precision `x < thr` exact for every float x: a thr that is a float is kept; else
// ru(thr) is the smallest float above thr, so no float lies in [thr, ru(thr)) and x < thr <=> x < ru(thr).  At the ends: thr >
// FLT_MAX becomes +inf, below which every finite float lies (all are < thr); thr < -FLT_MAX becomes -FLT_MAX, below which only
// -inf lies (the only float < thr).  NaN stays NaN and compares false on either side; the padding is -inf, never cold.
template <int PG, int UNIT, bool COLD>
__global__ void __launch_bounds__(256, PG <= 10 ? 3 : 2)
k_hot_words(const float *__restrict__ x, int64_t C, int64_t ld_t,
            const double *__restrict__ thr, int n_doy, int P,
            const int4 *__restrict__ words, const int *__restrict__ blk_start, const int *__restrict__ blk_words,
            int K, uint32_t *__restrict__ hot)
{
    extern __shared__ float thr_s[];                      // [percentile group][32 doy][PG][33]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int db = blockIdx.y;
    const int64_t c0 = (int64_t)blockIdx.x * kTileCells;
    const int Ppad = (P + PG - 1) / PG * PG;
    const int nd = min(kTileDoy, n_doy - db * kTileDoy);

    // Threshold tile.  Per cell the (doy, percentile) block of this tile is nd * P contiguous doubles in the reference's
    // [C, n_doy, P] order: a warp reads them with consecutive lanes, kFillLoads independent loads per lane in flight
    // (the fill is pure HBM latency), and scatters them to [group][doy][PG][cell].  Padding percentiles / days: +inf (-inf
    // for COLD), which no sample exceeds (falls below).
    const int n_el = nd * P;                               // doubles per cell
    if (nd < kTileDoy || Ppad != P)
        for (int i = tid; i < (Ppad / PG) * kTileDoy * PG * kTilePad; i += 256) thr_s[i] = __int_as_float(COLD ? 0xff800000 : 0x7f800000);
    __syncthreads();
    const float inv_p = 1.0f / (float)P;                   // e / P for e < 1024, P <= 32: (e + 0.5) / P is >= 1 / 64 away from every
    for (int e0 = 0; e0 < n_el; e0 += 32 * kFillLoads) {   // integer, far more than the error of the float product
        int dst[kFillLoads];
#pragma unroll
        for (int i = 0; i < kFillLoads; i++) {
            const int e = e0 + 32 * i + lane;
            const int j = __float2int_rz(((float)e + 0.5f) * inv_p), p = e - j * P, g = p / PG, q = p - g * PG;
            dst[i] = e < n_el ? ((g * kTileDoy + j) * PG + q) * kTilePad : -1;
        }
        for (int cell = warp; cell < kTileCells; cell += 8) {
            if (c0 + cell >= C) break;
            const double *src = thr + ((c0 + cell) * n_doy + (int64_t)db * kTileDoy) * P + e0 + lane;
            double v[kFillLoads];
#pragma unroll
            for (int i = 0; i < kFillLoads; i++) v[i] = dst[i] >= 0 ? __ldg(src + 32 * i) : 0.0;
#pragma unroll
            for (int i = 0; i < kFillLoads; i++)
                if (dst[i] >= 0) thr_s[dst[i] + cell] = COLD ? __double2float_ru(v[i]) : __double2float_rd(v[i]);
        }
    }
    __syncthreads();

    const int64_t c = c0 + lane;
    if (c >= C) return;
    // A warp takes kHotYears words (= years of this day-of-year block) at a time.  It first puts kHotDays days of each
    // of them in flight (kHotYears * kHotDays independent 128-byte loads per warp), then compares them against the days'
    // thresholds, which are read from shared memory into registers once per kHotYears samples.  Bits are collected at
    // the day's position inside the 32-day block (an immediate) and shifted to the word's own origin when stored.
    const int w_begin = blk_start[db], w_end = blk_start[db + 1];
    const int64_t plane_words = (int64_t)K * C;
    for (int i0 = w_begin + warp * kHotYears; i0 < w_end; i0 += 8 * kHotYears) {
        int kk[kHotYears], jo[kHotYears], nb[kHotYears];
        const float *xp[kHotYears];
        int j_hi = 0;
#pragma unroll
        for (int y = 0; y < kHotYears; y++) {
            const bool live = i0 + y < w_end;
            kk[y] = blk_words[live ? i0 + y : i0];
            const int4 w = words[kk[y]];                   // {t0, nbits, doy of bit 0, -}
            jo[y] = w.z & (kTileDoy - 1);
            nb[y] = live ? w.y : 0;
            xp[y] = x + ((int64_t)w.x - jo[y]) * ld_t + c; // day jd of the block is sample xp[y][jd * ld_t]
            if (live) j_hi = max(j_hi, jo[y] + nb[y]);
        }
        for (int pg = 0; pg < Ppad; pg += PG) {
            uint32_t m[kHotYears][PG];
#pragma unroll
            for (int y = 0; y < kHotYears; y++)
#pragma unroll
                for (int q = 0; q < PG; q++) m[y][q] = 0u;
            const float *ts = thr_s + (size_t)(pg / PG) * (kTileDoy * PG * kTilePad) + lane;
            uint32_t *hp[kHotYears];                               // word kk[y] of percentile pg of this cell; percentile planes are K * C words apart
#pragma unroll
            for (int y = 0; y < kHotYears; y++) hp[y] = hot + ((int64_t)pg * K + kk[y]) * C + c;
            hot_half<PG, 0, UNIT, COLD>(m, xp, jo, nb, ld_t, ts);
            if (j_hi > kHotDays) hot_half<PG, kHotDays, UNIT, COLD>(m, xp, jo, nb, ld_t, ts);      // warp-uniform
#pragma unroll
            for (int y = 0; y < kHotYears; y++)
#pragma unroll
                for (int q = 0; q < PG; q++)
                    if (nb[y] > 0 && pg + q < P) hp[y][(int64_t)q * plane_words] = m[y][q] >> jo[y];
        }
    }
}

// ----------------------------------------------------------------------------------------------------
// k_unpack_mask: hot words -> u8 [P, T, C]   (parity checks of the hot-day mask only)
// ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_unpack_mask(const uint32_t *__restrict__ hot, int64_t C, int64_t T, int P, int K, const int4 *__restrict__ words,
              uint8_t *__restrict__ mask)
{
    const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int k = blockIdx.y;
    if (c >= C) return;
    const int4 w = words[k];
    for (int p = 0; p < P; p++) {
        const uint32_t m = hot[((int64_t)p * K + k) * C + c];
        for (int j = 0; j < w.y; j++) mask[((int64_t)p * T + (w.x + j)) * C + c] = (m >> j) & 1u;
    }
}

// ----------------------------------------------------------------------------------------------------
// k_scan
// ----------------------------------------------------------------------------------------------------
static std::atomic<int> g_scan_filter{1};        // test hook (hdp_b200_metrics_run_filter): 0 = k_scan queues every run

struct ScanTables {
    uint32_t max_subs_plane[32];     // bit k of max_subs of every definition (bit-sliced constants)
    int ge_len, brk_len;             // table lengths: max(min_dur) + 2, max(max_break) + 2
    int f_on, f_lmin, f_bmax;        // run filter: on/off, min over definitions of min_dur, max over definitions of max_break
};

// k_scan's ONSET state: per accumulator register the packed onset and end lanes (day of the season of the first / last in-season
// heatwave day, the packing of HWF), and `seen`, bit i = definition i has had an in-season block.  Empty without ONSET.
template <bool ONSET, int NG>
struct ScanOnset {
    uint32_t ons[NG], end[NG], seen;
    __device__ __forceinline__ void reset()
    {
#pragma unroll
        for (int j = 0; j < NG; j++) { ons[j] = 0u; end[j] = 0u; }
        seen = 0u;
    }
};
template <int NG>
struct ScanOnset<false, NG> {
    __device__ __forceinline__ void reset() {}
};

constexpr int kScanWarps = 8;
constexpr int kScanQ = 16;                                       // queued words per lane (power of two)
constexpr int kScanQueueWords = 3 * kScanQ * 32;                  // u32 per warp: run starts, run ends, first day of the word

// p + bytes as one 64-bit add the compiler keeps: written as `p += n`, the flush's pointers were turned back into element indices
// and every store rebuilt its address from them
__device__ __forceinline__ uint16_t *add_ptr(uint16_t *p, int64_t bytes)
{
    uint16_t *r;
    asm("add.s64 %0, %1, %2;" : "=l"(r) : "l"(p), "l"(bytes));
    return r;
}

__device__ __forceinline__ void stg_u16(uint16_t *p, uint32_t v)
{
    asm volatile("st.global.u16 [%0], %1;" ::"l"(p), "h"((unsigned short)v) : "memory");
}

// k_scan.  One warp per (32 neighbouring cells, percentile), one lane per cell.  Two alternating phases:
//
//  A (warp-synchronous over the hot words, in time order): the lanes read word k of their cells (one coalesced
//    load, prefetched four words ahead), DROP THE RUNS THAT CANNOT MATTER and queue what is left of the word, as run
//    start / run end bit masks, in a per-lane ring buffer in shared memory.  Let lmin = min over definitions of
//    min_duration and bmax = max over definitions of max_break, call a run long if it has >= lmin days, and a cluster a
//    maximal sequence of runs whose breaks are all <= bmax.  Before the first long run of its cluster a run finds
//    in_heatwave clear for every definition (the break before the cluster cleared it, reference index_heatwaves,
//    hdp/metric.py:43-58) and, being short, leaves it clear: branch A needs the length, C and D need in_heatwave.  It
//    changes no state and gets no label - and the longer break the next kept run then sees clears in_heatwave just the
//    same - so only the runs from the first long run of a cluster on are kept: keep_i = long_i | (near_i & keep_(i-1)).
//    This is evaluated with bit operations on the word and its neighbours (b = days of long runs; G = days at most bmax
//    after a hot day, so a cluster is one contiguous run of G; an add floods each cluster upwards from its long days).
//    Where a neighbouring word is not known yet the run is kept.  Words without a surviving run start or end are
//    not queued at all.
//  B (lane-asynchronous): every lane pops the runs of its own queue and advances ALL definitions' state machines
//    BIT-PARALLEL: bit i of each state word belongs to definition i, so one run costs the same for 1 or 32 definitions.
//      inhw        bit i = in_heatwave of definition i
//      rem[k]      bit-sliced down counter: remaining subsequent events = max_subs - sub_events
//      fresh       bit i = the next labelled run of definition i starts a heatwave id not yet seen in the open season
//    Season accumulators are packed SIMD-in-register: four definitions per register (8-bit lanes) when no season is
//    longer than 255 days, else two (16-bit lanes): cnt (days of the current id in the open season), HWF, HWN, HWD.
//    A lane stops at the first run that starts after its open season; when every lane has stopped the season is closed
//    with the whole warp converged on the stores.
//
// Season tables: int4 {start, end, output row, -} per hemisphere, sorted and disjoint within a table
// (the host splits overlapping tables into several passes, one launch each).
// (Three CTAs per SM for every accumulator-group count: with 24 definitions the 80-register build spills 100 - 400 bytes per
// thread, but two CTAs with 128 registers and no spills measured SLOWER - 34.0 against 32.1 ms on wide_sweep: the kernel needs
// the warps more than the registers.)
// ONSET: also HWO and HWE, the first and last heatwave day of every season (planes 4 and 5 of u16 [6, P, D, Y, C]), from two more
// packed accumulators per register: the onset of the first in-season block of a labelled run and the end of the last one.  The run
// filter drops only runs that get no label, so it cannot drop a block.
// LMIN / BMAX > = 0: the run filter's two constants (smallest min_duration, largest max_break of the definition set) at compile
// time, which unrolls its shift loops completely - 12 % of the kernel on the reference's documented definitions (README.md:51:
// min duration 3 .. 5, at most one break day: LMIN = 3, BMAX = 1).  LMIN = 0: run-time values (any definition set).
template <int NG, int KS, bool kBytes, int LMIN = 0, int BMAX = 0, bool ONSET = false>
__global__ void __launch_bounds__(kScanWarps * 32, 3)
k_scan(const uint32_t *__restrict__ hot, int64_t C, int K, int T, const int4 *__restrict__ words,
       int P, int D, const __grid_constant__ ScanTables tabs, const uint32_t *__restrict__ ge_tab, const uint32_t *__restrict__ brk_tab,
       const int4 *__restrict__ seasons_north, int n_north, const int4 *__restrict__ seasons_south, int n_south, int Y,
       const uint8_t *__restrict__ is_south, uint16_t *__restrict__ out)
{
    constexpr int PER = kBytes ? 4 : 2, BITS = kBytes ? 8 : 16;
    constexpr uint32_t LANE_MASK = kBytes ? 0xffu : 0xffffu;
    extern __shared__ uint32_t smem_scan[];
    uint32_t *queues = smem_scan;                                 // [warps][3][kScanQ][32]
    uint32_t *ge_s = queues + kScanWarps * kScanQueueWords;       // [ge_len]  definitions with min_dur <= len
    uint32_t *brk_s = ge_s + tabs.ge_len;                         // [brk_len] definitions with max_break < gap
    // [K + 1] per hot word {first day, days, unknown days of the NEXT word (they count as hot), unknown days after that};
    // word K is a virtual cold day at T that closes a run still open at the end of the series
    int4 *word_meta = (int4 *)(smem_scan + ((kScanWarps * kScanQueueWords + tabs.ge_len + tabs.brk_len + 3) & ~3));
    uint32_t *hwa_rcp = (uint32_t *)(word_meta + K + 1);         // [256] 8-bit lanes only: the HWA divisors' reciprocals
    const int tid = threadIdx.x, nthreads = kScanWarps * 32;
    if (kBytes)
        for (int i = tid; i < 256; i += nthreads) hwa_rcp[i] = scan_hwa_rcp(i);
    for (int i = tid; i < tabs.ge_len; i += nthreads) ge_s[i] = ge_tab[i];
    for (int i = tid; i < tabs.brk_len; i += nthreads) brk_s[i] = brk_tab[i];
    for (int i = tid; i <= K; i += nthreads) {
        int4 m = make_int4(T, 1, 0, 0);
        if (i < K) {
            const int4 w = words[i];
            m.x = w.x; m.y = w.y;
            if (i + 1 < K) {                                      // days past the end of the series are known: cold
                const int nb1 = words[i + 1].y;
                m.z = nb1 == 32 ? 0 : (int)(0xffffffffu << nb1);
                m.w = w.y == 32 ? 0 : (int)(0xffffffffu << w.y);
            }
        }
        word_meta[i] = m;
    }
    __syncthreads();

    // warp -> (percentile, group of 32 cells), percentile-major: the warps of a CTA work on the same percentile, so they
    // have similar numbers of runs and the CTA's shared memory is not held by one slow warp; the first percentile (with
    // sorted percentiles the one with the most hot days) is scheduled first, the lightest last, which shortens the tail
    const int lane = tid & 31;
    const int64_t n_cg = (C + 31) / 32;
    const int64_t wg = (int64_t)blockIdx.x * kScanWarps + (tid >> 5);
    const int p = (int)(wg / n_cg);
    const int64_t cg = wg - (int64_t)p * n_cg;
    if (p >= P) return;                                           // warp-uniform
    const bool alive = cg * 32 + lane < C;                        // lanes past the last cell shadow it (the warp votes with all 32 lanes)
    const int64_t c = alive ? cg * 32 + lane : C - 1;
    // 32-bit shared-state-space addresses: queue slot i of this lane is q_st + 128 i (run starts), + kQEn (run ends), + kQT0 (first day)
    const uint32_t q_st = smem_u32(queues + (tid >> 5) * kScanQueueWords + lane);
    constexpr uint32_t kQEn = kScanQ * 128, kQT0 = 2 * kScanQ * 128;
    const uint32_t ge_a = smem_u32(ge_s), brk_a = smem_u32(brk_s), meta_a = smem_u32(word_meta);

    const bool south = is_south != nullptr && is_south[c] != 0;
    const int4 *seas = south ? seasons_south : seasons_north;
    const int n_seasons = south ? n_south : n_north;
    int ys = 0;
    int a_cur = INT_MAX, b_cur = INT_MAX, row_cur = 0;
    if (n_seasons > 0) { const int4 s4 = seas[0]; a_cur = s4.x; b_cur = s4.y; row_cur = s4.z; }

    uint32_t inhw = 0u, sublt = 0u, fresh = 0xffffffffu;
    uint32_t rem[KS];
#pragma unroll
    for (int k = 0; k < KS; k++) { rem[k] = tabs.max_subs_plane[k]; sublt |= rem[k]; }     // sub_events = 0
    uint32_t cntg[NG], hwfg[NG], hwng[NG], hwdg[NG];              // definitions PER * j .. PER * j + PER - 1
#pragma unroll
    for (int j = 0; j < NG; j++) { cntg[j] = 0u; hwfg[j] = 0u; hwng[j] = 0u; hwdg[j] = 0u; }
    ScanOnset<ONSET, NG> on;
    on.reset();

    // metric m of definition d, season row r of this lane's cell: out_pc[m * P * D * Y * C + d * Y * C + r * C]
    uint16_t *const out_pc = out + (int64_t)p * D * Y * C + c;
    auto lane_of = [](uint32_t v, int h) -> uint32_t {            // accumulator lane h of a register, zero-extended (one PRMT)
        return kBytes ? __byte_perm(v, 0u, 0x4440 + h) : (v >> (BITS * h)) & LANE_MASK;
    };
    auto flush = [&]() {                                          // close season `ys`
        if (alive) {
            const int64_t dstride_b = (int64_t)Y * C * sizeof(uint16_t), plane_b = P * D * dstride_b;
            uint16_t *o = out_pc + (int64_t)row_cur * C;
#pragma unroll
            for (int j = 0; j < NG; j++) {
#pragma unroll
                for (int h = 0; h < PER; h++) {
                    if (PER * j + h < D) {                        // warp-uniform
                        const uint32_t f = lane_of(hwfg[j], h), nn = lane_of(hwng[j], h);
                        uint16_t *const o1 = add_ptr(o, plane_b), *const o2 = add_ptr(o1, plane_b), *const o3 = add_ptr(o2, plane_b);
                        stg_u16(o, f);
                        stg_u16(o1, nn);
                        stg_u16(o2, lane_of(hwdg[j], h));
                        // trunc(mean) = f / nn in integers, metric.py:340; 8-bit lanes: f * ceil(2^16 / nn) >> 16, exact for
                        // f, nn < 256 (scan_hwa_rcp)
                        stg_u16(o3, kBytes ? (f * hwa_rcp[nn]) >> 16 : nn ? f / nn : 0u);
                        if constexpr (ONSET) {
                            uint16_t *const o4 = add_ptr(o3, plane_b), *const o5 = add_ptr(o4, plane_b);
                            stg_u16(o4, scan_onset_value(f, lane_of(on.ons[j], h)));
                            stg_u16(o5, scan_onset_value(f, lane_of(on.end[j], h)));
                        }
                    }
                    o = add_ptr(o, dstride_b);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < NG; j++) { cntg[j] = 0u; hwfg[j] = 0u; hwng[j] = 0u; hwdg[j] = 0u; }
        on.reset();
        fresh = 0xffffffffu;
        ys++;
        if (ys < n_seasons) { const int4 s4 = seas[ys]; a_cur = s4.x; b_cur = s4.y; row_cur = s4.z; }
        else { a_cur = INT_MAX; b_cur = INT_MAX; }
    };

    // definition bits -> one 0/1 per accumulator lane.  The bits are those of definitions < D <= PER * NG (labels are made from
    // the definition tables), so the last group needs no mask.
    auto spread = [](uint32_t bits, int j) -> uint32_t {
        const uint32_t t = bits >> (PER * j), g = j == NG - 1 ? t : t & ((1u << PER) - 1u);
        return kBytes ? (g * 0x00204081u) & 0x01010101u : (g * 0x00008001u) & 0x00010001u;
    };
    // accounting of `days` heatwave days of the definitions in `lab` to the open season (HWF/HWN/HWD, metric.py:63-137): the
    // in-season block [max(s, a_cur), max(s, a_cur) + days) of a labelled run that starts on day s
    auto account = [&](uint32_t lab, uint32_t days, int s) {
        const uint32_t newly = lab & fresh;                       // first labelled run of an id inside this season
        fresh &= ~lab;
#pragma unroll
        for (int j = 0; j < NG; j++) {
            const uint32_t sel = spread(lab, j), neu = spread(newly, j), add = days * sel;
            cntg[j] = (cntg[j] & ~(neu * LANE_MASK)) + add;
            hwfg[j] += add;
            hwng[j] += neu;
            hwdg[j] = kBytes ? __vmaxu4(hwdg[j], cntg[j]) : __vmaxu2(hwdg[j], cntg[j]);
        }
        if constexpr (ONSET) {
            const uint32_t first = lab & ~on.seen, off = (uint32_t)(max(s, a_cur) - a_cur);     // the block's first day of the season
#pragma unroll
            for (int j = 0; j < NG; j++) scan_onset_update(on.ons[j], on.end[j], spread(first, j), spread(lab, j), off, off + days - 1u, LANE_MASK);
            on.seen |= lab;
        }
    };

    // ---- phase A state ----
    const uint32_t *hp = hot + (int64_t)p * K * C + c;
    int k_ext = 0;                                                // next word to extract (warp-uniform); word K is the virtual one
    uint32_t w0 = K > 0 ? hp[0] : 0u, w1 = K > 1 ? hp[C] : 0u, w2 = K > 2 ? hp[2 * C] : 0u, w3 = K > 3 ? hp[3 * C] : 0u;
    const uint32_t *hp_ahead = hp + 4 * C;                        // word k_ext + 4
    const int64_t pf_off = (int64_t)kScanQ * C;
    uint32_t tail = 0u, a_tail = 0u;                              // hot days / `long` seeds of the 32 days before word k_ext (bit 31 = yesterday)
    uint32_t live_in = 0u, open_f = 0u;                           // a live cluster / a kept run reaches the end of the previous word
    uint32_t qr = 0u, qw = 0u;                                    // ring buffer read / write counters
    const bool f_on = LMIN > 0 || tabs.f_on != 0;
    const int f_lmin = LMIN > 0 ? LMIN : tabs.f_lmin, f_bmax = LMIN > 0 ? BMAX : tabs.f_bmax;

    // one word: `cur` = word k_ext of this lane's cell, `nxt` = word k_ext + 1
    auto extract_word = [&](const uint32_t cur, const uint32_t nxt, bool live) {
        {
            const uint4 wm = lds_v4(meta_a + 16u * (uint32_t)k_ext);   // warp-uniform
            const int t0 = (int)wm.x, nb = (int)wm.y;
            const uint32_t vmask = 0xffffffffu >> (32 - nb);
            uint32_t keep = cur;
            if (f_on) {
                // E = the 64 days starting at this word (lo, hi): the next word follows at bit nb
                const uint32_t fut = nxt | (uint32_t)wm.z;
                uint32_t lo = cur, hi = fut;
                if (nb < 32) {                                     // warp-uniform
                    lo = cur | (fut << nb);
                    hi = (fut >> (32 - nb)) | (uint32_t)wm.w;
                }
                // a_j: days j .. j + lmin - 1 are all hot;  b_j: day j belongs to lmin consecutive hot days (a long run)
                uint32_t a = lo;
#pragma unroll
                for (int j = 1; j < 4; j++) if (j < f_lmin) a &= __funnelshift_r(lo, hi, j);
                for (int j = 4; j < f_lmin; j++) a &= __funnelshift_r(lo, hi, j);
                a &= vmask;
                uint32_t b = a;
#pragma unroll
                for (int j = 1; j < 4; j++) if (j < f_lmin) b |= __funnelshift_l(a_tail, a, j);
                for (int j = 4; j < f_lmin; j++) b |= __funnelshift_l(a_tail, a, j);
                // G_j: day j is hot or at most bmax days after a hot day - runs whose breaks are all <= bmax form one
                // contiguous cluster of G
                uint32_t G = cur;
#pragma unroll
                for (int j = 1; j < 4; j++) if (j <= f_bmax) G |= __funnelshift_l(tail, cur, j);
                for (int j = 4; j <= f_bmax; j++) G |= __funnelshift_l(tail, cur, j);
                G &= vmask;
                // a cluster matters from its first long run on: flood every cluster upwards from its long days (and from
                // day 0 if the cluster was already live at the end of the previous word); the add carries through G
                const uint32_t seed = b | (live_in & G & 1u);
                const uint32_t flooded = (((G + seed) ^ G) & G) | seed;
                keep = flooded & cur;
                live_in = flooded >> (nb - 1);                     // (bit 0 is what is used)
                tail = nb == 32 ? cur : __funnelshift_r(tail, cur, nb);
                a_tail = nb == 32 ? a : __funnelshift_r(a_tail, a, nb);
            }
            const uint32_t prevk = (keep << 1) | open_f;           // bit i = day i - 1 is a kept hot day
            const uint32_t st = keep & ~prevk, en = ~keep & prevk & vmask;
            open_f = (keep >> (nb - 1)) & 1u;
            if (live && (st | en) != 0u) {
                const uint32_t slot = q_st + (qw & (kScanQ - 1)) * 128u;
                sts_u32(slot, st); sts_u32(slot + kQEn, en); sts_u32(slot + kQT0, (uint32_t)t0);
                qw++;
            }
        }
    };
    // word k_ext + 4 (words past the end read as cold); the L2 prefetch reaches for the next burst's words
    auto next_word = [&]() -> uint32_t {
        const uint32_t v = k_ext + 4 < K ? __ldg(hp_ahead) : 0u;
        if (k_ext + 4 + kScanQ < K) asm volatile("prefetch.global.L2 [%0];" ::"l"(hp_ahead + pf_off));
        hp_ahead += C;
        k_ext++;
        return v;
    };
    // Four words per round with the registers taking turns, so that a word fetched now is not touched before it is needed four
    // words later (rotating w0 <- w1 <- w2 <- w3 reads the register a load is still in flight for: the whole warp then waits for
    // every word - 11 % of this kernel's stall samples in round 1's profile); the rotation is left to the last < 4 words of a burst.
    auto extract = [&](int n_words, bool live) {
        int i = 0;
        for (; i + 4 <= n_words; i += 4) {
            extract_word(w0, w1, live); w0 = next_word();
            extract_word(w1, w2, live); w1 = next_word();
            extract_word(w2, w3, live); w2 = next_word();
            extract_word(w3, w0, live); w3 = next_word();
        }
        for (; i < n_words; i++) {
            extract_word(w0, w1, live);
            const uint32_t v = next_word();
            w0 = w1; w1 = w2; w2 = w3; w3 = v;
        }
    };

    // ---- phase B state ----
    int prev_e = -(1 << 29);      // end of the previous (kept) hot run
    int run_start = -1;           // start of the hot run still open at the end of the previous queued word
    const int ge_cap = tabs.ge_len - 1, brk_cap = tabs.brk_len - 1;
    int t0 = 0;
    uint32_t starts = 0u, ends = 0u;
    uint32_t pend_lab = 0u;       // labelled run that continues past the end of the season being closed
    int pend_s = 0, pend_e = 0;

    // One iteration per season of the lanes' tables: consume every run that starts before the season ends, then close
    // the season with the warp converged on the stores.
    for (;;) {
        const bool open = ys < n_seasons;
        if (!__any_sync(0xffffffffu, open)) break;
        // lane state inside a season: 0 = consuming runs, 1 = done (nothing more to do before the season closes),
        // 2 = starved (its queue is empty and there are words left to extract)
        int state = open ? 0 : 1;
        if (!open) qr = qw;                                       // a lane without seasons left drops what it has queued
        if (open && pend_lab) {
            const int days = min(pend_e, b_cur) - max(pend_s, a_cur);
            if (days > 0) account(pend_lab, (uint32_t)days, pend_s);
            if (pend_e <= b_cur) pend_lab = 0u; else state = 1;
        }
        for (;;) {
            if (state == 2) state = 0;
            while (__any_sync(0xffffffffu, state == 0)) {
                if (state == 0 && ends == 0u) {
                    // ---- the word is used up: take the next one from the queue ----
                    if (starts) { run_start = t0 + __ffs(starts) - 1; starts = 0u; }   // at most one start is left: the run stays open
                    if (qr == qw) {
                        state = k_ext > K ? 1 : 2;                // series exhausted : starved
                    } else {
                        const uint32_t slot = q_st + (qr & (kScanQ - 1)) * 128u;
                        starts = lds_u32(slot); ends = lds_u32(slot + kQEn); t0 = (int)lds_u32(slot + kQT0);
                        qr++;
                    }
                }
                if (state == 0 && ends != 0u) {
                    // ---- the next hot run [s, e): leave it queued if it starts after this season ----
                    const int s = run_start >= 0 ? run_start : t0 + __ffs(starts) - 1;
                    if (s >= b_cur) state = 1;
                    else {
                        const int e = t0 + __ffs(ends) - 1;
                        ends &= ends - 1;
                        if (run_start >= 0) run_start = -1; else starts &= starts - 1;
                        const int len = e - s, gap = s - prev_e;
                        prev_e = e;

                        // reference index_heatwaves branches A-D for all definitions at once (metric.py:43-58)
                        const uint32_t ge = lds_u32(ge_a + 4u * (uint32_t)min(len, ge_cap));    // len >= min_duration
                        inhw &= ~lds_u32(brk_a + 4u * (uint32_t)min(gap, brk_cap));            // B: the break before this run was too long
                        const uint32_t A = ~inhw & ge;                // A: a new heatwave starts
                        const uint32_t Cm = inhw & sublt;             // C: subsequent event of the current heatwave
                        const uint32_t Dm = inhw & ~sublt;            // D: subsequent events used up
                        const uint32_t Dn = Dm & ge;                  //    ... long enough: new heatwave id
                        const uint32_t lab = A | Cm | Dn;
                        fresh |= A | Dn;
                        inhw = (inhw | A) & ~(Dm & ~ge);
                        uint32_t borrow = Cm;
                        sublt = 0u;
#pragma unroll
                        for (int q = 0; q < KS; q++) {                // rem -= 1 where C, rem = max_subs where D
                            const uint32_t t = ~rem[q] & borrow;
                            rem[q] = ((rem[q] ^ borrow) & ~Dm) | (tabs.max_subs_plane[q] & Dm);
                            borrow = t;
                            sublt |= rem[q];
                        }
                        const int days = min(e, b_cur) - max(s, a_cur);
                        if (lab != 0u && days > 0) account(lab, (uint32_t)days, s);
                        if (lab != 0u && e > b_cur) { pend_lab = lab; pend_s = s; pend_e = e; state = 1; }
                    }
                }
            }
            if (!__any_sync(0xffffffffu, state != 1)) break;      // every lane has reached the end of its season
            // some lane ran out of queued words: extract as many as fit the fullest queue (a word adds at most one entry)
            const int room = kScanQ - (int)__reduce_max_sync(0xffffffffu, open ? qw - qr : 0u);
            if (room == 0) break;                                 // blocked by a lane waiting for its next season: close those first
            extract(min(room, K + 1 - k_ext), open);
        }
        if (open && state == 1) flush();
    }
}

// ----------------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------------
static_assert(kTileDoy == 32, "word_length (seams.h) cuts words at 32-day blocks of the day-of-year axis");

// Cuts the time axis into hot-day words (word_length) and groups them by day-of-year block.
static int build_words(const int32_t *doy_map, int64_t T, int n_doy, WordPlan &plan)
{
    plan.n_blk = (n_doy + kTileDoy - 1) / kTileDoy;
    for (int64_t t = 0; t < T;) {
        const int d0 = doy_map[t];
        if (d0 < 0 || d0 >= n_doy) return HDP_B200_ERR_INVALID;
        const int nb = word_length(doy_map, t, T);
        plan.words.push_back(make_int4((int)t, nb, d0, 0));
        t += nb;
    }
    const int K = (int)plan.words.size();
    plan.blk_start.assign(plan.n_blk + 1, 0);
    for (int k = 0; k < K; k++) plan.blk_start[plan.words[k].z / kTileDoy + 1]++;
    for (int b = 0; b < plan.n_blk; b++) plan.blk_start[b + 1] += plan.blk_start[b];
    plan.blk_words.resize(K);
    std::vector<int> fill(plan.blk_start.begin(), plan.blk_start.end() - 1);
    for (int k = 0; k < K; k++) plan.blk_words[fill[plan.words[k].z / kTileDoy]++] = k;
    return HDP_B200_OK;
}

static int64_t words_upper_bound(int64_t T, int n_doy)
{
    // regular daily calendars: every (partial) year contributes at most n_blk + 1 words
    const int64_t n_blk = (n_doy + kTileDoy - 1) / kTileDoy;
    return (T / std::max(n_doy, 1) + 2) * (n_blk + 1) + 1;
}

static int64_t count_words(const int32_t *doy_map, int64_t T)
{
    int64_t K = 0;
    for (int64_t t = 0; t < T; K++) t += word_length(doy_map, t, T);
    return K;
}

// A threshold table without a day-of-year axis (n_doy = 1: the no-season and fixed-value variants, every day reads row 0) would
// cut the series into one-day words, because word_length needs consecutive days of year, and a run of a few decades would then
// have more words than k_scan and k_intensity keep in shared memory.  The pass sees such a table as kTileDoy identical rows
// instead (replicated into the workspace, replicate_rows) with day t on row t mod kTileDoy, so its words are 32 days long.
static int pass_n_doy(int n_doy) { return n_doy == 1 ? kTileDoy : n_doy; }

// The day-of-year map the pass cuts into words: h_doy_map itself, or for n_doy = 1 (where every entry must be 0) t mod kTileDoy.
static int pass_doy_map(const int32_t *h_doy_map, int64_t T, int n_doy, std::vector<int32_t> &own, const int32_t *&map)
{
    map = h_doy_map;
    if (n_doy != 1) return HDP_B200_OK;
    own.resize((size_t)T);
    for (int64_t t = 0; t < T; t++) {
        if (h_doy_map[t] != 0) return HDP_B200_ERR_INVALID;
        own[(size_t)t] = (int32_t)(t % kTileDoy);
    }
    map = own.data();
    return HDP_B200_OK;
}

// thr [C, 1, P] -> rep [C, kTileDoy, P]: row 0 of every cell, then copies that double the rows already there.
static int replicate_rows(const double *thr, int64_t C, int P, double *rep, cudaStream_t st)
{
    const size_t row = (size_t)P * sizeof(double), pitch = kTileDoy * row;
    HDP_CUDA_TRY(cudaMemcpy2DAsync(rep, pitch, thr, row, row, (size_t)C, cudaMemcpyDeviceToDevice, st));
    for (int n = 1; n < kTileDoy; n *= 2)
        HDP_CUDA_TRY(cudaMemcpy2DAsync(rep + (size_t)n * P, pitch, rep, pitch, n * row, (size_t)C, cudaMemcpyDeviceToDevice, st));
    return HDP_B200_OK;
}

int pick_pg(int P)
{
    const int cand[] = {4, 8, 10, 16, 20};
    int best = 4, best_waste = INT_MAX;
    for (int pg : cand) {
        const int waste = (P + pg - 1) / pg * pg - P;
        if (waste < best_waste || (waste == best_waste && pg > best && pg <= 20)) { best = pg; best_waste = waste; }
    }
    return best;
}

// Workspace layout; `intensity` appends the intensity pass's season tables behind what the metric pass uses, then each of the
// n_measures measures its normalised copy (need_norm[m]) and, for n_doy = 1, its replicated thresholds.
static Layout carve(void *ws, size_t ws_bytes, int64_t C, int64_t T, int n_measures, const bool *need_norm, int64_t K, int n_doy, int P,
                    int Y, bool intensity)
{
    Layout L;
    Carver cv(ws, ws_bytes);
    L.words = cv.take<int4>((size_t)K + 1);
    L.blk_start = cv.take<int>((size_t)(pass_n_doy(n_doy) + kTileDoy - 1) / kTileDoy + 1);
    L.blk_words = cv.take<int>((size_t)K + 1);
    L.seasons = cv.take<int4>((size_t)2 * (Y + 1));
    L.lut = cv.take<uint32_t>((size_t)2 * 8192);
    L.hot = cv.take<uint32_t>((size_t)P * K * C);
    if (intensity) L.int_seasons = cv.take<int4>((size_t)2 * (Y + 1));
    for (int m = 0; m < n_measures; m++) {
        if (need_norm[m]) L.xn[m] = cv.take<float>((size_t)C * T);
        if (n_doy == 1) L.thr_rep[m] = cv.take<double>((size_t)C * kTileDoy * P);
    }
    L.total = cv.off;
    return L;
}

static bool bad_dims(int64_t C, int64_t T, int n_doy, int P)
{
    return C < 0 || T < 0 || n_doy <= 0 || P <= 0 || T > 0x3fffffff;
}

size_t metric_pass_workspace_bytes(int64_t C, int64_t T, const int64_t *ld_c, int n_measures, int n_doy, int P, int Y,
                                   const int32_t *h_doy_map, bool intensity)
{
    if (bad_dims(C, T, n_doy, P) || Y < 0) return 0;
    const int64_t K = n_doy == 1 ? (T + kTileDoy - 1) / kTileDoy : h_doy_map ? count_words(h_doy_map, T) : words_upper_bound(T, n_doy);
    bool need_norm[2] = {};
    for (int m = 0; m < n_measures; m++) need_norm[m] = ld_c[m] != 1;
    return carve(nullptr, 0, C, T, n_measures, need_norm, K, n_doy, P, Y, intensity).total;
}

// Prepares each of the n_measures measures (its thresholds replicated for n_doy = 1, its samples copied to time-major L.xn[m], ld_t
// = C, when ld_c != 1) and runs k_hot_words on one measure, k_hot_pair on two: the words then mark the days on which both measures
// pass their thresholds.  On success plan / L describe what lives in the workspace, L.thr / L.n_doy the thresholds and L.x / L.ld_t
// the samples the kernels read.  `unit` is a plain unit code (0 - 2); `cold` makes the words cold-day bits.
static int run_hot_words(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                         int Y, void *ws, size_t ws_bytes, cudaStream_t st, WordPlan &plan, Layout &L,
                         int64_t carve_cells = 0, bool tables_resident = false, int unit = 0, bool intensity = false, bool cold = false)
{
    if (unit < 0 || unit > 2) return HDP_B200_ERR_INVALID;
    std::vector<int32_t> own_map;
    const int32_t *doy_map = nullptr;
    int rc = pass_doy_map(h_doy_map, T, n_doy, own_map, doy_map);
    if (rc != HDP_B200_OK) return rc;
    rc = build_words(doy_map, T, pass_n_doy(n_doy), plan);
    if (rc != HDP_B200_OK) return rc;
    const int K = (int)plan.words.size();
    bool need_norm[2] = {};
    for (int m = 0; m < n_measures; m++) need_norm[m] = ms[m].ld_c != 1;
    L = carve(ws, ws_bytes, std::max(C, carve_cells), T, n_measures, need_norm, K, n_doy, P, Y, intensity);
    if (ws == nullptr || L.total > ws_bytes) return HDP_B200_ERR_WORKSPACE;
    L.n_doy = pass_n_doy(n_doy);
    for (int m = 0; m < n_measures; m++) {
        L.thr[m] = ms[m].thr;
        L.x[m] = ms[m].x;
        L.ld_t[m] = ms[m].ld_t;
    }
    if (C == 0 || T == 0) return HDP_B200_OK;
    for (int m = 0; m < n_measures; m++) {
        if (L.thr_rep[m]) {
            rc = replicate_rows(ms[m].thr, C, P, L.thr_rep[m], st);
            if (rc != HDP_B200_OK) return rc;
            L.thr[m] = L.thr_rep[m];
        }
        if (L.xn[m]) {
            rc = normalize_layout(ms[m].x, C, T, ms[m].ld_t, ms[m].ld_c, L.xn[m], st);
            if (rc != HDP_B200_OK) return rc;
            L.x[m] = L.xn[m];
            L.ld_t[m] = C;
        }
    }
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.words, plan.words.data(), sizeof(int4) * K, cudaMemcpyHostToDevice, st));
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.blk_start, plan.blk_start.data(), sizeof(int) * plan.blk_start.size(), cudaMemcpyHostToDevice, st));
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.blk_words, plan.blk_words.data(), sizeof(int) * K, cudaMemcpyHostToDevice, st));
    if (n_measures == 2) return run_hot_pair(L, plan, C, P, st, unit, cold);

    const int pg = pick_pg(P);
    const int Ppad = (P + pg - 1) / pg * pg;
    const size_t smem = (size_t)kTileDoy * Ppad * kTilePad * sizeof(float);
    dim3 grid((unsigned)((C + kTileCells - 1) / kTileCells), (unsigned)plan.n_blk);
    const auto kernel = hot_kernel(pg, unit, cold, [](auto PG, auto U, auto CO) {
        return k_hot_words<decltype(PG)::value, decltype(U)::value, decltype(CO)::value>;
    });
    KernelTimer timer(kHotWords, st);
    HDP_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, 256, smem, st>>>(L.x[0], C, L.ld_t[0], L.thr[0], L.n_doy, P, L.words, L.blk_start, L.blk_words, K, L.hot);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

// k_scan's season tables: per hemisphere, passes of sorted, disjoint seasons (one launch each).
struct ScanSeason { int a, b, row; };
using ScanPasses = std::vector<std::vector<ScanSeason>>;

// Splits a hemisphere's season table (season_table, sorted by start) into passes: each season goes to the first pass it does
// not overlap.  Seasons of more than 65 535 days do not fit the u16 output.
static int scan_passes(const int32_t *tab, int Y, ScanPasses &passes)
{
    for (int y = 0; y < Y; y++) {
        const ScanSeason s = {tab[4 * y], tab[4 * y + 1], tab[4 * y + 2]};
        if (s.b - s.a > 65535) return HDP_B200_ERR_UNSUPPORTED;
        size_t i = 0;
        while (i < passes.size() && passes[i].back().b > s.a) i++;
        if (i == passes.size()) passes.emplace_back();
        passes[i].push_back(s);
    }
    return HDP_B200_OK;
}

// What k_scan runs for a definition set and its season passes: the bit-sliced definition tables and the instantiation.
// run_scan launches it and hdp_b200_metrics_kernel_choice reports it.
struct ScanConfig {
    ScanTables tabs;
    std::vector<uint32_t> lut;       // [ge_len] definitions with min_dur <= len, then [brk_len] definitions with max_break < gap
    bool bytes = true;               // 8-bit accumulator lanes (four definitions per register), else 16-bit (two)
    int ng = 0, ks = 0;              // accumulator registers (template NG), bit planes of the max_subs counters (template KS)
    int lmin = 0, bmax = 0;          // compile-time run-filter constants of the instantiation; 0, 0 = run-time values
    size_t n_pass = 0;               // launches: the larger pass count of the two hemispheres
};

static int scan_config(const int32_t *h_defs, int D, int64_t T, const ScanPasses (&passes)[2], ScanConfig &cfg)
{
    cfg.n_pass = std::max(passes[0].size(), passes[1].size());
    // bit-sliced definition tables (see k_scan)
    ScanTables &tabs = cfg.tabs;
    int max_min_dur = 0, max_break_all = 0;
    int64_t max_subs_all = 0;
    std::vector<int64_t> subs(D);
    for (int i = 0; i < D; i++) {
        max_min_dur = std::max(max_min_dur, h_defs[3 * i]);
        max_break_all = std::max(max_break_all, h_defs[3 * i + 1]);
        subs[i] = std::min<int64_t>(std::max<int64_t>(h_defs[3 * i + 2], 0), T);   // more subsequent events than days cannot happen
        max_subs_all = std::max(max_subs_all, subs[i]);
    }
    if (max_min_dur > 8190 || max_break_all > 8190) return HDP_B200_ERR_UNSUPPORTED;
    tabs.ge_len = max_min_dur + 2;
    tabs.brk_len = max_break_all + 2;
    int ks_needed = 1;
    while ((max_subs_all >> ks_needed) != 0) ks_needed++;
    for (int k = 0; k < 32; k++) {
        tabs.max_subs_plane[k] = 0u;
        for (int i = 0; i < D; i++) tabs.max_subs_plane[k] |= (uint32_t)((subs[i] >> k) & 1) << i;
    }
    cfg.lut.assign(tabs.ge_len + tabs.brk_len, 0u);
    for (int l = 0; l < tabs.ge_len; l++)
        for (int i = 0; i < D; i++) if (h_defs[3 * i] <= l) cfg.lut[l] |= 1u << i;
    for (int g = 0; g < tabs.brk_len; g++)
        for (int i = 0; i < D; i++) if (h_defs[3 * i + 1] < g) cfg.lut[tabs.ge_len + g] |= 1u << i;
    // run filter (see k_scan): only when the look-back / look-ahead fits the 32-day neighbourhood
    int min_min_dur = INT_MAX;
    for (int i = 0; i < D; i++) min_min_dur = std::min(min_min_dur, h_defs[3 * i]);
    tabs.f_lmin = min_min_dur;
    tabs.f_bmax = max_break_all;
    tabs.f_on = (min_min_dur >= 2 && min_min_dur <= 32 && max_break_all >= 0 && max_break_all <= 30 && g_scan_filter) ? 1 : 0;
    // accumulators: four definitions per register when every season fits 8-bit lanes, else two
    int max_season = 0;
    for (int h = 0; h < 2; h++)
        for (const auto &pass : passes[h])
            for (const ScanSeason &se : pass) max_season = std::max(max_season, se.b - se.a);
    cfg.bytes = max_season <= 255;
    const int per = cfg.bytes ? 4 : 2;
    const int ng = (D + per - 1) / per;
    cfg.ng = ng <= 2 ? 2 : ng <= 3 ? 3 : ng <= 4 ? 4 : ng <= 6 ? 6 : ng <= 8 ? 8 : ng <= 12 ? 12 : 16;
    cfg.ks = ks_needed <= 1 ? 1 : ks_needed <= 2 ? 2 : 32;          // bit planes of the max_subs counters: 1, 2 or all 32
    // compile-time filter constants for the usual shapes (seasons of at most 255 days, common definition sets)
    if (cfg.bytes && cfg.ks == 1 && tabs.f_on && tabs.f_lmin == 3 && (tabs.f_bmax == 1 || tabs.f_bmax == 2)) {
        cfg.lmin = 3;
        cfg.bmax = tabs.f_bmax;
    }
    return HDP_B200_OK;
}

// k_scan over the hot words in L (one launch per pass): the integer metrics u16 [4, P, D, Y, C], with `onset` u16 [6, P, D, Y, C]
// (HWO, HWE behind them, from the ONSET twin of the same instantiation).
static int run_scan(const Layout &L, const WordPlan &plan, int64_t C, int64_t T, int P, const int32_t *h_defs, int D,
                    const ScanPasses (&passes)[2], int Y, const uint8_t *d_is_south, uint16_t *d_out, cudaStream_t st, bool tables_resident,
                    bool onset)
{
    const int K = (int)plan.words.size();
    ScanConfig cfg;
    const int rc = scan_config(h_defs, D, T, passes, cfg);
    if (rc != HDP_B200_OK) return rc;
    const ScanTables &tabs = cfg.tabs;
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.lut, cfg.lut.data(), sizeof(uint32_t) * cfg.lut.size(), cudaMemcpyHostToDevice, st));
    const uint32_t *ge_tab = L.lut, *brk_tab = L.lut + tabs.ge_len;
    size_t scan_smem = (((size_t)kScanWarps * kScanQueueWords + cfg.lut.size() + 3) & ~(size_t)3) * sizeof(uint32_t) + ((size_t)K + 1) * sizeof(int4);
    if (scan_smem > 200 * 1024) return HDP_B200_ERR_UNSUPPORTED;             // > ~9 000 hot words (~800 years of daily data)
    if (cfg.bytes) scan_smem += 256 * sizeof(uint32_t);                      // k_scan's hwa_rcp
    const int64_t n_warps = ((C + 31) / 32) * P;                             // one warp per (32 cells, percentile)
    const unsigned scan_grid = (unsigned)((n_warps + kScanWarps - 1) / kScanWarps);

    // all passes of both hemispheres live side by side in the workspace: north passes, then south passes
    std::vector<int4> tab;
    std::vector<size_t> off[2];
    for (int h = 0; h < 2; h++)
        for (const auto &pass : passes[h]) {
            off[h].push_back(tab.size());
            for (const ScanSeason &s : pass) tab.push_back(make_int4(s.a, s.b, s.row, 0));
        }
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.seasons, tab.data(), sizeof(int4) * tab.size(), cudaMemcpyHostToDevice, st));
    for (size_t ip = 0; ip < cfg.n_pass; ip++) {
        const int4 *sn = ip < passes[0].size() ? L.seasons + off[0][ip] : L.seasons;
        const int4 *ss = ip < passes[1].size() ? L.seasons + off[1][ip] : L.seasons;
        const int nn = ip < passes[0].size() ? (int)passes[0][ip].size() : 0;
        const int ns = ip < passes[1].size() ? (int)passes[1][ip].size() : 0;
        KernelTimer timer(kScan, st);
        // the instantiation, with ONSET = ON
        auto launch = [&](auto on) -> int {
            constexpr bool ON = decltype(on)::value;
#define HDP_LAUNCH_SCAN(NG, KS, BY)                                                                                      \
            do {                                                                                                             \
                HDP_CUDA_TRY(cudaFuncSetAttribute(k_scan<NG, KS, BY, 0, 0, ON>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem)); \
                k_scan<NG, KS, BY, 0, 0, ON><<<scan_grid, kScanWarps * 32, scan_smem, st>>>(L.hot, C, K, (int)T, L.words, P, D, tabs, ge_tab, brk_tab, \
                                                                                  sn, nn, ss, ns, Y, d_is_south, d_out);     \
            } while (0)
#define HDP_LAUNCH_SCAN_F(NG, BY, LM, BM)                                                                                \
            do {                                                                                                             \
                HDP_CUDA_TRY(cudaFuncSetAttribute(k_scan<NG, 1, BY, LM, BM, ON>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem)); \
                k_scan<NG, 1, BY, LM, BM, ON><<<scan_grid, kScanWarps * 32, scan_smem, st>>>(L.hot, C, K, (int)T, L.words, P, D, tabs, ge_tab, \
                                                                                         brk_tab, sn, nn, ss, ns, Y, d_is_south, d_out); \
            } while (0)
#define HDP_SCAN_KS(NG, BY)                                                \
            switch (cfg.ks) {                                                  \
            case 1:                                                            \
                if (BY && cfg.lmin == 3 && cfg.bmax == 1) HDP_LAUNCH_SCAN_F(NG, true, 3, 1);                          \
                else if (BY && cfg.lmin == 3 && cfg.bmax == 2) HDP_LAUNCH_SCAN_F(NG, true, 3, 2);                     \
                else HDP_LAUNCH_SCAN(NG, 1, BY);                               \
                break;                                                         \
            case 2: HDP_LAUNCH_SCAN(NG, 2, BY); break;                         \
            default: HDP_LAUNCH_SCAN(NG, 32, BY); break;                       \
            }
            if (cfg.bytes) {
                switch (cfg.ng) {                                                  // D <= 32: at most 8 registers of 4
                case 2: HDP_SCAN_KS(2, true); break;
                case 3: HDP_SCAN_KS(3, true); break;
                case 4: HDP_SCAN_KS(4, true); break;
                case 6: HDP_SCAN_KS(6, true); break;
                default: HDP_SCAN_KS(8, true); break;
                }
            } else {
                switch (cfg.ng) {
                case 2: HDP_SCAN_KS(2, false); break;
                case 3: HDP_SCAN_KS(3, false); break;
                case 4: HDP_SCAN_KS(4, false); break;
                case 6: HDP_SCAN_KS(6, false); break;
                case 8: HDP_SCAN_KS(8, false); break;
                case 12: HDP_SCAN_KS(12, false); break;
                default: HDP_SCAN_KS(16, false); break;
                }
            }
#undef HDP_SCAN_KS
#undef HDP_LAUNCH_SCAN_F
#undef HDP_LAUNCH_SCAN
            return HDP_B200_OK;
        };
        const int lrc = onset ? launch(std::true_type()) : launch(std::false_type());
        if (lrc != HDP_B200_OK) return lrc;
        HDP_LAUNCH_CHECK();
    }
    return HDP_B200_OK;
}

// Every measure of a pass must have samples and thresholds once there is work
static bool missing_measure(const Measure *ms, int n_measures, int64_t C, int64_t T)
{
    for (int m = 0; m < n_measures; m++)
        if (C > 0 && T > 0 && (!ms[m].x || !ms[m].thr)) return true;
    return false;
}

int metric_pass(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                const int32_t *h_defs, int D,
                const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                const uint8_t *d_is_south, uint16_t *d_out, float *d_int,
                void *d_workspace, size_t workspace_bytes, void *stream, int64_t carve_cells, bool tables_resident, int input_unit)
{
    if (bad_dims(C, T, n_doy, P) || D <= 0 || Y < 0) return HDP_B200_ERR_INVALID;
    if ((T > 0 && !h_doy_map) || !h_defs || (Y > 0 && (!h_season_north || !h_season_south))) return HDP_B200_ERR_INVALID;
    if (missing_measure(ms, n_measures, C, T)) return HDP_B200_ERR_INVALID;
    if (P > HDP_B200_MAX_PERCENTILES || D > HDP_B200_MAX_DEFINITIONS) return HDP_B200_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    // input_unit of the C ABI = unit code | HDP_B200_COLD | HDP_B200_ONSET; the kernels' launchers see them as plain values
    const bool cold = (input_unit & HDP_B200_COLD) != 0, onset = (input_unit & HDP_B200_ONSET) != 0;
    const int unit = input_unit & ~(HDP_B200_COLD | HDP_B200_ONSET);
    if (onset && !d_out) return HDP_B200_ERR_INVALID;                                   // HWO / HWE are planes of the u16 output

    // the season tables of both hemispheres, north then south (Y + 1 rows apart, as k_intensity reads them)
    std::vector<int32_t> seasons((size_t)8 * (Y + 1), 0);
    ScanPasses passes[2];
    for (int h = 0; h < 2; h++) {
        int32_t *tab = seasons.data() + (size_t)4 * (Y + 1) * h;
        const bool disjoint = intensity_season_table(h == 0 ? h_season_north : h_season_south, Y, T, tab);
        if (d_int && !disjoint) return HDP_B200_ERR_UNSUPPORTED;                        // k_intensity: one open season per lane
        if (d_out) {
            const int rc = scan_passes(tab, Y, passes[h]);
            if (rc != HDP_B200_OK) return rc;
        }
    }

    WordPlan plan;
    Layout L;
    int rc = run_hot_words(ms, n_measures, C, T, n_doy, P, h_doy_map, Y, d_workspace, workspace_bytes, st, plan, L,
                           carve_cells, tables_resident, unit, d_int != nullptr, cold);
    if (rc != HDP_B200_OK || C == 0 || Y == 0) return rc;
    if (d_out) {
        rc = run_scan(L, plan, C, T, P, h_defs, D, passes, Y, d_is_south, d_out, st, tables_resident, onset);
        if (rc != HDP_B200_OK) return rc;
    }
    for (int m = 0; d_int && m < n_measures && rc == HDP_B200_OK; m++)     // one block per measure, on the same words
        rc = run_intensity(L, plan, m, C, T, P, h_defs, D, seasons, Y, d_is_south, d_int + (size_t)m * 3 * P * D * Y * C, st,
                           tables_resident || m > 0, unit, cold);
    return rc;
}

// hdp_b200_hot_days and hdp_b200_compound_hot_days: the hot words, unpacked to u8 [P, T, C]
static int hot_days_pass(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                         uint8_t *d_mask, void *d_workspace, size_t workspace_bytes, void *stream, int unit, bool cold)
{
    if (bad_dims(C, T, n_doy, P) || !h_doy_map && T > 0) return HDP_B200_ERR_INVALID;
    if (missing_measure(ms, n_measures, C, T) || (C > 0 && T > 0 && !d_mask)) return HDP_B200_ERR_INVALID;
    if (P > HDP_B200_MAX_PERCENTILES) return HDP_B200_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    WordPlan plan;
    Layout L;
    int rc = run_hot_words(ms, n_measures, C, T, n_doy, P, h_doy_map, 0, d_workspace, workspace_bytes, st, plan, L,
                           0, false, unit, false, cold);
    if (rc != HDP_B200_OK || C == 0 || T == 0) return rc;
    const int K = (int)plan.words.size();
    dim3 grid((unsigned)((C + 255) / 256), (unsigned)K);
    if (K > 65535) return HDP_B200_ERR_UNSUPPORTED;
    KernelTimer timer(kUnpackMask, st);
    k_unpack_mask<<<grid, 256, 0, st>>>(L.hot, C, T, P, K, L.words, d_mask);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace hdp

using namespace hdp;

extern "C" {

size_t hdp_b200_metrics_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                        int n_doy, int P, int D, int Y, const int32_t *h_doy_map)
{
    (void)ld_t; (void)D;
    return metric_pass_workspace_bytes(C, T, &ld_c, 1, n_doy, P, Y, h_doy_map, false);
}

void hdp_b200_metrics_run_filter(int on) { g_scan_filter = on != 0; }

int hdp_b200_metrics_kernel_choice(const int32_t *h_defs, int D, const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                                   int64_t T, int *info)
{
    if (!h_defs || !info || D <= 0 || Y < 0 || T < 0 || T > 0x3fffffff || (Y > 0 && (!h_season_north || !h_season_south)))
        return HDP_B200_ERR_INVALID;
    if (D > HDP_B200_MAX_DEFINITIONS) return HDP_B200_ERR_UNSUPPORTED;
    std::vector<int32_t> tab((size_t)4 * (Y + 1));
    ScanPasses passes[2];
    for (int h = 0; h < 2; h++) {
        season_table(h == 0 ? h_season_north : h_season_south, Y, T, tab.data());
        const int rc = scan_passes(tab.data(), Y, passes[h]);
        if (rc != HDP_B200_OK) return rc;
    }
    ScanConfig cfg;
    const int rc = scan_config(h_defs, D, T, passes, cfg);
    if (rc != HDP_B200_OK) return rc;
    info[0] = cfg.bytes ? 8 : 16; info[1] = cfg.ng; info[2] = cfg.ks; info[3] = cfg.tabs.f_on;
    info[4] = cfg.lmin; info[5] = cfg.bmax; info[6] = (int)cfg.n_pass;
    return HDP_B200_OK;
}

int hdp_b200_hot_days(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                      const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                      uint8_t *d_mask, void *d_workspace, size_t workspace_bytes, void *stream)
{
    const Measure m = {d_measure, ld_t, ld_c, d_thr};
    return hot_days_pass(&m, 1, C, T, n_doy, P, h_doy_map, d_mask, d_workspace, workspace_bytes, stream, 0, false);
}

int hdp_b200_compound_hot_days(const float *d_a, int64_t ld_t_a, int64_t ld_c_a, const float *d_b, int64_t ld_t_b, int64_t ld_c_b,
                               int64_t C, int64_t T, const double *d_thr_a, const double *d_thr_b, int n_doy, int P,
                               const int32_t *h_doy_map, uint8_t *d_mask, void *d_workspace, size_t workspace_bytes, void *stream,
                               int input_unit)
{
    const Measure ms[2] = {{d_a, ld_t_a, ld_c_a, d_thr_a}, {d_b, ld_t_b, ld_c_b, d_thr_b}};
    return hot_days_pass(ms, 2, C, T, n_doy, P, h_doy_map, d_mask, d_workspace, workspace_bytes, stream, input_unit & ~HDP_B200_COLD,
                         (input_unit & HDP_B200_COLD) != 0);
}

int hdp_b200_metrics(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                     const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                     const int32_t *h_defs, int D,
                     const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                     const uint8_t *d_is_south, uint16_t *d_out,
                     void *d_workspace, size_t workspace_bytes, void *stream, int input_unit)
{
    if (C > 0 && Y > 0 && !d_out) return HDP_B200_ERR_INVALID;
    const Measure m = {d_measure, ld_t, ld_c, d_thr};
    return metric_pass(&m, 1, C, T, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y, d_is_south, d_out, nullptr,
                       d_workspace, workspace_bytes, stream, C, false, input_unit);
}

}  // extern "C"
