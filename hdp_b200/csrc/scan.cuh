// scan.cuh - k_scan, the run scan of the metric pass, and its launcher.  metric.cu instantiates the plain and ONSET instances,
// extent.cu the EXTENT twins (a translation unit of their own, so that the parallel build is not bound by metric.cu).
#pragma once

#include <limits.h>
#include <vector>

#include "intensity.h"
#include "metric.cuh"

namespace hdp {

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

// *p += v, two's complement, without a return value
__device__ __forceinline__ void red_add_u64(int64_t *p, uint64_t v)
{
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
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
// EXTENT: also the heatwave spatial extent.  Every in-season block [lo, lo + days) that account() credits to the definitions `lab`
// adds +w at diff[r, p, i, lo] and -w at diff[r, p, i, lo + days] for each definition i in lab (w, r: the lane's cell's weight and
// region), so the prefix sum over t of a diff row (k_extent_prefix, extent.cu) is the weighted count of cells on a heatwave day on
// day t.  Lanes that emit nothing (padding lanes, cells in no region) have w = 0.  The flush stores only when `out` is given.
template <int NG, int KS, bool kBytes, int LMIN = 0, int BMAX = 0, bool ONSET = false, bool EXTENT = false>
__global__ void __launch_bounds__(kScanWarps * 32, 3)
k_scan(const uint32_t *__restrict__ hot, int64_t C, int K, int T, const int4 *__restrict__ words,
       int P, int D, const __grid_constant__ ScanTables tabs, const uint32_t *__restrict__ ge_tab, const uint32_t *__restrict__ brk_tab,
       const int4 *__restrict__ seasons_north, int n_north, const int4 *__restrict__ seasons_south, int n_south, int Y,
       const uint8_t *__restrict__ is_south, uint16_t *__restrict__ out, const __grid_constant__ ScanExtent ext)
{
    static_assert(!(ONSET && EXTENT), "onset and extent are not combined");
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
    uint32_t ext_w = 0u;                                          // EXTENT: this lane's weight, and its region's diff rows
    int64_t *ext_rows = nullptr;
    if constexpr (EXTENT) {
        const int r = ext.region != nullptr ? ext.region[c] : 0;
        if (alive && r >= 0 && r < ext.R) {
            ext_w = ext.weight != nullptr ? ext.weight[c] : 1u;
            ext_rows = ext.diff + ((int64_t)r * P + p) * D * ((int64_t)T + 1);
        }
    }

    // metric m of definition d, season row r of this lane's cell: out_pc[m * P * D * Y * C + d * Y * C + r * C]
    uint16_t *const out_pc = out + (int64_t)p * D * Y * C + c;
    auto lane_of = [](uint32_t v, int h) -> uint32_t {            // accumulator lane h of a register, zero-extended (one PRMT)
        return kBytes ? __byte_perm(v, 0u, 0x4440 + h) : (v >> (BITS * h)) & LANE_MASK;
    };
    auto flush = [&]() {                                          // close season `ys`
        if (alive && (!EXTENT || out != nullptr)) {
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
        if constexpr (EXTENT) {
            if (ext_w != 0u) {
                const int lo = max(s, a_cur);
                for (uint32_t m = lab; m != 0u; m &= m - 1u) {
                    int64_t *const row = ext_rows + (int64_t)(__ffs(m) - 1) * ((int64_t)T + 1);
                    red_add_u64(row + lo, ext_w);
                    red_add_u64(row + lo + days, 0ull - ext_w);
                }
            }
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

// One k_scan launch: grid, shared memory and every kernel argument but the definition tables of the ScanConfig
struct ScanLaunch {
    unsigned grid = 0;
    size_t smem = 0;
    cudaStream_t st = nullptr;
    const uint32_t *hot = nullptr;
    int64_t C = 0;
    int K = 0, T = 0;
    const int4 *words = nullptr;
    int P = 0, D = 0;
    const uint32_t *ge_tab = nullptr, *brk_tab = nullptr;
    const int4 *sn = nullptr, *ss = nullptr;
    int nn = 0, ns = 0, Y = 0;
    const uint8_t *is_south = nullptr;
    uint16_t *out = nullptr;
    ScanExtent ext;
};

// Launches the instantiation cfg names, with ONSET = ON and EXTENT = EX.  Instantiated in metric.cu (EX = false) and extent.cu
// (EX = true), so that each translation unit compiles its own kernels only.
template <bool ON, bool EX>
int launch_scan(const ScanConfig &cfg, const ScanLaunch &a)
{
#define HDP_LAUNCH_SCAN(NG, KS, BY, LM, BM)                                                                                       \
    do {                                                                                                                          \
        HDP_CUDA_TRY(cudaFuncSetAttribute(k_scan<NG, KS, BY, LM, BM, ON, EX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)a.smem)); \
        k_scan<NG, KS, BY, LM, BM, ON, EX><<<a.grid, kScanWarps * 32, a.smem, a.st>>>(a.hot, a.C, a.K, a.T, a.words, a.P, a.D, cfg.tabs,     \
                                                                                    a.ge_tab, a.brk_tab, a.sn, a.nn, a.ss, a.ns, a.Y,      \
                                                                                    a.is_south, a.out, a.ext);                            \
    } while (0)
#define HDP_SCAN_KS(NG, BY)                                                                                                       \
    switch (cfg.ks) {                                                                                                             \
    case 1:                                                                                                                       \
        if (BY && cfg.lmin == 3 && cfg.bmax == 1) HDP_LAUNCH_SCAN(NG, 1, true, 3, 1);                                             \
        else if (BY && cfg.lmin == 3 && cfg.bmax == 2) HDP_LAUNCH_SCAN(NG, 1, true, 3, 2);                                        \
        else HDP_LAUNCH_SCAN(NG, 1, BY, 0, 0);                                                                                    \
        break;                                                                                                                    \
    case 2: HDP_LAUNCH_SCAN(NG, 2, BY, 0, 0); break;                                                                              \
    default: HDP_LAUNCH_SCAN(NG, 32, BY, 0, 0); break;                                                                            \
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
#undef HDP_LAUNCH_SCAN
    return HDP_B200_OK;
}
extern template int launch_scan<false, true>(const ScanConfig &, const ScanLaunch &);     // (extent.cu)

}  // namespace hdp
