// intensity.h - the per-run and per-season accounting of the heatwave intensity metrics (HWC, HWI, HWP), as plain functions
// that compile for the device (intensity.cu, one lane per cell) and for the host (tests/intensity_host.cpp replays the lane
// loop on the CPU against the oracle, the way tests/seams_host.cpp checks seams.h).
//
// Contract (cell c, percentile p, definition d, season y):
//   e_t  = (double)x_c(t) - thr[c, doy(t), p]                    one float64 subtraction, x after the input unit conversion
//   set  = days t of the season slice [lo, hi) whose heatwave id is > 0 (exactly the days HWF counts; every one is hot, e_t > 0)
//   HWC  = S: the maximal blocks of consecutive set days in time order; per block r = 0, r = r + e_t day by day, then S = S + r
//   HWI  = S / HWF (one float64 division; 0 when HWF = 0)
//   HWP  = max e_t over the set (0 when the set is empty)
// each rounded once to float32.  A block is one labelled hot run clipped to the season: distinct runs are separated by at least
// one cold day.
//
// Cold spells (CSC, CSI, CSP; HDP_B200_COLD): the same accounting over the runs of cold days ((double)x < thr) with the deficit
// e_t = thr - (double)x in place of the exceedance (e_t > 0 on every day of the set again).  thr - x is bit for bit the
// exceedance (-x) - (-thr): negation is exact and a - b is a + (-b), so the cold result equals the warm one on negated inputs.
#pragma once

#include <stdint.h>

#include "seams.h"

namespace hdp {

struct IntensityAcc {
    double sum = 0.0;          // S
    double peak = 0.0;         // largest e_t so far (e_t > 0 for every day of the set)
    int64_t days = 0;          // HWF
};

HDP_HD double intensity_excess(float x, double thr) { return (double)x - thr; }
HDP_HD double intensity_deficit(float x, double thr) { return thr - (double)x; }

// e_t of one day: the exceedance of a heatwave pass, the deficit of a cold-spell pass
HDP_HD double intensity_e(float x, double thr, bool cold) { return cold ? intensity_deficit(x, thr) : intensity_excess(x, thr); }

// one day of a block: r = r + e (time order), m = max(m, e)
HDP_HD void intensity_day(double &r, double &m, double e)
{
    r = r + e;
    m = e > m ? e : m;
}

// a block of `days` set days with partial sum r and maximum m, added to one definition's season accumulator
HDP_HD void intensity_block(IntensityAcc &a, double r, double m, int64_t days)
{
    a.sum = a.sum + r;
    a.peak = m > a.peak ? m : a.peak;
    a.days += days;
}

HDP_HD void intensity_values(const IntensityAcc &a, float &hwc, float &hwi, float &hwp)
{
    hwc = (float)a.sum;
    hwi = a.days > 0 ? (float)(a.sum / (double)a.days) : 0.0f;
    hwp = (float)a.peak;
}

// index of the lowest set bit of v != 0
HDP_HD int low_bit(uint32_t v)
{
#ifdef __CUDA_ARCH__
    return __ffs(v) - 1;
#else
    return __builtin_ctz(v);
#endif
}

// ---- season tables ------------------------------------------------------------------------------------------------------
// A lane keeps ONE open season, so a hemisphere's seasons must be disjoint.  Builds tab as season_table (seams.h) does and returns
// whether it qualifies: empty seasons may sit anywhere, but no two non-empty seasons may overlap.
HDP_HD bool intensity_season_table(const int32_t *raw, int Y, int64_t T, int32_t *tab)
{
    season_table(raw, Y, T, tab);
    int64_t end = INT64_MIN;                                                // end of the last non-empty season
    for (int y = 0; y < Y; y++) {
        if (tab[4 * y + 1] == tab[4 * y]) continue;
        if (tab[4 * y] < end) return false;
        end = tab[4 * y + 1];
    }
    return true;
}

// ---- one lane --------------------------------------------------------------------------------------------------------------
// The hot runs [s, e) of one lane in time order, popped from its hot-day words (k_hot_words).  Word k starts at day
// word_t0[k * stride] and ends where word k + 1 starts (the last one at T); bit j is day t0 + j.  Word K is a virtual cold day at
// T that closes a run still open at the end of the series.
struct HotRuns {
    const int *word_t0;
    int stride, K, T;
    int k = 0, t0 = 0;                   // the current word and its first day
    uint32_t starts = 0u, ends = 0u;     // its run starts and run ends not popped yet
    uint32_t carry = 0u;                 // the last day of the previous word was hot
    int open_s = -1, open_k = 0;         // the run still open at the end of the previous word: first day, word of that day

    // word k_ with hot-day bits w (0 for word K)
    HDP_HD void word(int k_, uint32_t w)
    {
        k = k_;
        t0 = k < K ? word_t0[k * stride] : T;
        const int nb = k + 1 < K ? word_t0[(k + 1) * stride] - t0 : k < K ? T - t0 : 1;
        const uint32_t vmask = nb == 32 ? 0xffffffffu : (1u << nb) - 1u;
        const uint32_t prev = (w << 1) | carry;
        starts = w & ~prev;
        ends = ~w & prev & vmask;
        carry = (w >> (nb - 1)) & 1u;
    }
    // the next run that ends in the current word, and the word ks of its first day; false when none is left
    HDP_HD bool pop(int &s, int &e, int &ks)
    {
        if (ends == 0u) {
            if (starts != 0u) { open_s = t0 + low_bit(starts); open_k = k; starts = 0u; }   // (at most one: it ends later)
            return false;
        }
        if (open_s >= 0) { s = open_s; ks = open_k; open_s = -1; }
        else { s = t0 + low_bit(starts); ks = k; starts &= starts - 1u; }
        e = t0 + low_bit(ends);
        ends &= ends - 1u;
        return true;
    }
};

// The hot run [s, e) through every definition's index_heatwaves state machine (st[d * stride]; defs i32 [D, 3]): bit d of the
// result is set when definition d labels the run.
HDP_HD uint32_t label_run(IndexState *st, int stride, const int *defs, int D, int64_t s, int64_t e)
{
    uint32_t lab = 0u;
    for (int d = 0; d < D; d++) {
        IndexState sd = st[d * stride];
        if (index_run(sd, s, e, defs[3 * d], defs[3 * d + 1], defs[3 * d + 2]) != 0) lab |= 1u << d;
        st[d * stride] = sd;
    }
    return lab;
}

struct IntensityLane {
    const int32_t *seas = nullptr;   // i32 [n, 4] as built by season_table
    int n = 0, ys = 0;
    int64_t a = 0, b = 0;            // the open season [a, b)
    int row = 0;                     // its output row
    HDP_HD void start(const int32_t *s, int n_) { seas = s; n = n_; ys = -1; next(); }
    HDP_HD void next()
    {
        ys++;
        if (ys < n) { a = seas[4 * ys]; b = seas[4 * ys + 1]; row = seas[4 * ys + 2]; }
    }
    HDP_HD bool open() const { return ys < n; }
};

// The hot run [s, e), labelled by the definitions whose bit is set in `lab` (D <= 32), reaches the lane.  Every season that ends
// at or before s is closed first (flush() writes acc of the open season to row L.row and clears it); then each season the run
// overlaps receives the run's in-season block: block(lo, hi, r, m) adds e_t of the days lo .. hi - 1 in time order
// (intensity_day), and every labelling definition's accumulator (acc[d * stride]) takes it.  A season that ends inside the run is
// closed at once.
template <class Block, class Flush>
HDP_HD void intensity_run(IntensityLane &L, int64_t s, int64_t e, uint32_t lab, IntensityAcc *acc, int stride, Block &&block,
                          Flush &&flush)
{
    while (L.open() && L.b <= s) { flush(); L.next(); }
    if (lab == 0u) return;
    while (L.open() && L.a < e) {
        const int64_t lo = s > L.a ? s : L.a, hi = e < L.b ? e : L.b;
        if (hi > lo) {
            double r = 0.0, m = 0.0;
            block(lo, hi, r, m);
            for (uint32_t bits = lab; bits != 0u; bits &= bits - 1u) intensity_block(acc[low_bit(bits) * stride], r, m, hi - lo);
        }
        if (e <= L.b) break;
        flush();
        L.next();
    }
}

}  // namespace hdp
