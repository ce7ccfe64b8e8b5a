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

// ---- season tables ------------------------------------------------------------------------------------------------------
// A lane keeps ONE open season, so a hemisphere's seasons must be disjoint.  raw i32 [Y, 2] (Python slice semantics) ->
// tab i32 [Y, 4] {lo, hi, row, 0} sorted by lo (stable).  Empty seasons may sit anywhere; any two non-empty seasons must not
// overlap.  Returns false otherwise.
HDP_HD bool intensity_season_table(const int32_t *raw, int Y, int64_t T, int32_t *tab)
{
    for (int y = 0; y < Y; y++) {
        int64_t lo, hi;
        season_slice(raw[2 * y], raw[2 * y + 1], T, lo, hi);
        int i = y;                                                          // insertion sort by lo, stable
        while (i > 0 && tab[4 * (i - 1)] > lo) {
            for (int k = 0; k < 4; k++) tab[4 * i + k] = tab[4 * (i - 1) + k];
            i--;
        }
        tab[4 * i] = (int32_t)lo; tab[4 * i + 1] = (int32_t)hi; tab[4 * i + 2] = y; tab[4 * i + 3] = 0;
    }
    int64_t end = INT64_MIN;                                                // end of the last non-empty season
    for (int y = 0; y < Y; y++) {
        if (tab[4 * y + 1] == tab[4 * y]) continue;
        if (tab[4 * y] < end) return false;
        end = tab[4 * y + 1];
    }
    return true;
}

// ---- one lane --------------------------------------------------------------------------------------------------------------
struct IntensityLane {
    const int32_t *seas = nullptr;   // i32 [n, 4] as built by intensity_season_table
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
            for (uint32_t bits = lab; bits != 0u; bits &= bits - 1u) {
#ifdef __CUDA_ARCH__
                const int d = __ffs(bits) - 1;
#else
                const int d = __builtin_ctz(bits);
#endif
                intensity_block(acc[d * stride], r, m, hi - lo);
            }
        }
        if (e <= L.b) break;
        flush();
        L.next();
    }
}

}  // namespace hdp
