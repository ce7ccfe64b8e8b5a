// seams.h - the per-run and per-season logic of the reference's path-2 BUILDING BLOCKS, as plain functions that compile for
// the device (seams.cu) and for the host (tests/seams_host.cpp, which replays the kernels' lane loops on the CPU against the
// oracle: the logic below is checked without a GPU, the kernels add only the warp plumbing around it).  It also holds the two
// rules of the fused pass that its host replay (tests/intensity_host.cpp) shares: the season table and the cut into hot-day words.
//
// Reference = AgentOxygen/HDP v1.0.2:
//   index_heatwaves      hdp/metric.py:11-60
//   heatwave_number      hdp/metric.py:63-82
//   heatwave_frequency   hdp/metric.py:85-102
//   heatwave_duration    hdp/metric.py:105-137
//   heatwave_average     hdp/metric.py:140-172
#pragma once

#include <stdint.h>

#ifdef __CUDACC__
#define HDP_HD __host__ __device__ __forceinline__
#else
#define HDP_HD inline
#endif

namespace hdp {

// ---- index_heatwaves ------------------------------------------------------------------------------------------------------
// The reference walks the transitions of the zero-padded mask (metric.py:27-41).  A hot run [s, e) is a +1 transition at s whose
// next transition is the -1 at e; the -1 transition of the PREVIOUS run sees `s - prev_e` cold days (branch B, :47-48) and is
// visited before this run's +1.  So one call per hot run, in time order, reproduces the loop.
struct IndexState {
    int64_t id = 0;            // current_hw_index
    int64_t sub = 0;           // sub_events: reset in branch D only - it carries across heatwaves ended by a break (:58)
    int64_t prev_e = 0;        // first cold day after the previous run
    bool in_hw = false;
    bool has_prev = false;
};

// Label of the hot run [s, e): the heatwave id written to hw[s:e], or 0 if the run stays unlabelled.
HDP_HD int64_t index_run(IndexState &st, int64_t s, int64_t e, int64_t min_duration, int64_t max_break, int64_t max_subs)
{
    if (st.has_prev && s - st.prev_e > max_break) st.in_hw = false;        // B (:47-48)
    st.prev_e = e;
    st.has_prev = true;
    const int64_t len = e - s;
    if (len >= min_duration && !st.in_hw) {                                 // A (:43-46)
        st.id += 1;
        st.in_hw = true;
        return st.id;
    }
    if (st.in_hw && st.sub < max_subs) {                                    // C (:49-51): any length
        st.sub += 1;
        return st.id;
    }
    if (st.in_hw) {                                                         // D (:52-58)
        int64_t label = 0;
        if (len >= min_duration) {
            st.id += 1;
            label = st.id;
        } else {
            st.in_hw = false;
        }
        st.sub = 0;
        return label;
    }
    return 0;
}

// ---- season slices --------------------------------------------------------------------------------------------------------
// hw_ts[a:b] with Python's slice rules (metric.py:79,100,122,157) -> 0 <= lo <= hi <= T
HDP_HD void season_slice(int64_t a, int64_t b, int64_t T, int64_t &lo, int64_t &hi)
{
    if (a < 0) { a += T; if (a < 0) a = 0; }
    if (b < 0) { b += T; if (b < 0) b = 0; }
    if (a > T) a = T;
    if (b > T) b = T;
    if (b < a) b = a;
    lo = a;
    hi = b;
}

// raw i32 [Y, 2] (season_slice semantics) -> tab i32 [Y, 4] {lo, hi, row, 0}, stably sorted by lo: the season table of one
// hemisphere as the fused metric pass (metric.cu) and its intensity kernel walk it.
HDP_HD void season_table(const int32_t *raw, int Y, int64_t T, int32_t *tab)
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
}

// ---- hot-day words --------------------------------------------------------------------------------------------------------
// The fused metric pass cuts the time axis into words of <= 32 consecutive days whose days of year are consecutive and stay inside
// one 32-day block of the day-of-year axis, so that every word of a block shares one threshold tile (k_hot_words, metric.cu).
// Length of the word that starts at day t.
HDP_HD int word_length(const int32_t *doy_map, int64_t t, int64_t T)
{
    int nb = 1;
    while (t + nb < T && nb < 32 && doy_map[t + nb] == doy_map[t] + nb && (doy_map[t + nb] & 31) != 0) nb++;
    return nb;
}

// What one lane of a warp adds up over its elements i = lane, lane + n_lanes, ... of the slice v[0 .. n).
// `multi` = the slice holds more than one distinct value; `vmin` = its smallest value.  The reference takes np.unique of the
// slice and - when there is more than one distinct value - drops the FIRST (smallest) one whatever it is (:124-128: it is
// the 0 of the cold days whenever heatwaves are separated by cold days); every remaining distinct value contributes the
// number of days that carry it, a remaining 0 contributes 0 (:131-134).
struct SeasonAcc {
    int64_t hot = 0;           // days with id > 0                      -> HWF
    int64_t uniq = 0;          // distinct values                       -> length of hw_lengths
    int64_t uniq_nz = 0;       // distinct non-zero values              -> HWN
    int64_t sum = 0;           // sum of hw_lengths                     -> HWA numerator
    int64_t longest = 0;       // max of hw_lengths                     -> HWD
};

HDP_HD void season_lane(const int64_t *v, int64_t n, int lane, int n_lanes, bool multi, int64_t vmin, SeasonAcc &acc)
{
    for (int64_t i = lane; i < n; i += n_lanes) {
        const int64_t x = v[i];
        acc.hot += x > 0;
        int64_t count = 0;
        bool first = true;                                                  // no earlier day carries the same value
        for (int64_t j = 0; j < n; j++) {
            const bool eq = v[j] == x;
            count += eq;
            if (eq && j < i) first = false;
        }
        if (!first) continue;
        acc.uniq += 1;
        acc.uniq_nz += x != 0;
        if (multi && x == vmin) continue;                                   // unique_indices[1:]
        const int64_t len = x != 0 ? count : 0;
        acc.sum += len;
        if (len > acc.longest) acc.longest = len;
    }
}

HDP_HD void season_merge(SeasonAcc &a, const SeasonAcc &b)
{
    a.hot += b.hot;
    a.uniq += b.uniq;
    a.uniq_nz += b.uniq_nz;
    a.sum += b.sum;
    if (b.longest > a.longest) a.longest = b.longest;
}

// np.mean(hw_lengths) (:171): Numba accumulates the int64 lengths in float64 and divides by the element count.  An empty
// slice has no lengths at all (the reference raises there: the host layer does the same before launching); 0 is stored.
HDP_HD double season_average(const SeasonAcc &a, int64_t n, bool multi)
{
    if (n <= 0) return 0.0;
    return (double)a.sum / (double)(multi ? a.uniq - 1 : 1);
}

}  // namespace hdp
