// intensity_host.cpp - TEST INFRASTRUCTURE: replays the lane loop of k_intensity (hdp_b200/csrc/intensity.cu) on the CPU around
// the very same per-run / per-season functions (hdp_b200/csrc/intensity.h, and index_run of seams.h), so that
// tests/test_intensity_host.py can check that logic against the oracle without a GPU.  Not part of the product.
//     g++ -O2 -shared -fPIC -I hdp_b200/csrc tests/intensity_host.cpp -o <tmp>/libintensity_host.so
#include <stdint.h>
#include <vector>

#include "intensity.h"

using namespace hdp;

extern "C" {

// One cell, one percentile: x f32 [T] (Celsius), thr f64 [n_doy], doy_map i32 [T], defs i32 [D, 3], seasons i32 [Y, 2]
// -> out f32 [3, D, Y] (HWC, HWI, HWP).  Returns 0, or -2 for a season table with overlapping non-empty seasons.
int intensity_host_cell(const float *x, const double *thr, const int32_t *doy_map, int64_t T, const int32_t *defs, int D,
                        const int32_t *seasons, int Y, float *out)
{
    std::vector<int32_t> tab((size_t)4 * (Y + 1));
    if (!intensity_season_table(seasons, Y, T, tab.data())) return -2;
    // words of at most 32 days with consecutive days of year that do not cross a 32-day block (metric.cu build_words)
    std::vector<int> w_t0, w_doy;
    for (int64_t t = 0; t < T;) {
        int nb = 1;
        while (t + nb < T && nb < 32 && doy_map[t + nb] == doy_map[t] + nb && (doy_map[t + nb] & 31) != 0) nb++;
        w_t0.push_back((int)t);
        w_doy.push_back(doy_map[t]);
        t += nb;
    }
    const int K = (int)w_t0.size();
    std::vector<IndexState> ist(D);
    std::vector<IntensityAcc> acc(D);
    IntensityLane L;
    L.start(tab.data(), Y);
    auto flush = [&]() {
        for (int d = 0; d < D; d++) {
            intensity_values(acc[d], out[(0 * D + d) * Y + L.row], out[(1 * D + d) * Y + L.row], out[(2 * D + d) * Y + L.row]);
            acc[d] = IntensityAcc();
        }
    };
    int kw = 0;
    auto block = [&](int64_t lo, int64_t hi, double &r, double &m) {
        for (int64_t t = lo; t < hi; t++) {
            while (kw + 1 < K && w_t0[kw + 1] <= t) kw++;
            const int doy = w_doy[kw] + (int)(t - w_t0[kw]);
            intensity_day(r, m, intensity_excess(x[t], thr[doy]));
        }
    };
    int run_start = -1, run_word = 0;
    uint32_t carry = 0u;
    for (int k = 0; k <= K && L.open(); k++) {
        const int t0 = k < K ? w_t0[k] : (int)T;
        const int nb = k + 1 < K ? w_t0[k + 1] - t0 : k < K ? (int)T - t0 : 1;
        uint32_t w = 0u;                                                    // the hot-day word of k_hot_words
        for (int j = 0; j < nb && k < K; j++)
            if ((double)x[t0 + j] > thr[w_doy[k] + j]) w |= 1u << j;
        const uint32_t vmask = nb == 32 ? 0xffffffffu : (1u << nb) - 1u;
        const uint32_t prev = (w << 1) | carry;
        uint32_t starts = w & ~prev, ends = ~w & prev & vmask;
        carry = (w >> (nb - 1)) & 1u;
        while (ends != 0u) {
            int s, ks;
            if (run_start >= 0) { s = run_start; ks = run_word; run_start = -1; }
            else { s = t0 + __builtin_ctz(starts); ks = k; starts &= starts - 1u; }
            const int e = t0 + __builtin_ctz(ends);
            ends &= ends - 1u;
            uint32_t lab = 0u;
            for (int d = 0; d < D; d++)
                if (index_run(ist[d], s, e, defs[3 * d], defs[3 * d + 1], defs[3 * d + 2]) != 0) lab |= 1u << d;
            kw = ks;
            intensity_run(L, s, e, lab, acc.data(), 1, block, flush);
        }
        if (starts != 0u) { run_start = t0 + __builtin_ctz(starts); run_word = k; }
    }
    while (L.open()) { flush(); L.next(); }
    return 0;
}

}  // extern "C"
