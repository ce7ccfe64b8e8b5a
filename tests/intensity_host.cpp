// intensity_host.cpp - TEST INFRASTRUCTURE: replays the lane loop of k_intensity (hdp_b200/csrc/intensity.cu) on the CPU around
// the very same functions (hdp_b200/csrc/intensity.h; the season table, the cut into words and index_run of seams.h), so that
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
    std::vector<int> w_t0, w_doy;
    std::vector<uint32_t> w_hot;                                            // the hot-day words of k_hot_words
    for (int64_t t = 0; t < T;) {
        const int nb = word_length(doy_map, t, T);
        uint32_t w = 0u;
        for (int j = 0; j < nb; j++)
            if ((double)x[t + j] > thr[doy_map[t] + j]) w |= 1u << j;
        w_t0.push_back((int)t);
        w_doy.push_back(doy_map[t]);
        w_hot.push_back(w);
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
    HotRuns runs{w_t0.data(), 1, K, (int)T};
    for (int k = 0; k <= K && L.open(); k++) {
        runs.word(k, k < K ? w_hot[k] : 0u);
        int s, e;
        while (runs.pop(s, e, kw)) intensity_run(L, s, e, label_run(ist.data(), 1, defs, D, s, e), acc.data(), 1, block, flush);
    }
    while (L.open()) { flush(); L.next(); }
    return 0;
}

}  // extern "C"
