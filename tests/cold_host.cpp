// cold_host.cpp - TEST INFRASTRUCTURE: the lane loop of k_intensity (hdp_b200/csrc/intensity.cu) replayed on the CPU in either
// direction, around the very same functions (hdp_b200/csrc/intensity.h: intensity_e, the run popper, the season accounting), so
// that tests/test_cold_host.py can check the cold-spell accounting against the oracle on negated inputs without a GPU.  The
// heatwave-only replay of tests/intensity_host.cpp is left as it is.  Not part of the product.
//     g++ -O2 -shared -fPIC -I hdp_b200/csrc tests/cold_host.cpp -o <tmp>/libcold_host.so
#include <stdint.h>
#include <vector>

#include "intensity.h"

using namespace hdp;

extern "C" {

// One cell, one percentile: x f32 [T] (Celsius), thr f64 [n_doy], doy_map i32 [T], defs i32 [D, 3], seasons i32 [Y, 2]; cold = 0
// heatwaves (x > thr, exceedance), 1 cold spells (x < thr, deficit) -> out f32 [3, D, Y].  Returns 0, or -2 for a season table
// with overlapping non-empty seasons.
int cold_host_cell(const float *x, const double *thr, const int32_t *doy_map, int64_t T, const int32_t *defs, int D,
                   const int32_t *seasons, int Y, int cold, float *out)
{
    std::vector<int32_t> tab((size_t)4 * (Y + 1));
    if (!intensity_season_table(seasons, Y, T, tab.data())) return -2;
    std::vector<int> w_t0, w_doy;
    std::vector<uint32_t> w_bits;                                           // the day words of k_hot_words
    for (int64_t t = 0; t < T;) {
        const int nb = word_length(doy_map, t, T);
        uint32_t w = 0u;
        for (int j = 0; j < nb; j++) {
            const double v = x[t + j], th = thr[doy_map[t] + j];
            if (cold ? v < th : v > th) w |= 1u << j;
        }
        w_t0.push_back((int)t);
        w_doy.push_back(doy_map[t]);
        w_bits.push_back(w);
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
            intensity_day(r, m, intensity_e(x[t], thr[doy], cold != 0));
        }
    };
    HotRuns runs{w_t0.data(), 1, K, (int)T};
    for (int k = 0; k <= K && L.open(); k++) {
        runs.word(k, k < K ? w_bits[k] : 0u);
        int s, e;
        while (runs.pop(s, e, kw)) intensity_run(L, s, e, label_run(ist.data(), 1, defs, D, s, e), acc.data(), 1, block, flush);
    }
    while (L.open()) { flush(); L.next(); }
    return 0;
}

}  // extern "C"
