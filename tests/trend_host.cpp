// trend_host.cpp - TEST INFRASTRUCTURE: hdp_b200/csrc/trend.h replayed on the CPU, series by series, with the loops of k_trend
// (trend.cu) run by one thread: compaction, the point walk for S, the tie counts and the middle values, then the 8-pass radix select of
// the four order statistics over recomputed slopes.  tests/test_trend_host.py compares it with tests/trend_oracle.py bit for bit.
// Not part of the product.
//     g++ -O2 -std=c++17 -ffp-contract=off -shared -fPIC -I hdp_b200/csrc tests/trend_host.cpp -o <tmp>/libtrend_host.so
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#include "trend.h"

using namespace hdp;

template <typename T>
static void series(const T *x, int Y, int64_t C, int missing, double zq, double out[kTrendPlanes])
{
    std::vector<double> ys;
    std::vector<int> xs;
    for (int y = 0; y < Y; y++) {
        const T v = x[(int64_t)y * C];
        const bool ok = sizeof(T) == 2 ? (int)v != missing : (bool)isfinite((double)v);
        if (ok) { ys.push_back((double)v); xs.push_back(y); }
    }
    const int n = (int)ys.size();
    const int64_t ylo = trend_mid_lo(n), yhi = n / 2;
    int64_t S = 0, tie_sum = 0;
    double mid[2] = {0.0, 0.0};
    for (int i = 0; i < n; i++) {
        TrendPoint p;
        const uint64_t ki = trend_key(ys[i]);
        for (int k = 0; k < n; k++) trend_point(p, ys[i], ki, ys[k], k > i);
        S += p.S;
        tie_sum += trend_tie_term(p.ties);
        if (p.below <= ylo && ylo < p.below + p.same) mid[0] = ys[i];
        if (p.below <= yhi && yhi < p.below + p.same) mid[1] = ys[i];
    }
    const double var = trend_mk_var(n, tie_sum);
    const int64_t N = (int64_t)n * (n - 1) / 2;
    double a[kTrendTargets] = {0.0, 0.0, 0.0, 0.0};
    if (N > 0) {
        int64_t r[kTrendTargets];
        trend_ranks(N, var, zq, r);
        TrendSelect sel;
        sel.start(r);
        std::vector<uint32_t> hist(kTrendTargets * kTrendBins);
        for (int shift = 56; shift >= 0; shift -= 8) {
            sel.groups();
            memset(hist.data(), 0, hist.size() * 4);
            for (int i = 0, j = 1; i < n - 1; trend_pair_advance(i, j, 1, n)) {
                const int b = sel.bin(trend_key(trend_slope(ys[i], ys[j], xs[i], xs[j])), shift);
                if (b >= 0) hist[b]++;
            }
            for (int t = 0; t < kTrendTargets; t++) {
                int64_t before = 0;
                const int d = trend_digit(hist.data() + sel.gid[t] * kTrendBins, kTrendBins, sel.rank[t], before);
                sel.take(t, d, before, shift);
            }
        }
        for (int t = 0; t < kTrendTargets; t++) a[t] = trend_unkey(sel.pre[t]);
    }
    const double xmed = n > 0 ? trend_mid(n, (double)xs[ylo], (double)xs[yhi]) : 0.0;
    const double ymed = n > 0 ? trend_mid(n, mid[0], mid[1]) : 0.0;
    trend_finish(n, S, var, ymed, xmed, a, out);
}

extern "C" {

// x [rows, Y, C] of uint16 (dtype 1) or float32 (dtype 2) -> out f64 [8, rows, C], as hdp_b200_trend
int trend_host(const void *x, int dtype, int64_t rows, int Y, int64_t C, int64_t missing, double zq, double *out)
{
    if (Y > kTrendMaxY) return -2;
    double o[kTrendPlanes];
    for (int64_t r = 0; r < rows; r++)
        for (int64_t c = 0; c < C; c++) {
            if (dtype == 1) series((const uint16_t *)x + r * Y * C + c, Y, C, (int)missing, zq, o);
            else series((const float *)x + r * Y * C + c, Y, C, -1, zq, o);
            for (int q = 0; q < kTrendPlanes; q++) out[q * rows * C + r * C + c] = o[q];
        }
    return 0;
}

}  // extern "C"
