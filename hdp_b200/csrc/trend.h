// trend.h - the per-series rules of the trend statistics (hdp_b200_trend): Theil-Sen slope with its Sen (1968) confidence interval
// and the Mann-Kendall test, as plain functions that compile for the device (trend.cu, one warp per series) and for the host
// (tests/trend_host.cpp replays the warp's loops on the CPU against the NumPy oracle, tests/trend_oracle.py).
//
// Contract (one series y[0 .. Y-1], x = season index):
//   valid       u16: y != missing (no sentinel when missing < 0); f32: y finite.  n valid seasons, values widened to f64
//   slopes      s_ij = (y_j - y_i) / (double)(j - i) over the N = n(n-1)/2 pairs i < j of valid seasons
//   median      of a sorted ascending: a[N/2] for odd N, (a[N/2-1] + a[N/2]) * 0.5 for even N
//   slope       median of the slopes; intercept = median(y_valid) - slope * median(x_valid)
//   MK S        sum of sign(y_j - y_i) over the pairs;  var = (n(n-1)(2n+5) - sum_i (t_i - 1)(2 t_i + 5)) / 18, t_i = #{k: y_k == y_i}
//   p           z = (S - sgn S) / sqrt(var) (0 when var = 0), p = erfc(|z| / sqrt(2))
//   CI          sigma = sqrt(max(var, 0)), Ru = min(rint((N - zq sigma) / 2), N - 1), Rl = max(rint((N + zq sigma) / 2) - 1, 0):
//               slope_low = a[Rl], slope_high = a[Ru]
//   n < 2       slope, intercept, slope_low, slope_high, p NaN; S = var = 0
// "Sorted ascending" is the order of trend_key below: -0.0 sorts before +0.0, which fixes the bits of every order statistic.
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#include "seams.h"

#ifdef __CUDA_ARCH__
#define HDP_TREND_UNROLL _Pragma("unroll")
#else
#define HDP_TREND_UNROLL
#endif

namespace hdp {

constexpr int kTrendMaxY = 512;        // longest series: more seasons return HDP_B200_ERR_UNSUPPORTED
constexpr int kTrendPlanes = 8;        // slope, intercept, slope_low, slope_high, mk_s, mk_var, mk_p, n
constexpr int kTrendTargets = 4;       // order statistics selected per series: the two median ranks, Rl, Ru
constexpr int kTrendBins = 256;        // radix digit: 8 bits, 8 passes over the 64-bit key

HDP_HD uint64_t trend_bits(double v)
{
#ifdef __CUDA_ARCH__
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t u;
    memcpy(&u, &v, 8);
    return u;
#endif
}

HDP_HD double trend_double(uint64_t u)
{
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)u);
#else
    double v;
    memcpy(&v, &u, 8);
    return v;
#endif
}

// Order-preserving 64-bit key of a non-NaN double: key(a) < key(b) <=> a < b, and -0.0 before +0.0.
HDP_HD uint64_t trend_key(double v)
{
    const uint64_t u = trend_bits(v);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

HDP_HD double trend_unkey(uint64_t k) { return trend_double((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k); }

// s_ij: one f64 subtraction, one correctly rounded f64 division
HDP_HD double trend_slope(double yi, double yj, int xi, int xj) { return (yj - yi) / (double)(xj - xi); }

// The pairs (i, j), i < j < n, in row-major order of the upper triangle.  Moves (i, j) `step` pairs on; i >= n - 1 once past the end.
// A lane starts at (0, 1) moved on by its lane index and then steps by the warp width.
HDP_HD void trend_pair_advance(int &i, int &j, int step, int n)
{
    j += step;
    while (j >= n && i < n - 1) {
        i++;
        j -= n - i - 1;
    }
}

// The median ranks and the confidence-interval ranks of N >= 1 slopes, for MK variance var and zq = Phi^-1(alpha / 2) < 0.
HDP_HD void trend_ranks(int64_t N, double var, double zq, int64_t r[kTrendTargets])
{
    r[0] = N % 2 ? N / 2 : N / 2 - 1;
    r[1] = N / 2;
    const double sigma = sqrt(var > 0.0 ? var : 0.0), zs = zq * sigma, dN = (double)N;
    const double u = rint((dN - zs) * 0.5), l = rint((dN + zs) * 0.5) - 1.0;
    r[3] = u < (double)(N - 1) ? (int64_t)u : N - 1;
    r[2] = l > 0.0 ? (int64_t)l : 0;
}

// the median of m sorted values from its two middle ones a[(m-1)/2] (lo) and a[m/2] (hi); lo == hi for odd m
HDP_HD double trend_mid(int64_t m, double lo, double hi) { return m % 2 ? hi : (lo + hi) * 0.5; }

// the two middle ranks of m values (equal for odd m)
HDP_HD int64_t trend_mid_lo(int64_t m) { return (m - 1) / 2; }

// one valid value y_k against y_i in the walk over k for a fixed i (S, the tie count t_i and the rank of y_i among the values)
struct TrendPoint {
    int64_t S = 0;       // sum over k > i of sign(y_k - y_i)
    int64_t ties = 0;    // t_i: #{k: y_k == y_i}, i included
    int64_t below = 0;   // #{k: key(y_k) < key(y_i)}
    int64_t same = 0;    // #{k: key(y_k) == key(y_i)}, i included
};

HDP_HD void trend_point(TrendPoint &p, double yi, uint64_t ki, double yk, bool later)
{
    const double d = yk - yi;
    if (later) p.S += (d > 0.0) - (d < 0.0);
    p.ties += yk == yi;
    const uint64_t kk = trend_key(yk);
    p.below += kk < ki;
    p.same += kk == ki;
}

// (t - 1)(2t + 5): one valid value's share of the tie correction of the MK variance
HDP_HD int64_t trend_tie_term(int64_t t) { return (t - 1) * (2 * t + 5); }

// MK variance: the numerator is exact in int64, then converted and divided by 18 once
HDP_HD double trend_mk_var(int64_t n, int64_t tie_sum) { return (double)(n * (n - 1) * (2 * n + 5) - tie_sum) / 18.0; }

HDP_HD double trend_mk_p(int64_t S, double var)
{
    const double z = var > 0.0 ? (double)(S - ((S > 0) - (S < 0))) / sqrt(var) : 0.0;
    return erfc(fabs(z) * 0.70710678118654752440);
}

// The radix selection of the four order statistics: per target its key prefix so far and its rank within the keys that share that
// prefix.  Targets with equal prefixes share one histogram (group) in a pass; a key belongs to at most one group.
struct TrendSelect {
    uint64_t pre[kTrendTargets];
    int64_t rank[kTrendTargets];
    uint64_t gpre[kTrendTargets];     // the prefix of each group of this pass
    int gid[kTrendTargets];           // the group of each target
    int ng;                           // number of groups

    HDP_HD void start(const int64_t r[kTrendTargets])
    {
        HDP_TREND_UNROLL
        for (int t = 0; t < kTrendTargets; t++) { pre[t] = 0; rank[t] = r[t]; }
    }
    // the groups of the pass over digit (key >> shift) & 255
    HDP_HD void groups()
    {
        ng = 0;
        HDP_TREND_UNROLL
        for (int t = 0; t < kTrendTargets; t++) {
            int g = ng;
            HDP_TREND_UNROLL
            for (int u = 0; u < kTrendTargets; u++)
                if (u < ng && gpre[u] == pre[t]) g = u;
            gid[t] = g;
            HDP_TREND_UNROLL
            for (int u = 0; u < kTrendTargets; u++)       // gpre[ng] = pre[t] with a static index: no local memory
                if (g == ng && u == ng) gpre[u] = pre[t];
            ng += g == ng;
        }
    }
    // histogram bin (group * 256 + digit) of a key in the pass over `shift`, -1 when its prefix is no group's
    HDP_HD int bin(uint64_t key, int shift) const
    {
        const uint64_t hi = shift >= 56 ? 0ull : ~0ull << (shift + 8);
        int b = -1;
        HDP_TREND_UNROLL
        for (int g = 0; g < kTrendTargets; g++)
            if (g < ng && b < 0 && ((key ^ gpre[g]) & hi) == 0ull) b = g * kTrendBins + (int)((key >> shift) & 0xffu);
        return b;
    }
    // target t's rank falls on digit d, after `before` keys of its group's smaller digits
    HDP_HD void take(int t, int d, int64_t before, int shift)
    {
        pre[t] |= (uint64_t)d << shift;
        rank[t] -= before;
    }
};

// The bin of rank r among the counts h[0 .. bins-1] (r < their sum), and the count of the bins below it.  The replay scans a whole
// 256-bin histogram with it; in trend.cu each lane scans its 8 bins after a warp scan has found the lane.
HDP_HD int trend_digit(const uint32_t *h, int bins, int64_t r, int64_t &before)
{
    int64_t acc = 0;
    for (int d = 0; d < bins; d++) {
        if (r < acc + h[d]) { before = acc; return d; }
        acc += h[d];
    }
    before = acc;
    return bins - 1;
}

// The eight outputs of one series.  n valid seasons; S and tie_sum from the point walk; ymed, xmed the medians of the valid values
// and of their season indices; a[4] the selected slopes (ranks of trend_ranks, needs var: see trend_ranks' caller).
HDP_HD void trend_finish(int64_t n, int64_t S, double var, double ymed, double xmed, const double a[kTrendTargets], double out[kTrendPlanes])
{
    const int64_t N = n * (n - 1) / 2;
    const double nan = trend_double(0x7ff8000000000000ull);
    const double slope = N > 0 ? trend_mid(N, a[0], a[1]) : nan;
    out[0] = slope;
    out[1] = N > 0 ? ymed - slope * xmed : nan;
    out[2] = N > 0 ? a[2] : nan;
    out[3] = N > 0 ? a[3] : nan;
    out[4] = (double)S;
    out[5] = var;
    out[6] = N > 0 ? trend_mk_p(S, var) : nan;
    out[7] = (double)n;
}

}  // namespace hdp
