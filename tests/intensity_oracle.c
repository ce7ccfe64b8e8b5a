/*
 * intensity_oracle.c - TEST INFRASTRUCTURE: CPU restatement of the heatwave intensity metrics (HWC, HWI, HWP; contract in
 * include/hdp_b200.h, hdp_b200_intensity), the checker of the intensity tests.  It is built on the oracle's own hot-day and
 * index_heatwaves code (oracle/hdp_oracle.c, included unchanged) and sums in the contract's canonical order.  Not part of the
 * product: tests/intensity_oracle.py compiles it into a temporary directory.
 *     gcc -O2 -fPIC -shared -ffp-contract=off [-fopenmp] -I oracle tests/intensity_oracle.c -o <tmp>/libintensity_oracle.so -lm
 */
#include "hdp_oracle.c"

/* Heatwave intensity (no reference counterpart; contract in include/hdp_b200.h, hdp_b200_intensity) for one cell, one
 * percentile, one definition: e_t = (double)measure[t] - threshold[doy_map[t]] over the days of each season slice whose
 * heatwave id (index_heatwaves of the hot-day mask) is > 0.  out is float32 [3 * Y]: HWC (per maximal block of consecutive such
 * days r = 0, r = r + e_t in time order, then S = S + r), HWI (S / HWF), HWP (max e_t); 0 without heatwave days. */
HDP_API int hdp_oracle_heatwave_intensity(const float *measure, const double *threshold, const int64_t *doy_map,
                                          int64_t T, int64_t min_duration, int64_t max_break, int64_t max_subs,
                                          const int64_t *season_ranges, int64_t Y, float *out)
{
    uint8_t *hot = (uint8_t *)malloc((size_t)(T > 0 ? T : 1));
    int64_t *hw = (int64_t *)malloc(sizeof(int64_t) * (size_t)(T > 0 ? T : 1));
    int rc = -1;
    int64_t y, t, lo, hi;
    if (hot && hw) {
        hdp_oracle_indicate_hot_days(measure, threshold, doy_map, T, hot);
        rc = hdp_oracle_index_heatwaves(hot, T, min_duration, max_break, max_subs, hw);
        for (y = 0; rc == 0 && y < Y; y++) {
            double S = 0.0, r = 0.0, peak = 0.0;
            int64_t days = 0;
            py_slice(season_ranges[2 * y], season_ranges[2 * y + 1], T, &lo, &hi);
            for (t = lo; t < hi; t++) {
                double e;
                if (hw[t] <= 0) continue;
                if (t == lo || hw[t - 1] <= 0) r = 0.0;                 /* a block starts */
                e = (double)measure[t] - threshold[doy_map[t]];
                r = r + e;
                if (e > peak) peak = e;
                days++;
                if (t + 1 == hi || hw[t + 1] <= 0) S = S + r;          /* the block ends */
            }
            out[y] = (float)S;
            out[Y + y] = days > 0 ? (float)(S / (double)days) : 0.0f;
            out[2 * Y + y] = (float)peak;
        }
    }
    free(hot); free(hw);
    return rc;
}

/* Batch driver of hdp_oracle_heatwave_intensity in the layout of hdp_oracle_metrics_batch: out float32 [P, D, C, 3, Y]. */
HDP_API int hdp_oracle_intensity_batch(const float *measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                       const double *thresholds, int64_t n_doy, int P,
                                       const int64_t *doy_map, const int64_t *defs, int D,
                                       const int64_t *seasons_north, const int64_t *seasons_south, int64_t Y,
                                       const uint8_t *is_south, float *out, int threads)
{
    int64_t c;
    int failed = 0;
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel
#endif
    {
        float *series = (float *)malloc(sizeof(float) * (size_t)(T > 0 ? T : 1));
        double *thr = (double *)malloc(sizeof(double) * (size_t)(n_doy > 0 ? n_doy : 1));
        if (!series || !thr) {
            failed = 1;
        } else {
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 4)
#endif
            for (c = 0; c < C; c++) {
                int64_t t, d;
                int p, k;
                const int64_t *seasons = is_south[c] ? seasons_south : seasons_north;
                for (t = 0; t < T; t++) series[t] = measure[t * ld_t + c * ld_c];
                for (p = 0; p < P; p++) {
                    for (d = 0; d < n_doy; d++) thr[d] = thresholds[(c * n_doy + d) * P + p];
                    for (k = 0; k < D; k++) {
                        float *o = out + ((((int64_t)p * D + k) * C + c) * 3) * Y;
                        if (hdp_oracle_heatwave_intensity(series, thr, doy_map, T, defs[3 * k], defs[3 * k + 1],
                                                          defs[3 * k + 2], seasons, Y, o) != 0)
                            failed = 1;
                    }
                }
            }
        }
        free(series);
        free(thr);
    }
    return failed ? -1 : 0;
}
