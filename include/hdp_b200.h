/*
 * hdp_b200.h - C ABI of libhdp_b200.so: the two HDP hot paths on B200 (sm_100a).
 *
 * HDP (AgentOxygen/HDP v1.0.2) is pure Python + Numba and has no FFI of its own; the seams this
 * library replaces are the two array-level kernels directly under its public functions, plus the
 * per-block sweeps around them.  "reference" file:line below are relative to the HDP source tree.
 *
 *   hdp_b200_thresholds   replaces  compute_percentiles gufunc            hdp/threshold.py:52-78
 *                                   + compute_percentiles_wrapper          hdp/threshold.py:81-93
 *                                   (np.quantile as compiled by Numba:     numba/np/arraymath.py:1655-1704, 1754-1768)
 *   hdp_b200_metrics      replaces  compute_heatwave_metrics              hdp/metric.py:304-341
 *                                   (indicate_hot_days :280-301, index_heatwaves :11-60,
 *                                    heatwave_frequency/number/duration/average :63-172)
 *                                   + compute_heatwave_metrics_wrapper     hdp/metric.py:344-369
 *   hdp_b200_hot_days     replaces  indicate_hot_days                     hdp/metric.py:280-301
 *   hdp_b200_intensity    (no reference counterpart) heatwave intensity: cumulative, mean and peak exceedance of the
 *                         threshold over the heatwave days of every season, optionally with the metrics in the same pass
 *   hdp_b200_index_heatwaves   replaces  index_heatwaves                  hdp/metric.py:11-60     (the building blocks under
 *   hdp_b200_season_metrics    replaces  heatwave_frequency / number / duration / average  hdp/metric.py:63-172   their own names)
 *   hdp_b200_extent       (no reference counterpart) heatwave spatial extent: the weighted number of cells of each region on a
 *                         heatwave day, for every day
 *   hdp_b200_trend        (no reference counterpart) Theil-Sen slope, its confidence interval and the Mann-Kendall test of every
 *                         season series of a metric or intensity output
 *   *_host variants       the same calls with HOST buffers (cell chunks pipelined H2D -> kernels -> D2H on three streams).
 *
 * Conventions
 *   - Pointers named d_*  are DEVICE pointers owned by the caller (e.g. torch tensors).
 *   - Pointers named h_*  are HOST pointers to small index tables (KBs); they are copied inside the call
 *     and may be freed as soon as the call returns.
 *   - Every device call takes a cudaStream_t (as void*), enqueues its work on it and returns without
 *     synchronising the device (small pageable-host table uploads are the only host-blocking step).
 *   - No allocation inside the device calls: scratch comes from the caller-sized workspace
 *     (hdp_b200_*_workspace_bytes).  The *_host variants own their device buffers
 *     (kept between calls, see hdp_b200_host_release).
 *   - Return value: 0 = ok; > 0 = a cudaError_t; < 0 = one of the HDP_B200_ERR_* codes.  Nothing throws.
 *   - Element (t, c) of a measure array lives at base[t*ld_t + c*ld_c] (strides in ELEMENTS).
 *     The fast path is time-major, cell-contiguous (ld_c == 1); any other layout is first
 *     normalised into the workspace by a transposing copy.
 *   - Thread-compatible: concurrent calls must use different workspaces.
 */
#ifndef HDP_B200_H
#define HDP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HDP_B200_ABI_VERSION 6

#define HDP_B200_OK                 0
#define HDP_B200_ERR_INVALID       (-1)  /* null pointer, negative size, quantile outside [0,1] or NaN, bad table entry */
#define HDP_B200_ERR_UNSUPPORTED   (-2)  /* shape outside what the kernels support (see hdp_b200_strerror) */
#define HDP_B200_ERR_WORKSPACE     (-3)  /* workspace pointer null or smaller than *_workspace_bytes() */
#define HDP_B200_ERR_NO_DEVICE     (-4)  /* no CUDA device / not an sm_100 device */
#define HDP_B200_ERR_NOMEM         (-5)  /* host-side allocation failed */

#define HDP_B200_MAX_PERCENTILES   32
#define HDP_B200_MAX_DEFINITIONS   32
#define HDP_B200_MAX_WINDOW        32768 /* samples pooled per day-of-year window (W * n_y) */
#define HDP_B200_MAX_REGIONS       256   /* regions of hdp_b200_extent */

int         hdp_b200_abi_version(void);
const char *hdp_b200_strerror(int code);
/* SM count and compute capability of the current device; HDP_B200_ERR_NO_DEVICE if there is none. */
int         hdp_b200_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* ---------------------------------------------------------------------------------------------------
 * Path 1 - thresholds.   reference: hdp/threshold.py:52-93
 *
 *   d_temps       f32 baseline series, element (t, c) at [t*ld_t + c*ld_c], t < T_b, c < C
 *   h_time_index  i32 [n_doy, n_y]  time indices of each day-of-year row, -1 padded (threshold.py:28-39);
 *                 negative entries index from the end of the series like the reference's gufunc does
 *   h_win_rows    i32 [n_doy, W]    rows of time_index pooled by the window of each row (threshold.py:41-48);
 *                 window_samples[d] == time_index[win_rows[d]].ravel() is the reference's table
 *   h_q           f64 [P]           quantiles in [0, 1]
 *   d_out         f64 [C, n_doy, P] (the reference's (<cells>, doy, percentile) order)
 *   input_unit    unit of the samples, converted to Celsius AS THEY ARE LOADED with the reference's float32 arithmetic
 *                 (hdp/measure.py:10-41): 0 = Celsius (no conversion), 1 = Kelvin (x - 273.15), 2 = Fahrenheit ((x - 32) / 1.8).
 *                 Raw model output then needs no converted copy: format_standard_measures' unit step is fused into the load
 *                 stage of the kernels on the hot path (k_thr_net, k_hot_words; other threshold kernels convert a copy first).
 * ------------------------------------------------------------------------------------------------- */
#define HDP_B200_UNIT_CELSIUS    0
#define HDP_B200_UNIT_KELVIN     1
#define HDP_B200_UNIT_FAHRENHEIT 2

size_t hdp_b200_thresholds_workspace_bytes(int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                                           int n_doy, int n_y, int W, int P, int input_unit);

int hdp_b200_thresholds(const float *d_temps, int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                        const int32_t *h_time_index, const int32_t *h_win_rows, int n_doy, int n_y, int W,
                        const double *h_q, int P,
                        double *d_out,
                        void *d_workspace, size_t workspace_bytes, void *stream, int input_unit);

/* Test hook: which kernel hdp_b200_thresholds uses.  0 = default (k_thr_net, the lane-per-cell network kernel, where the
 * tables and quantiles allow - high quantiles, windows of consecutive rows, at most 32 samples per row - with k_thr_seg
 * behind it for cells with NaN / inf samples; else k_thr_seg with its candidate filter - for high quantiles in its light
 * variant k_thr_cand, with k_thr_seg behind it for the warps that one hands over - else k_thr_ranked, else
 * k_thr_generic); 1 = k_thr_generic for everything (gather + sort: any table, rows pooled any number of times);
 * 2 = k_thr_ranked instead of the segment kernels; 3 = k_thr_seg without the candidate filter; 4 = k_thr_seg with the
 * candidate filter but without k_thr_cand; 5 = the default without k_thr_net; 6 = the default with k_thr_net keeping every
 * list in shared memory (no tensor-memory variant k_thr_net_tm). */
void hdp_b200_thresholds_force_generic(int on);

/* Which kernel hdp_b200_thresholds would run for these tables and quantiles (host logic only: no device needed).
 * info[0] = 0 k_thr_generic, 1 k_thr_ranked, 2 k_thr_seg, 3 k_thr_cand + k_thr_seg, 4 k_thr_net; for k_thr_net info[1..7] =
 * {samples per row (padded), list length K, blocks per window, rows per block, irregular days, warps per CTA of the
 * tensor-memory variant (0 = shared memory only), suffix lists kept in tensor memory}; for the segment kernels info[4] = days
 * per segment. */
int hdp_b200_thresholds_kernel_choice(const int32_t *h_time_index, const int32_t *h_win_rows, int64_t T_b, int n_doy, int n_y, int W,
                                      const double *h_q, int P, int *info);

/* Host-buffer variant (chunked H2D / kernels / D2H pipeline, see csrc/host.cu).  d_keep: optional DEVICE buffer
 * f64 [C, n_doy, P]; when given, the thresholds are also left there, so that the metric pass that follows
 * (hdp_b200_metrics_host with d_thr = d_keep) does not upload them again - in the reference workflow
 * compute_thresholds -> compute_group_metrics the thresholds then cross PCIe once (to the caller), not three times. */
int hdp_b200_thresholds_host(const float *h_temps, int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                             const int32_t *h_time_index, const int32_t *h_win_rows, int n_doy, int n_y, int W,
                             const double *h_q, int P,
                             double *h_out, double *d_keep, int input_unit);

/* ---------------------------------------------------------------------------------------------------
 * Path 2 - heatwave metrics.   reference: hdp/metric.py:11-172, 280-369
 *
 *   d_measure     f32 series, element (t, c) at [t*ld_t + c*ld_c], t < T, c < C
 *   d_thr         f64 [C, n_doy, P]   thresholds, exactly what path 1 writes
 *   h_doy_map     i32 [T]             day-of-year row of every time step (metric.py:265-277), 0 <= v < n_doy
 *                                     (HDP_B200_ERR_INVALID for any other entry, before anything is written)
 *   h_defs        i32 [D, 3]          [min_duration, max_break, max_subs] per definition (metric.py:11)
 *   h_season_north / h_season_south   i32 [Y, 2] season [start, end) time indices per hemisphere
 *                 (metric.py:175-262); Python slice semantics are applied to negative / out-of-range values
 *   d_is_south    u8 [C] 1 = use the southern table (lat < 0, metric.py:247-252); NULL = all northern
 *   d_out         u16 [4, P, D, Y, C]  metric-major: HWF, HWN, HWD, HWA (= HWF / HWN truncated, metric.py:336-340);
 *                 the reference's int64 (percentile, definition, <cells>, metric, year) array is
 *                 out[m][p][d][y][c] widened.  Every value is <= the longest season, which must be < 65536.
 *   input_unit    as for hdp_b200_thresholds, optionally OR-ed with HDP_B200_COLD (here and in hdp_b200_metrics_host,
 *                 hdp_b200_intensity and hdp_b200_intensity_host) and with HDP_B200_ONSET (below: d_out gets 6 planes).
 *
 * Cold spells (HDP_B200_COLD): a day counts when (double)x(t) < thr[c, doy_map[t], p] instead of x(t) > thr (NaN on either side:
 * never; a -inf sample is cold unless thr is -inf), and the planes are CSF, CSN, CSD, CSA: exactly the rules of HWF, HWN, HWD,
 * HWA applied to the cold days, in the same layout.  The cold result equals the heatwave result for -x and -thr bit for bit.
 * The season tables are used as given: the cold season of a hemisphere is usually the other hemisphere's warm season.
 * Libraries of ABI version 6 without cold spells reject the flag with HDP_B200_ERR_INVALID.  The threshold entry points take
 * no direction and reject it too.
 * ------------------------------------------------------------------------------------------------- */
#define HDP_B200_COLD 0x100

/* Heatwave onset and end (HDP_B200_ONSET, OR-ed into input_unit of hdp_b200_metrics, hdp_b200_intensity, hdp_b200_compound and
 * their _host variants, with or without HDP_B200_COLD): the u16 output (d_out / h_out) is then [6, P, D, Y, C], planes 0 - 3
 * exactly the result without the flag and
 *   plane 4  HWO  min(H) - lo: the day of the season (0 = its first day) of its first heatwave day
 *   plane 5  HWE  max(H) - lo: the day of the season of its last heatwave day
 * where [lo, hi) is the season slice after the slice semantics above and H the days t in [lo, hi) whose heatwave id is > 0 (the
 * days HWF counts).  Both are 0xFFFF where H is empty (HWF = 0, also for an empty season); a value is < hi - lo <= 65 535, so the
 * sentinel is never a day.  HWO = 0xFFFF <=> HWE = 0xFFFF <=> HWF = 0; otherwise HWO <= HWE and HWE - HWO + 1 >= HWF >= HWD.  A
 * heatwave that began before the season gives HWO = 0, one that continues past its end HWE = hi - lo - 1 (the clipping of HWF).
 * With HDP_B200_COLD: CSO, CSE over the cold-spell days; compound: over the compound days.  Without a u16 output (the intensity
 * and compound calls) the flag returns HDP_B200_ERR_INVALID; workspace sizes do not depend on it.  Libraries of ABI version 6
 * without onset reject the flag with HDP_B200_ERR_INVALID, and so do the threshold and hot-day entry points.
 * ------------------------------------------------------------------------------------------------- */
#define HDP_B200_ONSET 0x200

/* h_doy_map may be NULL: the size is then an upper bound for regular daily calendars (gap-free daily series); a series with missing
 * days or a seasonal subset cuts into more hot-day words and then gets HDP_B200_ERR_WORKSPACE from that size. */
size_t hdp_b200_metrics_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                        int n_doy, int P, int D, int Y, const int32_t *h_doy_map);

int hdp_b200_metrics(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                     const double *d_thr, int n_doy, int P,
                     const int32_t *h_doy_map,
                     const int32_t *h_defs, int D,
                     const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                     const uint8_t *d_is_south,
                     uint16_t *d_out,
                     void *d_workspace, size_t workspace_bytes, void *stream, int input_unit /* as for hdp_b200_thresholds */);

/* Test hook: 0 makes k_scan feed every hot run to the definitions' state machines instead of first dropping the runs
 * that cannot change any result (short runs after long breaks, see metric.cu); the outputs must be identical. */
void hdp_b200_metrics_run_filter(int on);

/* Which k_scan instantiation hdp_b200_metrics would launch for these definitions and season tables over T days (host logic
 * only: no device needed; the run filter setting above is taken into account).  info[0..6] = {accumulator lane bits: 8 (four
 * definitions per register) or 16 (two), accumulator registers NG, bit planes of the max_subs counters KS, run filter on,
 * compile-time filter constants LMIN and BMAX (0, 0 = the generic instantiation), launches (season passes)}.  Returns what
 * hdp_b200_metrics would return for the definitions and tables (e.g. HDP_B200_ERR_UNSUPPORTED for a season over 65 535 days). */
int hdp_b200_metrics_kernel_choice(const int32_t *h_defs, int D, const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                                   int64_t T, int *info);

/* Host-buffer variant.  Thresholds come from h_thr (host, uploaded chunk by chunk) unless d_thr (DEVICE f64
 * [C, n_doy, P], e.g. the d_keep of hdp_b200_thresholds_host) is given, in which case h_thr may be NULL. */
int hdp_b200_metrics_host(const float *h_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                          const double *h_thr, const double *d_thr, int n_doy, int P,
                          const int32_t *h_doy_map,
                          const int32_t *h_defs, int D,
                          const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                          const uint8_t *h_is_south,
                          uint16_t *h_out, int input_unit);

/* ---------------------------------------------------------------------------------------------------
 * Path 2 - heatwave intensity (opt-in; hdp_b200_metrics is unchanged).  Same inputs as hdp_b200_metrics.  For cell c,
 * percentile p, definition d and season y, with e_t = (double)x_c(t) - thr[c, doy_map[t], p] (x after the input_unit
 * conversion) over the days t of the season slice whose heatwave id is > 0 (exactly the days HWF counts, so e_t > 0):
 *
 *   HWC  cumulative intensity: per maximal block of consecutive such days, in time order, r = 0, r = r + e_t, then S = S + r
 *   HWI  mean intensity S / HWF (0 when HWF = 0)
 *   HWP  peak intensity: the largest e_t (0 when there is no heatwave day)
 *
 *   d_int         f32 [3, P, D, Y, C]  planes HWC, HWI, HWP, each rounded once from float64 (the canonical order above makes
 *                 the result reproducible bit for bit)
 *   d_out         optional u16 [4, P, D, Y, C] ([6, ...] with HDP_B200_ONSET, which needs it): when given, also exactly what
 *                 hdp_b200_metrics writes, from the same hot-day pass over the samples
 * The non-empty seasons of each hemisphere's table must be pairwise disjoint after slice clamping (every table built by
 * compute_hemisphere_ranges / get_range_indices is); other tables return HDP_B200_ERR_UNSUPPORTED.
 *
 * With HDP_B200_COLD in input_unit: CSC, CSI, CSP over the cold-spell days (see Path 2 above), with the deficit
 * e_t = thr[c, doy_map[t], p] - (double)x_c(t) > 0 in place of the exceedance, in the same order and layout (a -inf sample
 * gives inf); d_out then receives CSF, CSN, CSD, CSA.
 * ------------------------------------------------------------------------------------------------- */
/* h_doy_map may be NULL: the size is then an upper bound for regular daily calendars. */
size_t hdp_b200_intensity_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                          int n_doy, int P, int D, int Y, const int32_t *h_doy_map);

int hdp_b200_intensity(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                       const double *d_thr, int n_doy, int P,
                       const int32_t *h_doy_map,
                       const int32_t *h_defs, int D,
                       const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                       const uint8_t *d_is_south,
                       float *d_int, uint16_t *d_out,
                       void *d_workspace, size_t workspace_bytes, void *stream, int input_unit);

/* Host-buffer variant (the pipeline of hdp_b200_metrics_host: each measure chunk crosses PCIe once for both outputs).
 * h_out may be NULL; thresholds from h_thr unless d_thr (DEVICE) is given. */
int hdp_b200_intensity_host(const float *h_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                            const double *h_thr, const double *d_thr, int n_doy, int P,
                            const int32_t *h_doy_map,
                            const int32_t *h_defs, int D,
                            const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                            const uint8_t *h_is_south,
                            float *h_int, uint16_t *h_out, int input_unit);

/* ---------------------------------------------------------------------------------------------------
 * Path 2 - compound heatwaves (opt-in): the sweep over the days on which TWO measures of one grid, e.g. tmax and tmin (hot days
 * and hot nights), both exceed their own thresholds.  Measure A (d_a) and measure B (d_b) share C, T, doy_map, the season
 * tables and input_unit (which applies to both); each has its own strides and its own thresholds, f64 [C, n_doy, P] with the
 * same n_doy and P: percentile p of A is paired with percentile p of B.
 *
 *   compound hot day   (double)x_a(t) > thr_a[c, doy_map[t], p]  and  (double)x_b(t) > thr_b[c, doy_map[t], p]  (NaN on either
 *                      side of either comparison: not hot).  With HDP_B200_COLD both comparisons are < (cold days and cold
 *                      nights); the season tables are used as given.
 *   d_out              optional u16 [4, P, D, Y, C]: HWF, HWN, HWD, HWA (CSF ... CSA with HDP_B200_COLD) by exactly the rules of
 *                      hdp_b200_metrics, applied to the compound days; [6, ...] with HWO, HWE with HDP_B200_ONSET (which needs it)
 *   d_int              optional f32 [2, 3, P, D, Y, C]: block 0 = HWC, HWI, HWP of measure A (its exceedance x_a - thr_a over the
 *                      compound heatwave days), block 1 = the same for measure B; each block has the arithmetic and order of
 *                      hdp_b200_intensity (the deficit with HDP_B200_COLD), and the season tables must be disjoint as there
 * At least one of d_out and d_int must be given.  The result at percentile p equals hdp_b200_metrics / hdp_b200_intensity of
 * where(M_p, x_a, NaN) against thr_a (block 1: where(M_p, x_b, NaN) against thr_b), M_p being the compound mask.
 * ------------------------------------------------------------------------------------------------- */
/* h_doy_map may be NULL: the size is then an upper bound for regular daily calendars.  Serves hdp_b200_compound and
 * hdp_b200_compound_hot_days. */
size_t hdp_b200_compound_workspace_bytes(int64_t C, int64_t T, int64_t ld_c_a, int64_t ld_c_b, int n_doy, int P, int D, int Y,
                                         const int32_t *h_doy_map);

int hdp_b200_compound(const float *d_a, int64_t ld_t_a, int64_t ld_c_a, const float *d_b, int64_t ld_t_b, int64_t ld_c_b,
                      int64_t C, int64_t T, const double *d_thr_a, const double *d_thr_b, int n_doy, int P,
                      const int32_t *h_doy_map,
                      const int32_t *h_defs, int D,
                      const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                      const uint8_t *d_is_south,
                      uint16_t *d_out, float *d_int,
                      void *d_workspace, size_t workspace_bytes, void *stream, int input_unit);

/* Host-buffer variant (the pipeline of hdp_b200_metrics_host; both measures' cells of a chunk cross PCIe once).  Each threshold
 * array comes from the host (h_thr_*) unless its DEVICE copy (d_thr_*) is given. */
int hdp_b200_compound_host(const float *h_a, int64_t ld_t_a, int64_t ld_c_a, const float *h_b, int64_t ld_t_b, int64_t ld_c_b,
                           int64_t C, int64_t T, const double *h_thr_a, const double *d_thr_a, const double *h_thr_b, const double *d_thr_b,
                           int n_doy, int P, const int32_t *h_doy_map,
                           const int32_t *h_defs, int D,
                           const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                           const uint8_t *h_is_south,
                           uint16_t *h_out, float *h_int, int input_unit);

/* Compound mask only (parity checks): d_mask u8 [P, T, C], 1 on the compound hot (with HDP_B200_COLD: cold) days. */
int hdp_b200_compound_hot_days(const float *d_a, int64_t ld_t_a, int64_t ld_c_a, const float *d_b, int64_t ld_t_b, int64_t ld_c_b,
                               int64_t C, int64_t T, const double *d_thr_a, const double *d_thr_b, int n_doy, int P,
                               const int32_t *h_doy_map, uint8_t *d_mask,
                               void *d_workspace, size_t workspace_bytes, void *stream, int input_unit);

/* How the compound hot-day kernel k_hot_pair splits P percentiles (host logic only: no device needed): info[0..2] = {percentiles
 * per group PG, CTAs per (32 cells, day-of-year block) - slices of whole groups, each with both measures' threshold tiles -,
 * shared-memory bytes per CTA}. */
int hdp_b200_compound_plan(int P, int *info);

/* ---------------------------------------------------------------------------------------------------
 * Path 2 - heatwave spatial extent (opt-in): the daily weighted number of cells of each region that are on a heatwave day.  Same
 * inputs as hdp_b200_metrics, plus
 *
 *   d_weight      u32 [C]  integer weight of every cell; NULL = 1 each (the result is then a cell count)
 *   d_region      i32 [C]  region of every cell; NULL = every cell in region 0.  A value outside [0, R) puts the cell in no region:
 *                          it is ignored (defined behaviour, the device input needs no validation)
 *   R             regions, 1 <= R <= HDP_B200_MAX_REGIONS
 *   d_ext         i64 [R, P, D, T]  ACCUMULATED (+=; the caller zeroes it, and a loop over cell ranges adds into one array):
 *                 d_ext[r, p, d, t] += sum of w_c over the cells c of region r for which day t is a day that HWF[p, d, y, c] counts,
 *                 y the season of c's hemisphere table that contains t
 *   d_out         optional u16 [4, P, D, Y, C]: when given, exactly what hdp_b200_metrics writes, from the same pass
 *
 * "A day HWF counts": t lies in the season slice [lo, hi) after the slice semantics above and its heatwave id is > 0.  A day outside
 * every season of a cell's hemisphere adds nothing for that cell, and a heatwave that began before the season counts from lo on.  So
 *   sum_t d_ext[r, p, d, t] = sum_{c in r} w_c * sum_y HWF[p, d, y, c]
 * The sums are exact int64 (u32 weights, C < 2^31), so the result depends neither on order nor on how the cells are split.  The
 * non-empty seasons of each hemisphere's table must be pairwise disjoint after slice clamping (as for hdp_b200_intensity), else
 * HDP_B200_ERR_UNSUPPORTED.  HDP_B200_COLD: the cold-spell days (the result is bit for bit the heatwave result on -x, -thr).
 * HDP_B200_ONSET returns HDP_B200_ERR_INVALID.
 * ------------------------------------------------------------------------------------------------- */
/* h_doy_map may be NULL: the size is then an upper bound for regular daily calendars. */
size_t hdp_b200_extent_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                       int n_doy, int P, int D, int Y, int R, const int32_t *h_doy_map);

int hdp_b200_extent(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                    const double *d_thr, int n_doy, int P,
                    const int32_t *h_doy_map,
                    const int32_t *h_defs, int D,
                    const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                    const uint8_t *d_is_south, const uint32_t *d_weight, const int32_t *d_region, int R,
                    int64_t *d_ext, uint16_t *d_out,
                    void *d_workspace, size_t workspace_bytes, void *stream, int input_unit);

/* Host-buffer variant (the pipeline of hdp_b200_metrics_host; the difference array stays on the device across the cell chunks).
 * h_weight / h_region: HOST arrays as above (NULL allowed).  h_ext i64 [R, P, D, T] is written once at the end: OVERWRITTEN, not
 * accumulated.  h_out (optional) as d_out.  Thresholds from h_thr unless d_thr (DEVICE) is given. */
int hdp_b200_extent_host(const float *h_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                         const double *h_thr, const double *d_thr, int n_doy, int P,
                         const int32_t *h_doy_map,
                         const int32_t *h_defs, int D,
                         const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                         const uint8_t *h_is_south, const uint32_t *h_weight, const int32_t *h_region, int R,
                         int64_t *h_ext, uint16_t *h_out, int input_unit);

/* The *_host variants keep their streams, events and device buffers (grown on demand) in a per-device context between
 * calls; this frees them.  Safe to call at any time no *_host call is running. */
void hdp_b200_host_release(void);

/* Hot-day mask only (parity checks): d_mask u8 [P, T, C], 1 where measure > threshold[doy_map[t]]
 * compared in double precision, NaN -> 0 (metric.py:280-301).  Same workspace size as hdp_b200_metrics. */
int hdp_b200_hot_days(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                      const double *d_thr, int n_doy, int P,
                      const int32_t *h_doy_map,
                      uint8_t *d_mask,
                      void *d_workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * The building blocks of path 2 under the reference's own names.  hdp_b200_metrics never materialises what they exchange
 * (the per-day heatwave id series), but the reference exposes them and its unit tests call them directly
 * (hdp/tests/test_index_heatwaves.py, test_heatwave_{frequency,number,duration,average}.py); these two entry points give
 * the Python mirror (hdp_b200.metric.index_heatwaves, heatwave_*) a device implementation with the reference's semantics
 * for ARBITRARY inputs.  S independent series, each contiguous in time.
 *
 *   hdp_b200_index_heatwaves   d_hot u8 [S, T] (non-zero = hot day, metric.py:28-30), h_defs i32 [D, 3] as for
 *                              hdp_b200_metrics  ->  d_hw i64 [S, D, T] heatwave ids, 0 = no heatwave (metric.py:11-60)
 *   hdp_b200_season_metrics    d_hw i64 [S, T] ANY id series, d_seasons i64 [Y, 2] [start, end) with Python slice
 *                              semantics (DEVICE table: Y is unbounded)  ->  d_hwf, d_hwn, d_hwd i64 [S, Y], d_hwa f64 [S, Y]
 *                              (each may be NULL): days with id > 0 (metric.py:85-102), distinct non-zero ids (:63-82),
 *                              longest / mean number of days per id with the reference's handling of np.unique - the
 *                              smallest distinct value is dropped when there are several (:105-172).  An empty slice
 *                              yields 0 (the reference raises in duration / average: the Python mirror does too).
 * ------------------------------------------------------------------------------------------------- */
int hdp_b200_index_heatwaves(const uint8_t *d_hot, int64_t S, int64_t T, const int32_t *h_defs, int D, int64_t *d_hw, void *stream);
int hdp_b200_season_metrics(const int64_t *d_hw, int64_t S, int64_t T, const int64_t *d_seasons, int Y,
                            int64_t *d_hwf, int64_t *d_hwn, int64_t *d_hwd, double *d_hwa, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * Elementwise pre-pass of hdp.measure on the device ("next" row of the scope table; format_standard_measures itself
 * stays host Python).   reference: hdp/measure.py:10-94, 183-194.  All arrays are dense f32 of n elements; in-place
 * (d_out == d_temp) is allowed.  Results are bit-identical to the reference's Numba / NumPy float32 arithmetic.
 *
 *   hdp_b200_heat_index          out[F] = heat_index(temp[F], rh[%])                      the @nb.vectorize ufunc, measure.py:61-94
 *   hdp_b200_heat_index_measure  out[C] = F->C(heat_index(C->F(temp[C]), rh[%]))          the `{name}_hi` branch, measure.py:183-194;
 *                                rh_is_fraction != 0: rh is g/g and is scaled by 100 first
 *   hdp_b200_to_celsius          unit 0 = copy, 1 = Kelvin (temp - 273.15), 2 = Fahrenheit ((temp - 32) / 1.8), measure.py:10-41
 * ------------------------------------------------------------------------------------------------- */
int hdp_b200_heat_index(const float *d_temp_f, const float *d_rh_pct, int64_t n, float *d_out_f, void *stream);
int hdp_b200_heat_index_measure(const float *d_temp_c, const float *d_rh, int64_t n, int rh_is_fraction, float *d_out_c, void *stream);
int hdp_b200_to_celsius(const float *d_temp, int64_t n, int unit, float *d_out_c, void *stream);

/* Weighted mean over the cells of every row of a u16 [rows, C] array (the metric output is u16 [4 * P * D * Y, C]):
 * d_out[row] = sum_c d_w[c] * x[row, c] / w_sum, float64, fixed summation order.  With d_w = cos(latitude) this is the
 * reduction of the reference's figure deck (hdp/graphics/figure.py:14-15 compute_weighted_spatial_mean). */
int hdp_b200_weighted_mean(const uint16_t *d_x, int64_t rows, int64_t C, const double *d_w, double w_sum, double *d_out, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * Trend statistics of season series: Theil-Sen slope with its Sen (1968) confidence interval, and the Mann-Kendall test.
 *
 *   d_x      [rows, Y, C], cell-contiguous: series (r, c) is d_x[(r * Y + y) * C + c], y = 0 .. Y-1.  The metric output
 *            u16 [M, P, D, Y, C] is this layout with rows = M * P * D, the intensity output f32 [3, P, D, Y, C] likewise.
 *   dtype    HDP_B200_DTYPE_U16 or HDP_B200_DTYPE_F32
 *   missing  u16: the sentinel of a missing season (0xFFFF for the HWO / HWE / CSO / CSE planes), or -1 for none; ignored for f32,
 *            where every non-finite value (NaN, +-inf) is missing
 *   zq       Phi^-1(alpha / 2) < 0, the normal quantile of the two-sided (1 - alpha) confidence interval
 *   d_out    f64 [8, rows, C], planes slope, intercept, slope_low, slope_high, mk_s, mk_var, mk_p, n
 *
 * For one series, x = the season index (0 = first season: slopes are per season), n = the number of valid seasons, and only the
 * pairs i < j of valid seasons are used; values are widened to f64 before any arithmetic.
 *   slopes      s_ij = (y_j - y_i) / (double)(j - i): one f64 subtraction and one correctly rounded f64 division, N = n(n-1)/2 of them
 *   median      sorted ascending (-0.0 before +0.0): a[N/2] for odd N, (a[N/2-1] + a[N/2]) * 0.5 for even N; the same rule for y and x
 *   slope       the median of the slopes
 *   intercept   median(y_valid) - slope * median(x_valid) (Conover's "separate" form, as scipy.stats.theilslopes by default)
 *   mk_s        S = sum of sign(y_j - y_i) over the pairs
 *   mk_var      (n(n-1)(2n+5) - sum_i (t_i - 1)(2 t_i + 5)) / 18, t_i = #{valid k: y_k == y_i}; the numerator exact in int64
 *   mk_p        two-sided, continuity-corrected: z = (S - sgn S) / sqrt(var) when var > 0, else 0; p = erfc(|z| / sqrt(2))
 *   slope_low   a[Rl], Rl = max(rint((N + zq sigma) / 2) - 1, 0)     sigma = sqrt(max(var, 0)), rint rounds half to even
 *   slope_high  a[Ru], Ru = min(rint((N - zq sigma) / 2), N - 1)
 *   n           n
 * With n < 2: slope, intercept, slope_low, slope_high and mk_p are NaN, mk_s = mk_var = 0.  Every plane but mk_p is exact to the
 * bit; mk_p goes through the device's erfc.  Y up to 512; a longer series returns HDP_B200_ERR_UNSUPPORTED.  No workspace.
 * ------------------------------------------------------------------------------------------------- */
#define HDP_B200_DTYPE_U16 1
#define HDP_B200_DTYPE_F32 2

int hdp_b200_trend(const void *d_x, int dtype, int64_t rows, int Y, int64_t C, int64_t missing, double zq, double *d_out, void *stream);

/* Last kernel-launch counters (for bench.py's gpu_launches claim): number of kernels this library has
 * launched since it was loaded. */
int64_t hdp_b200_launch_count(void);

/* Per-kernel timing for bench.py's roofline: while enabled, every kernel launch is bracketed by CUDA events
 * on its own stream.  hdp_b200_timing_read waits for the recorded launches, writes (kernel id, milliseconds)
 * pairs in launch order (at most cap), forgets them and returns how many it wrote. */
#define HDP_B200_KERNEL_NORMALIZE    1
#define HDP_B200_KERNEL_THR_GENERIC  2
#define HDP_B200_KERNEL_HOT_WORDS    3
#define HDP_B200_KERNEL_SCAN         4
#define HDP_B200_KERNEL_UNPACK_MASK  5
#define HDP_B200_KERNEL_THR_SEG      6   /* k_thr_seg */
#define HDP_B200_KERNEL_THR_RANKED   7   /* k_thr_ranked */
#define HDP_B200_KERNEL_MEASURE      8   /* k_measure */
#define HDP_B200_KERNEL_THR_CAND     9   /* k_thr_cand */
#define HDP_B200_KERNEL_THR_NET     10   /* k_thr_net / k_thr_net_tm / k_thr_net_irr */
#define HDP_B200_KERNEL_SEAM        11   /* k_index_heatwaves, k_season_metrics */
#define HDP_B200_KERNEL_INTENSITY   12   /* k_intensity */
#define HDP_B200_KERNEL_HOT_PAIR    13   /* k_hot_pair */
#define HDP_B200_KERNEL_TREND       14   /* k_trend */
#define HDP_B200_KERNEL_EXTENT      15   /* k_extent_prefix (the EXTENT twins of k_scan time as HDP_B200_KERNEL_SCAN) */
void hdp_b200_timing_enable(int on);
int  hdp_b200_timing_read(int *ids, float *ms, int cap);

#ifdef __cplusplus
}
#endif
#endif /* HDP_B200_H */
