// metric.cu - path 2: hot-day masks and heatwave metrics for the whole percentile x definition sweep.
//
// Replaces (reference = AgentOxygen/HDP v1.0.2):
//   indicate_hot_days          hdp/metric.py:280-301
//   index_heatwaves            hdp/metric.py:11-60
//   heatwave_frequency/number/duration/average   hdp/metric.py:63-172
//   compute_heatwave_metrics   hdp/metric.py:304-341
//   compute_heatwave_metrics_wrapper (the percentile x definition x cell sweep)   hdp/metric.py:344-369
//
// Two kernels, both HBM-streaming integer/compare work (no tensor cores: nothing here is a contraction):
//
//   k_hot_words  (cells x day-of-year block) tiles.  A CTA owns 32 cells and 32 consecutive days of year,
//                keeps that [32 doy][P][32 cell] threshold tile in shared memory (rounded DOWN to f32, which
//                preserves the reference's double-precision `measure > threshold` exactly) and walks every
//                year of the measure through it, so each threshold is fetched from HBM once and each
//                measure sample once.  Output: one 32-bit word of hot-day bits per (percentile, word, cell).  A cold-spell
//                pass (HDP_B200_COLD) instantiates it with COLD: the tile is rounded UP and the bits mark `measure <
//                threshold`; everything downstream works on the bits and does not know which direction made them.
//   k_scan       one thread per (cell, percentile), lanes = cells (coalesced).  Walks the hot words in
//                time order, pops hot runs with bit tricks and feeds each run to all definitions' state
//                machines held in registers; season accumulators are flushed as u16 when a season closes.
//                The per-day heatwave id array of the reference is never materialised.  (The template is in scan.cuh.)
#include <limits.h>
#include <vector>
#include <algorithm>

#include "intensity.h"
#include "metric.cuh"
#include "scan.cuh"

namespace hdp {


// ----------------------------------------------------------------------------------------------------
// k_hot_words
// ----------------------------------------------------------------------------------------------------
constexpr int kHotDays = 16;  // days of each of kHotYears words whose samples are in flight together

template <int PG, int J0, int UNIT, bool COLD>
__device__ __forceinline__ void hot_half(uint32_t (&m)[kHotYears][PG], const float *const (&xp)[kHotYears], const int (&jo)[kHotYears],
                                         const int (&nb)[kHotYears], int64_t ld_t, const float *ts)
{
    float v[kHotYears][kHotDays];
#pragma unroll
    for (int y = 0; y < kHotYears; y++)
#pragma unroll
        for (int j = 0; j < kHotDays; j++)                 // NaN = never hot: days outside the word
            v[y][j] = (unsigned)(J0 + j - jo[y]) < (unsigned)nb[y] ? __ldg(xp[y] + (int64_t)(J0 + j) * ld_t) : __int_as_float(0x7fc00000);
    if (UNIT != 0) {                                       // Kelvin / Fahrenheit input, converted as it is loaded (NaN stays NaN)
#pragma unroll
        for (int y = 0; y < kHotYears; y++)
#pragma unroll
            for (int j = 0; j < kHotDays; j++) v[y][j] = to_celsius_f(v[y][j], UNIT);
    }
#pragma unroll
    for (int j = 0; j < kHotDays; j++) {
        float t[PG];
#pragma unroll
        for (int q = 0; q < PG; q++) t[q] = ts[((J0 + j) * PG + q) * kTilePad];
#pragma unroll
        for (int y = 0; y < kHotYears; y++)
#pragma unroll
            for (int q = 0; q < PG; q++) {
                if (COLD) or_if_lt(m[y][q], v[y][j], t[q], 1u << (J0 + j));
                else or_if_gt(m[y][q], v[y][j], t[q], 1u << (J0 + j));
            }
    }
}

// COLD: the bits mark days with (double)x < thr (cold spells) instead of (double)x > thr.  The tile is then rounded UP
// (__double2float_ru), which keeps the double-precision `x < thr` exact for every float x: a thr that is a float is kept; else
// ru(thr) is the smallest float above thr, so no float lies in [thr, ru(thr)) and x < thr <=> x < ru(thr).  At the ends: thr >
// FLT_MAX becomes +inf, below which every finite float lies (all are < thr); thr < -FLT_MAX becomes -FLT_MAX, below which only
// -inf lies (the only float < thr).  NaN stays NaN and compares false on either side; the padding is -inf, never cold.
template <int PG, int UNIT, bool COLD>
__global__ void __launch_bounds__(256, PG <= 10 ? 3 : 2)
k_hot_words(const float *__restrict__ x, int64_t C, int64_t ld_t,
            const double *__restrict__ thr, int n_doy, int P,
            const int4 *__restrict__ words, const int *__restrict__ blk_start, const int *__restrict__ blk_words,
            int K, uint32_t *__restrict__ hot)
{
    extern __shared__ float thr_s[];                      // [percentile group][32 doy][PG][33]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int db = blockIdx.y;
    const int64_t c0 = (int64_t)blockIdx.x * kTileCells;
    const int Ppad = (P + PG - 1) / PG * PG;
    const int nd = min(kTileDoy, n_doy - db * kTileDoy);

    // Threshold tile.  Per cell the (doy, percentile) block of this tile is nd * P contiguous doubles in the reference's
    // [C, n_doy, P] order: a warp reads them with consecutive lanes, kFillLoads independent loads per lane in flight
    // (the fill is pure HBM latency), and scatters them to [group][doy][PG][cell].  Padding percentiles / days: +inf (-inf
    // for COLD), which no sample exceeds (falls below).
    const int n_el = nd * P;                               // doubles per cell
    if (nd < kTileDoy || Ppad != P)
        for (int i = tid; i < (Ppad / PG) * kTileDoy * PG * kTilePad; i += 256) thr_s[i] = __int_as_float(COLD ? 0xff800000 : 0x7f800000);
    __syncthreads();
    const float inv_p = 1.0f / (float)P;                   // e / P for e < 1024, P <= 32: (e + 0.5) / P is >= 1 / 64 away from every
    for (int e0 = 0; e0 < n_el; e0 += 32 * kFillLoads) {   // integer, far more than the error of the float product
        int dst[kFillLoads];
#pragma unroll
        for (int i = 0; i < kFillLoads; i++) {
            const int e = e0 + 32 * i + lane;
            const int j = __float2int_rz(((float)e + 0.5f) * inv_p), p = e - j * P, g = p / PG, q = p - g * PG;
            dst[i] = e < n_el ? ((g * kTileDoy + j) * PG + q) * kTilePad : -1;
        }
        for (int cell = warp; cell < kTileCells; cell += 8) {
            if (c0 + cell >= C) break;
            const double *src = thr + ((c0 + cell) * n_doy + (int64_t)db * kTileDoy) * P + e0 + lane;
            double v[kFillLoads];
#pragma unroll
            for (int i = 0; i < kFillLoads; i++) v[i] = dst[i] >= 0 ? __ldg(src + 32 * i) : 0.0;
#pragma unroll
            for (int i = 0; i < kFillLoads; i++)
                if (dst[i] >= 0) thr_s[dst[i] + cell] = COLD ? __double2float_ru(v[i]) : __double2float_rd(v[i]);
        }
    }
    __syncthreads();

    const int64_t c = c0 + lane;
    if (c >= C) return;
    // A warp takes kHotYears words (= years of this day-of-year block) at a time.  It first puts kHotDays days of each
    // of them in flight (kHotYears * kHotDays independent 128-byte loads per warp), then compares them against the days'
    // thresholds, which are read from shared memory into registers once per kHotYears samples.  Bits are collected at
    // the day's position inside the 32-day block (an immediate) and shifted to the word's own origin when stored.
    const int w_begin = blk_start[db], w_end = blk_start[db + 1];
    const int64_t plane_words = (int64_t)K * C;
    for (int i0 = w_begin + warp * kHotYears; i0 < w_end; i0 += 8 * kHotYears) {
        int kk[kHotYears], jo[kHotYears], nb[kHotYears];
        const float *xp[kHotYears];
        int j_hi = 0;
#pragma unroll
        for (int y = 0; y < kHotYears; y++) {
            const bool live = i0 + y < w_end;
            kk[y] = blk_words[live ? i0 + y : i0];
            const int4 w = words[kk[y]];                   // {t0, nbits, doy of bit 0, -}
            jo[y] = w.z & (kTileDoy - 1);
            nb[y] = live ? w.y : 0;
            xp[y] = x + ((int64_t)w.x - jo[y]) * ld_t + c; // day jd of the block is sample xp[y][jd * ld_t]
            if (live) j_hi = max(j_hi, jo[y] + nb[y]);
        }
        for (int pg = 0; pg < Ppad; pg += PG) {
            uint32_t m[kHotYears][PG];
#pragma unroll
            for (int y = 0; y < kHotYears; y++)
#pragma unroll
                for (int q = 0; q < PG; q++) m[y][q] = 0u;
            const float *ts = thr_s + (size_t)(pg / PG) * (kTileDoy * PG * kTilePad) + lane;
            uint32_t *hp[kHotYears];                               // word kk[y] of percentile pg of this cell; percentile planes are K * C words apart
#pragma unroll
            for (int y = 0; y < kHotYears; y++) hp[y] = hot + ((int64_t)pg * K + kk[y]) * C + c;
            hot_half<PG, 0, UNIT, COLD>(m, xp, jo, nb, ld_t, ts);
            if (j_hi > kHotDays) hot_half<PG, kHotDays, UNIT, COLD>(m, xp, jo, nb, ld_t, ts);      // warp-uniform
#pragma unroll
            for (int y = 0; y < kHotYears; y++)
#pragma unroll
                for (int q = 0; q < PG; q++)
                    if (nb[y] > 0 && pg + q < P) hp[y][(int64_t)q * plane_words] = m[y][q] >> jo[y];
        }
    }
}

// ----------------------------------------------------------------------------------------------------
// k_unpack_mask: hot words -> u8 [P, T, C]   (parity checks of the hot-day mask only)
// ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_unpack_mask(const uint32_t *__restrict__ hot, int64_t C, int64_t T, int P, int K, const int4 *__restrict__ words,
              uint8_t *__restrict__ mask)
{
    const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int k = blockIdx.y;
    if (c >= C) return;
    const int4 w = words[k];
    for (int p = 0; p < P; p++) {
        const uint32_t m = hot[((int64_t)p * K + k) * C + c];
        for (int j = 0; j < w.y; j++) mask[((int64_t)p * T + (w.x + j)) * C + c] = (m >> j) & 1u;
    }
}

// ----------------------------------------------------------------------------------------------------
// k_scan (scan.cuh): the plain and ONSET instances live here, the EXTENT twins in extent.cu
// ----------------------------------------------------------------------------------------------------
static std::atomic<int> g_scan_filter{1};        // test hook (hdp_b200_metrics_run_filter): 0 = k_scan queues every run
template int launch_scan<false, false>(const ScanConfig &, const ScanLaunch &);
template int launch_scan<true, false>(const ScanConfig &, const ScanLaunch &);

// ----------------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------------
static_assert(kTileDoy == 32, "word_length (seams.h) cuts words at 32-day blocks of the day-of-year axis");

// Cuts the time axis into hot-day words (word_length) and groups them by day-of-year block.  A word holds consecutive days of
// year d0 .. d0 + nb - 1, so checking its first and last day checks every map entry: an entry >= n_doy inside a word (noleap
// thresholds with a standard-calendar run: 31 December of a leap year maps to 365 in the word that starts at 352) would otherwise
// meet k_hot_words' +inf tile padding and be silently never hot.
static int build_words(const int32_t *doy_map, int64_t T, int n_doy, WordPlan &plan)
{
    plan.n_blk = (n_doy + kTileDoy - 1) / kTileDoy;
    for (int64_t t = 0; t < T;) {
        const int d0 = doy_map[t];
        if (d0 < 0 || d0 >= n_doy) return HDP_B200_ERR_INVALID;
        const int nb = word_length(doy_map, t, T);
        if (d0 + nb - 1 >= n_doy) return HDP_B200_ERR_INVALID;
        plan.words.push_back(make_int4((int)t, nb, d0, 0));
        t += nb;
    }
    const int K = (int)plan.words.size();
    plan.blk_start.assign(plan.n_blk + 1, 0);
    for (int k = 0; k < K; k++) plan.blk_start[plan.words[k].z / kTileDoy + 1]++;
    for (int b = 0; b < plan.n_blk; b++) plan.blk_start[b + 1] += plan.blk_start[b];
    plan.blk_words.resize(K);
    std::vector<int> fill(plan.blk_start.begin(), plan.blk_start.end() - 1);
    for (int k = 0; k < K; k++) plan.blk_words[fill[plan.words[k].z / kTileDoy]++] = k;
    return HDP_B200_OK;
}

static int64_t words_upper_bound(int64_t T, int n_doy)
{
    // regular daily calendars: every (partial) year contributes at most n_blk + 1 words
    const int64_t n_blk = (n_doy + kTileDoy - 1) / kTileDoy;
    return (T / std::max(n_doy, 1) + 2) * (n_blk + 1) + 1;
}

static int64_t count_words(const int32_t *doy_map, int64_t T)
{
    int64_t K = 0;
    for (int64_t t = 0; t < T; K++) t += word_length(doy_map, t, T);
    return K;
}

// A threshold table without a day-of-year axis (n_doy = 1: the no-season and fixed-value variants, every day reads row 0) would
// cut the series into one-day words, because word_length needs consecutive days of year, and a run of a few decades would then
// have more words than k_scan and k_intensity keep in shared memory.  The pass sees such a table as kTileDoy identical rows
// instead (replicated into the workspace, replicate_rows) with day t on row t mod kTileDoy, so its words are 32 days long.
static int pass_n_doy(int n_doy) { return n_doy == 1 ? kTileDoy : n_doy; }

// The day-of-year map the pass cuts into words: h_doy_map itself, or for n_doy = 1 (where every entry must be 0) t mod kTileDoy.
static int pass_doy_map(const int32_t *h_doy_map, int64_t T, int n_doy, std::vector<int32_t> &own, const int32_t *&map)
{
    map = h_doy_map;
    if (n_doy != 1) return HDP_B200_OK;
    own.resize((size_t)T);
    for (int64_t t = 0; t < T; t++) {
        if (h_doy_map[t] != 0) return HDP_B200_ERR_INVALID;
        own[(size_t)t] = (int32_t)(t % kTileDoy);
    }
    map = own.data();
    return HDP_B200_OK;
}

// thr [C, 1, P] -> rep [C, kTileDoy, P]: row 0 of every cell, then copies that double the rows already there.
static int replicate_rows(const double *thr, int64_t C, int P, double *rep, cudaStream_t st)
{
    const size_t row = (size_t)P * sizeof(double), pitch = kTileDoy * row;
    HDP_CUDA_TRY(cudaMemcpy2DAsync(rep, pitch, thr, row, row, (size_t)C, cudaMemcpyDeviceToDevice, st));
    for (int n = 1; n < kTileDoy; n *= 2)
        HDP_CUDA_TRY(cudaMemcpy2DAsync(rep + (size_t)n * P, pitch, rep, pitch, n * row, (size_t)C, cudaMemcpyDeviceToDevice, st));
    return HDP_B200_OK;
}

int pick_pg(int P)
{
    const int cand[] = {4, 8, 10, 16, 20};
    int best = 4, best_waste = INT_MAX;
    for (int pg : cand) {
        const int waste = (P + pg - 1) / pg * pg - P;
        if (waste < best_waste || (waste == best_waste && pg > best && pg <= 20)) { best = pg; best_waste = waste; }
    }
    return best;
}

// Workspace layout; `intensity` appends the intensity pass's season tables behind what the metric pass uses, then each of the
// n_measures measures its normalised copy (need_norm[m]) and, for n_doy = 1, its replicated thresholds.
static Layout carve(void *ws, size_t ws_bytes, int64_t C, int64_t T, int n_measures, const bool *need_norm, int64_t K, int n_doy, int P,
                    int Y, bool intensity)
{
    Layout L;
    Carver cv(ws, ws_bytes);
    L.words = cv.take<int4>((size_t)K + 1);
    L.blk_start = cv.take<int>((size_t)(pass_n_doy(n_doy) + kTileDoy - 1) / kTileDoy + 1);
    L.blk_words = cv.take<int>((size_t)K + 1);
    L.seasons = cv.take<int4>((size_t)2 * (Y + 1));
    L.lut = cv.take<uint32_t>((size_t)2 * 8192);
    L.hot = cv.take<uint32_t>((size_t)P * K * C);
    if (intensity) L.int_seasons = cv.take<int4>((size_t)2 * (Y + 1));
    for (int m = 0; m < n_measures; m++) {
        if (need_norm[m]) L.xn[m] = cv.take<float>((size_t)C * T);
        if (n_doy == 1) L.thr_rep[m] = cv.take<double>((size_t)C * kTileDoy * P);
    }
    L.total = cv.off;
    return L;
}

static bool bad_dims(int64_t C, int64_t T, int n_doy, int P)
{
    return C < 0 || T < 0 || n_doy <= 0 || P <= 0 || T > 0x3fffffff;
}

size_t metric_pass_workspace_bytes(int64_t C, int64_t T, const int64_t *ld_c, int n_measures, int n_doy, int P, int Y,
                                   const int32_t *h_doy_map, bool intensity)
{
    if (bad_dims(C, T, n_doy, P) || Y < 0) return 0;
    const int64_t K = n_doy == 1 ? (T + kTileDoy - 1) / kTileDoy : h_doy_map ? count_words(h_doy_map, T) : words_upper_bound(T, n_doy);
    bool need_norm[2] = {};
    for (int m = 0; m < n_measures; m++) need_norm[m] = ld_c[m] != 1;
    return carve(nullptr, 0, C, T, n_measures, need_norm, K, n_doy, P, Y, intensity).total;
}

// Prepares each of the n_measures measures (its thresholds replicated for n_doy = 1, its samples copied to time-major L.xn[m], ld_t
// = C, when ld_c != 1) and runs k_hot_words on one measure, k_hot_pair on two: the words then mark the days on which both measures
// pass their thresholds.  On success plan / L describe what lives in the workspace, L.thr / L.n_doy the thresholds and L.x / L.ld_t
// the samples the kernels read.  `unit` is a plain unit code (0 - 2); `cold` makes the words cold-day bits.
static int run_hot_words(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                         int Y, void *ws, size_t ws_bytes, cudaStream_t st, WordPlan &plan, Layout &L,
                         int64_t carve_cells = 0, bool tables_resident = false, int unit = 0, bool intensity = false, bool cold = false)
{
    if (unit < 0 || unit > 2) return HDP_B200_ERR_INVALID;
    std::vector<int32_t> own_map;
    const int32_t *doy_map = nullptr;
    int rc = pass_doy_map(h_doy_map, T, n_doy, own_map, doy_map);
    if (rc != HDP_B200_OK) return rc;
    rc = build_words(doy_map, T, pass_n_doy(n_doy), plan);
    if (rc != HDP_B200_OK) return rc;
    const int K = (int)plan.words.size();
    bool need_norm[2] = {};
    for (int m = 0; m < n_measures; m++) need_norm[m] = ms[m].ld_c != 1;
    L = carve(ws, ws_bytes, std::max(C, carve_cells), T, n_measures, need_norm, K, n_doy, P, Y, intensity);
    if (ws == nullptr || L.total > ws_bytes) return HDP_B200_ERR_WORKSPACE;
    L.n_doy = pass_n_doy(n_doy);
    for (int m = 0; m < n_measures; m++) {
        L.thr[m] = ms[m].thr;
        L.x[m] = ms[m].x;
        L.ld_t[m] = ms[m].ld_t;
    }
    if (C == 0 || T == 0) return HDP_B200_OK;
    for (int m = 0; m < n_measures; m++) {
        if (L.thr_rep[m]) {
            rc = replicate_rows(ms[m].thr, C, P, L.thr_rep[m], st);
            if (rc != HDP_B200_OK) return rc;
            L.thr[m] = L.thr_rep[m];
        }
        if (L.xn[m]) {
            rc = normalize_layout(ms[m].x, C, T, ms[m].ld_t, ms[m].ld_c, L.xn[m], st);
            if (rc != HDP_B200_OK) return rc;
            L.x[m] = L.xn[m];
            L.ld_t[m] = C;
        }
    }
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.words, plan.words.data(), sizeof(int4) * K, cudaMemcpyHostToDevice, st));
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.blk_start, plan.blk_start.data(), sizeof(int) * plan.blk_start.size(), cudaMemcpyHostToDevice, st));
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.blk_words, plan.blk_words.data(), sizeof(int) * K, cudaMemcpyHostToDevice, st));
    if (n_measures == 2) return run_hot_pair(L, plan, C, P, st, unit, cold);

    const int pg = pick_pg(P);
    const int Ppad = (P + pg - 1) / pg * pg;
    const size_t smem = (size_t)kTileDoy * Ppad * kTilePad * sizeof(float);
    dim3 grid((unsigned)((C + kTileCells - 1) / kTileCells), (unsigned)plan.n_blk);
    const auto kernel = hot_kernel(pg, unit, cold, [](auto PG, auto U, auto CO) {
        return k_hot_words<decltype(PG)::value, decltype(U)::value, decltype(CO)::value>;
    });
    KernelTimer timer(kHotWords, st);
    HDP_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, 256, smem, st>>>(L.x[0], C, L.ld_t[0], L.thr[0], L.n_doy, P, L.words, L.blk_start, L.blk_words, K, L.hot);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

// k_scan's season tables: per hemisphere, passes of sorted, disjoint seasons (one launch each).
struct ScanSeason { int a, b, row; };
using ScanPasses = std::vector<std::vector<ScanSeason>>;

// Splits a hemisphere's season table (season_table, sorted by start) into passes: each season goes to the first pass it does
// not overlap.  Seasons of more than 65 535 days do not fit the u16 output.
static int scan_passes(const int32_t *tab, int Y, ScanPasses &passes)
{
    for (int y = 0; y < Y; y++) {
        const ScanSeason s = {tab[4 * y], tab[4 * y + 1], tab[4 * y + 2]};
        if (s.b - s.a > 65535) return HDP_B200_ERR_UNSUPPORTED;
        size_t i = 0;
        while (i < passes.size() && passes[i].back().b > s.a) i++;
        if (i == passes.size()) passes.emplace_back();
        passes[i].push_back(s);
    }
    return HDP_B200_OK;
}

static int scan_config(const int32_t *h_defs, int D, int64_t T, const ScanPasses (&passes)[2], ScanConfig &cfg)
{
    cfg.n_pass = std::max(passes[0].size(), passes[1].size());
    // bit-sliced definition tables (see k_scan)
    ScanTables &tabs = cfg.tabs;
    int max_min_dur = 0, max_break_all = 0;
    int64_t max_subs_all = 0;
    std::vector<int64_t> subs(D);
    for (int i = 0; i < D; i++) {
        max_min_dur = std::max(max_min_dur, h_defs[3 * i]);
        max_break_all = std::max(max_break_all, h_defs[3 * i + 1]);
        subs[i] = std::min<int64_t>(std::max<int64_t>(h_defs[3 * i + 2], 0), T);   // more subsequent events than days cannot happen
        max_subs_all = std::max(max_subs_all, subs[i]);
    }
    if (max_min_dur > 8190 || max_break_all > 8190) return HDP_B200_ERR_UNSUPPORTED;
    tabs.ge_len = max_min_dur + 2;
    tabs.brk_len = max_break_all + 2;
    int ks_needed = 1;
    while ((max_subs_all >> ks_needed) != 0) ks_needed++;
    for (int k = 0; k < 32; k++) {
        tabs.max_subs_plane[k] = 0u;
        for (int i = 0; i < D; i++) tabs.max_subs_plane[k] |= (uint32_t)((subs[i] >> k) & 1) << i;
    }
    cfg.lut.assign(tabs.ge_len + tabs.brk_len, 0u);
    for (int l = 0; l < tabs.ge_len; l++)
        for (int i = 0; i < D; i++) if (h_defs[3 * i] <= l) cfg.lut[l] |= 1u << i;
    for (int g = 0; g < tabs.brk_len; g++)
        for (int i = 0; i < D; i++) if (h_defs[3 * i + 1] < g) cfg.lut[tabs.ge_len + g] |= 1u << i;
    // run filter (see k_scan): only when the look-back / look-ahead fits the 32-day neighbourhood
    int min_min_dur = INT_MAX;
    for (int i = 0; i < D; i++) min_min_dur = std::min(min_min_dur, h_defs[3 * i]);
    tabs.f_lmin = min_min_dur;
    tabs.f_bmax = max_break_all;
    tabs.f_on = (min_min_dur >= 2 && min_min_dur <= 32 && max_break_all >= 0 && max_break_all <= 30 && g_scan_filter) ? 1 : 0;
    // accumulators: four definitions per register when every season fits 8-bit lanes, else two
    int max_season = 0;
    for (int h = 0; h < 2; h++)
        for (const auto &pass : passes[h])
            for (const ScanSeason &se : pass) max_season = std::max(max_season, se.b - se.a);
    cfg.bytes = max_season <= 255;
    const int per = cfg.bytes ? 4 : 2;
    const int ng = (D + per - 1) / per;
    cfg.ng = ng <= 2 ? 2 : ng <= 3 ? 3 : ng <= 4 ? 4 : ng <= 6 ? 6 : ng <= 8 ? 8 : ng <= 12 ? 12 : 16;
    cfg.ks = ks_needed <= 1 ? 1 : ks_needed <= 2 ? 2 : 32;          // bit planes of the max_subs counters: 1, 2 or all 32
    // compile-time filter constants for the usual shapes (seasons of at most 255 days, common definition sets)
    if (cfg.bytes && cfg.ks == 1 && tabs.f_on && tabs.f_lmin == 3 && (tabs.f_bmax == 1 || tabs.f_bmax == 2)) {
        cfg.lmin = 3;
        cfg.bmax = tabs.f_bmax;
    }
    return HDP_B200_OK;
}

// k_scan over the hot words in L (one launch per pass): the integer metrics u16 [4, P, D, Y, C], with `onset` u16 [6, P, D, Y, C]
// (HWO, HWE behind them, from the ONSET twin of the same instantiation).  With `ext` the EXTENT twin also adds the weights of the
// heatwave days to ext->diff (d_out may then be NULL).
static int run_scan(const Layout &L, const WordPlan &plan, int64_t C, int64_t T, int P, const int32_t *h_defs, int D,
                    const ScanPasses (&passes)[2], int Y, const uint8_t *d_is_south, uint16_t *d_out, cudaStream_t st, bool tables_resident,
                    bool onset, const ScanExtent *ext = nullptr)
{
    const int K = (int)plan.words.size();
    ScanConfig cfg;
    const int rc = scan_config(h_defs, D, T, passes, cfg);
    if (rc != HDP_B200_OK) return rc;
    const ScanTables &tabs = cfg.tabs;
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.lut, cfg.lut.data(), sizeof(uint32_t) * cfg.lut.size(), cudaMemcpyHostToDevice, st));
    size_t scan_smem = (((size_t)kScanWarps * kScanQueueWords + cfg.lut.size() + 3) & ~(size_t)3) * sizeof(uint32_t) + ((size_t)K + 1) * sizeof(int4);
    if (scan_smem > 200 * 1024) return HDP_B200_ERR_UNSUPPORTED;             // > ~9 000 hot words (~800 years of daily data)
    if (cfg.bytes) scan_smem += 256 * sizeof(uint32_t);                      // k_scan's hwa_rcp
    const int64_t n_warps = ((C + 31) / 32) * P;                             // one warp per (32 cells, percentile)

    // all passes of both hemispheres live side by side in the workspace: north passes, then south passes
    std::vector<int4> tab;
    std::vector<size_t> off[2];
    for (int h = 0; h < 2; h++)
        for (const auto &pass : passes[h]) {
            off[h].push_back(tab.size());
            for (const ScanSeason &s : pass) tab.push_back(make_int4(s.a, s.b, s.row, 0));
        }
    if (!tables_resident) HDP_CUDA_TRY(cudaMemcpyAsync(L.seasons, tab.data(), sizeof(int4) * tab.size(), cudaMemcpyHostToDevice, st));
    ScanLaunch a;
    a.grid = (unsigned)((n_warps + kScanWarps - 1) / kScanWarps);
    a.smem = scan_smem;
    a.st = st;
    a.hot = L.hot; a.C = C; a.K = K; a.T = (int)T; a.words = L.words; a.P = P; a.D = D;
    a.ge_tab = L.lut; a.brk_tab = L.lut + tabs.ge_len;
    a.Y = Y; a.is_south = d_is_south; a.out = d_out;
    if (ext) a.ext = *ext;
    for (size_t ip = 0; ip < cfg.n_pass; ip++) {
        a.sn = ip < passes[0].size() ? L.seasons + off[0][ip] : L.seasons;
        a.ss = ip < passes[1].size() ? L.seasons + off[1][ip] : L.seasons;
        a.nn = ip < passes[0].size() ? (int)passes[0][ip].size() : 0;
        a.ns = ip < passes[1].size() ? (int)passes[1][ip].size() : 0;
        KernelTimer timer(kScan, st);
        const int lrc = ext ? launch_scan<false, true>(cfg, a) : onset ? launch_scan<true, false>(cfg, a) : launch_scan<false, false>(cfg, a);
        if (lrc != HDP_B200_OK) return lrc;
        HDP_LAUNCH_CHECK();
    }
    return HDP_B200_OK;
}

// Every measure of a pass must have samples and thresholds once there is work
static bool missing_measure(const Measure *ms, int n_measures, int64_t C, int64_t T)
{
    for (int m = 0; m < n_measures; m++)
        if (C > 0 && T > 0 && (!ms[m].x || !ms[m].thr)) return true;
    return false;
}

int metric_pass(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                const int32_t *h_defs, int D,
                const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                const uint8_t *d_is_south, uint16_t *d_out, float *d_int,
                void *d_workspace, size_t workspace_bytes, void *stream, int64_t carve_cells, bool tables_resident, int input_unit,
                const ScanExtent *ext)
{
    if (bad_dims(C, T, n_doy, P) || D <= 0 || Y < 0) return HDP_B200_ERR_INVALID;
    if ((T > 0 && !h_doy_map) || !h_defs || (Y > 0 && (!h_season_north || !h_season_south))) return HDP_B200_ERR_INVALID;
    if (missing_measure(ms, n_measures, C, T)) return HDP_B200_ERR_INVALID;
    if (P > HDP_B200_MAX_PERCENTILES || D > HDP_B200_MAX_DEFINITIONS) return HDP_B200_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    // input_unit of the C ABI = unit code | HDP_B200_COLD | HDP_B200_ONSET; the kernels' launchers see them as plain values
    const bool cold = (input_unit & HDP_B200_COLD) != 0, onset = (input_unit & HDP_B200_ONSET) != 0;
    const int unit = input_unit & ~(HDP_B200_COLD | HDP_B200_ONSET);
    if (onset && !d_out) return HDP_B200_ERR_INVALID;                                   // HWO / HWE are planes of the u16 output
    if (ext && (onset || n_measures != 1)) return HDP_B200_ERR_INVALID;                 // extent: no ONSET twin, no compound pass

    // the season tables of both hemispheres, north then south (Y + 1 rows apart, as k_intensity reads them)
    std::vector<int32_t> seasons((size_t)8 * (Y + 1), 0);
    ScanPasses passes[2];
    for (int h = 0; h < 2; h++) {
        int32_t *tab = seasons.data() + (size_t)4 * (Y + 1) * h;
        const bool disjoint = intensity_season_table(h == 0 ? h_season_north : h_season_south, Y, T, tab);
        if ((d_int || ext) && !disjoint) return HDP_B200_ERR_UNSUPPORTED;               // k_intensity: one open season per lane;
        if (d_out || ext) {                                                             // extent: no day counted twice
            const int rc = scan_passes(tab, Y, passes[h]);
            if (rc != HDP_B200_OK) return rc;
        }
    }

    WordPlan plan;
    Layout L;
    int rc = run_hot_words(ms, n_measures, C, T, n_doy, P, h_doy_map, Y, d_workspace, workspace_bytes, st, plan, L,
                           carve_cells, tables_resident, unit, d_int != nullptr, cold);
    if (rc != HDP_B200_OK || C == 0 || Y == 0) return rc;
    if (d_out || ext) {
        rc = run_scan(L, plan, C, T, P, h_defs, D, passes, Y, d_is_south, d_out, st, tables_resident, onset, ext);
        if (rc != HDP_B200_OK) return rc;
    }
    for (int m = 0; d_int && m < n_measures && rc == HDP_B200_OK; m++)     // one block per measure, on the same words
        rc = run_intensity(L, plan, m, C, T, P, h_defs, D, seasons, Y, d_is_south, d_int + (size_t)m * 3 * P * D * Y * C, st,
                           tables_resident || m > 0, unit, cold);
    return rc;
}

// hdp_b200_hot_days and hdp_b200_compound_hot_days: the hot words, unpacked to u8 [P, T, C]
static int hot_days_pass(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                         uint8_t *d_mask, void *d_workspace, size_t workspace_bytes, void *stream, int unit, bool cold)
{
    if (bad_dims(C, T, n_doy, P) || !h_doy_map && T > 0) return HDP_B200_ERR_INVALID;
    if (missing_measure(ms, n_measures, C, T) || (C > 0 && T > 0 && !d_mask)) return HDP_B200_ERR_INVALID;
    if (P > HDP_B200_MAX_PERCENTILES) return HDP_B200_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    WordPlan plan;
    Layout L;
    int rc = run_hot_words(ms, n_measures, C, T, n_doy, P, h_doy_map, 0, d_workspace, workspace_bytes, st, plan, L,
                           0, false, unit, false, cold);
    if (rc != HDP_B200_OK || C == 0 || T == 0) return rc;
    const int K = (int)plan.words.size();
    dim3 grid((unsigned)((C + 255) / 256), (unsigned)K);
    if (K > 65535) return HDP_B200_ERR_UNSUPPORTED;
    KernelTimer timer(kUnpackMask, st);
    k_unpack_mask<<<grid, 256, 0, st>>>(L.hot, C, T, P, K, L.words, d_mask);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace hdp

using namespace hdp;

extern "C" {

size_t hdp_b200_metrics_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                                        int n_doy, int P, int D, int Y, const int32_t *h_doy_map)
{
    (void)ld_t; (void)D;
    return metric_pass_workspace_bytes(C, T, &ld_c, 1, n_doy, P, Y, h_doy_map, false);
}

void hdp_b200_metrics_run_filter(int on) { g_scan_filter = on != 0; }

int hdp_b200_metrics_kernel_choice(const int32_t *h_defs, int D, const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                                   int64_t T, int *info)
{
    if (!h_defs || !info || D <= 0 || Y < 0 || T < 0 || T > 0x3fffffff || (Y > 0 && (!h_season_north || !h_season_south)))
        return HDP_B200_ERR_INVALID;
    if (D > HDP_B200_MAX_DEFINITIONS) return HDP_B200_ERR_UNSUPPORTED;
    std::vector<int32_t> tab((size_t)4 * (Y + 1));
    ScanPasses passes[2];
    for (int h = 0; h < 2; h++) {
        season_table(h == 0 ? h_season_north : h_season_south, Y, T, tab.data());
        const int rc = scan_passes(tab.data(), Y, passes[h]);
        if (rc != HDP_B200_OK) return rc;
    }
    ScanConfig cfg;
    const int rc = scan_config(h_defs, D, T, passes, cfg);
    if (rc != HDP_B200_OK) return rc;
    info[0] = cfg.bytes ? 8 : 16; info[1] = cfg.ng; info[2] = cfg.ks; info[3] = cfg.tabs.f_on;
    info[4] = cfg.lmin; info[5] = cfg.bmax; info[6] = (int)cfg.n_pass;
    return HDP_B200_OK;
}

int hdp_b200_hot_days(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                      const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                      uint8_t *d_mask, void *d_workspace, size_t workspace_bytes, void *stream)
{
    const Measure m = {d_measure, ld_t, ld_c, d_thr};
    return hot_days_pass(&m, 1, C, T, n_doy, P, h_doy_map, d_mask, d_workspace, workspace_bytes, stream, 0, false);
}

int hdp_b200_compound_hot_days(const float *d_a, int64_t ld_t_a, int64_t ld_c_a, const float *d_b, int64_t ld_t_b, int64_t ld_c_b,
                               int64_t C, int64_t T, const double *d_thr_a, const double *d_thr_b, int n_doy, int P,
                               const int32_t *h_doy_map, uint8_t *d_mask, void *d_workspace, size_t workspace_bytes, void *stream,
                               int input_unit)
{
    const Measure ms[2] = {{d_a, ld_t_a, ld_c_a, d_thr_a}, {d_b, ld_t_b, ld_c_b, d_thr_b}};
    return hot_days_pass(ms, 2, C, T, n_doy, P, h_doy_map, d_mask, d_workspace, workspace_bytes, stream, input_unit & ~HDP_B200_COLD,
                         (input_unit & HDP_B200_COLD) != 0);
}

int hdp_b200_metrics(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                     const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                     const int32_t *h_defs, int D,
                     const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                     const uint8_t *d_is_south, uint16_t *d_out,
                     void *d_workspace, size_t workspace_bytes, void *stream, int input_unit)
{
    if (C > 0 && Y > 0 && !d_out) return HDP_B200_ERR_INVALID;
    const Measure m = {d_measure, ld_t, ld_c, d_thr};
    return metric_pass(&m, 1, C, T, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y, d_is_south, d_out, nullptr,
                       d_workspace, workspace_bytes, stream, C, false, input_unit);
}

}  // extern "C"
