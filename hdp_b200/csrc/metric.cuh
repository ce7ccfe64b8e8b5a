// metric.cuh - the pieces of metric.cu (path 2) that the intensity pass (intensity.cu) runs too: the hot-day words of
// k_hot_words, the workspace layout they live in, and the k_scan launch of the integer metrics.
#pragma once

#include <vector>

#include "common.cuh"

namespace hdp {

struct WordPlan {
    std::vector<int4> words;        // {t0, nbits, doy of bit 0, 0}
    std::vector<int> blk_start;     // [n_blk + 1]
    std::vector<int> blk_words;     // word ids grouped by day-of-year block
    int n_blk = 0;
};

struct Layout {
    size_t total = 0;
    float *xn = nullptr;
    int4 *words = nullptr;
    int *blk_start = nullptr, *blk_words = nullptr;
    int4 *seasons = nullptr;
    uint32_t *lut = nullptr;
    uint32_t *hot = nullptr;
    int4 *int_seasons = nullptr;    // intensity pass only: its season tables (north, then south)
};

// Workspace layout; `intensity` appends the intensity pass's season tables behind what the metric pass uses.
Layout carve(void *ws, size_t ws_bytes, int64_t C, int64_t T, bool need_norm, int64_t K, int n_doy, int P, int Y, bool intensity = false);
int64_t count_words(const int32_t *doy_map, int64_t T);
int64_t words_upper_bound(int64_t T, int n_doy);
bool bad_dims(int64_t C, int64_t T, int n_doy, int P);

// Runs k_hot_words (after the layout-normalising copy when ld_c != 1: the samples then live in L.xn, time-major, ld_t = C);
// on success plan / L describe what lives in the workspace.
int run_hot_words(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                  const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                  int Y, void *ws, size_t ws_bytes, cudaStream_t st, WordPlan &plan, Layout &L,
                  int64_t carve_cells = 0, bool tables_resident = false, int input_unit = 0, bool intensity = false);

// The metric pass's season tables: clamped and split into passes of sorted, disjoint seasons per hemisphere.
struct ScanSeason { int a, b, row; };
using ScanPasses = std::vector<std::vector<ScanSeason>>;
int scan_passes(const int32_t *h_season_north, const int32_t *h_season_south, int Y, int64_t T, ScanPasses (&passes)[2]);

// k_scan over the hot words in L (one launch per pass): the integer metrics u16 [4, P, D, Y, C].
int run_scan(const Layout &L, const WordPlan &plan, int64_t C, int64_t T, int P, const int32_t *h_defs, int D,
             const ScanPasses (&passes)[2], int Y, const uint8_t *d_is_south, uint16_t *d_out, cudaStream_t st, bool tables_resident);

}  // namespace hdp
