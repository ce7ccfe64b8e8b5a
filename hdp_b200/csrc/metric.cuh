// metric.cuh - what the intensity kernel (intensity.cu) shares with the fused metric pass (metric.cu, metric_pass): the hot-day
// words of k_hot_words and the workspace layout they live in.
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

// Workspace of metric_pass; `intensity` appends the intensity pass's season tables behind what the metric pass uses.
size_t metric_pass_workspace_bytes(int64_t C, int64_t T, int64_t ld_c, int n_doy, int P, int Y, const int32_t *h_doy_map, bool intensity);

// k_intensity over the hot words in L: the intensity metrics f32 [3, P, D, Y, C].  `seasons` i32 [2, Y + 1, 4]: the season tables
// of both hemispheres as intensity_season_table (intensity.h) accepts them.
int run_intensity(const Layout &L, const WordPlan &plan, const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                  const double *d_thr, int n_doy, int P, const int32_t *h_defs, int D, const std::vector<int32_t> &seasons, int Y,
                  const uint8_t *d_is_south, float *d_int, cudaStream_t st, bool tables_resident, int input_unit);

}  // namespace hdp
