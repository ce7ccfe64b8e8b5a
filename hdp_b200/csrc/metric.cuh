// metric.cuh - what the hot-word kernels (k_hot_words in metric.cu, k_hot_pair in compound.cu) and the intensity kernel
// (intensity.cu) share with the fused metric pass (metric.cu, metric_pass): the tile constants, the instance dispatch, the hot-day
// words and the workspace layout they live in.
#pragma once

#include <type_traits>
#include <vector>

#include "common.cuh"

namespace hdp {

// The hot-word tiles of k_hot_words (metric.cu) and k_hot_pair (compound.cu)
constexpr int kTileCells = 32;
constexpr int kTileDoy = 32;
constexpr int kHotYears = 2;  // words (years) a warp compares against one register copy of the day's thresholds
constexpr int kFillLoads = 5;  // doubles of the threshold tile a lane has in flight
constexpr int kTilePad = 33;   // [.. ][33]: conflict-free both for the e-major fill and the lane-major reads

#ifdef __CUDACC__
// m |= bit where v > t (false when either side is NaN): one compare and one predicated OR with an immediate
__device__ __forceinline__ void or_if_gt(uint32_t &m, float v, float t, uint32_t bit)
{
    asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}" : "+r"(m) : "f"(v), "f"(t), "r"(bit));
}

// the same with v < t: the cold-day bits of a cold-spell pass
__device__ __forceinline__ void or_if_lt(uint32_t &m, float v, float t, uint32_t bit)
{
    asm("{\n\t.reg .pred p;\n\tsetp.lt.f32 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}" : "+r"(m) : "f"(v), "f"(t), "r"(bit));
}
#endif

// The instance of a hot-word kernel template <PG, UNIT, COLD> (k_hot_words, k_hot_pair) for percentile group size pg (pick_pg),
// plain unit code `unit` (0 - 2) and direction `cold`: inst(PG, UNIT, COLD), called with std::integral_constant arguments, names it.
template <class Inst>
auto hot_kernel(int pg, int unit, bool cold, Inst inst)
{
    using std::integral_constant;
    auto dir = [&](auto pg_c, auto unit_c) { return cold ? inst(pg_c, unit_c, std::true_type()) : inst(pg_c, unit_c, std::false_type()); };
    auto by_unit = [&](auto pg_c) {
        return unit == 0 ? dir(pg_c, integral_constant<int, 0>()) : unit == 1 ? dir(pg_c, integral_constant<int, 1>())
                                                                              : dir(pg_c, integral_constant<int, 2>());
    };
    switch (pg) {
    case 4: return by_unit(integral_constant<int, 4>());
    case 8: return by_unit(integral_constant<int, 8>());
    case 10: return by_unit(integral_constant<int, 10>());
    case 16: return by_unit(integral_constant<int, 16>());
    default: return by_unit(integral_constant<int, 20>());
    }
}

struct WordPlan {
    std::vector<int4> words;        // {t0, nbits, doy of bit 0, 0}
    std::vector<int> blk_start;     // [n_blk + 1]
    std::vector<int> blk_words;     // word ids grouped by day-of-year block
    int n_blk = 0;
};

struct Layout {
    size_t total = 0;
    int4 *words = nullptr;
    int *blk_start = nullptr, *blk_words = nullptr;
    int4 *seasons = nullptr;
    uint32_t *lut = nullptr;
    uint32_t *hot = nullptr;
    int4 *int_seasons = nullptr;    // intensity pass only: its season tables (north, then south)
    int n_doy = 0;
    // per measure of the pass (one, or two for a compound pass):
    float *xn[2] = {};              // ld_c != 1 only: the samples normalised to cell-contiguous [T, C]
    double *thr_rep[2] = {};        // n_doy = 1 only: the thresholds replicated to kTileDoy rows (metric.cu, pass_n_doy)
    const double *thr[2] = {};      // the thresholds the kernels read, [C, n_doy, P]: the caller's, or thr_rep
    const float *x[2] = {};         // the samples the kernels read, cell-contiguous, ld_t apart: the caller's, or xn
    int64_t ld_t[2] = {};
};

// Workspace of metric_pass over n_measures measures with cell strides ld_c[]; `intensity` appends the intensity pass's season tables
// behind what the metric pass uses.
size_t metric_pass_workspace_bytes(int64_t C, int64_t T, const int64_t *ld_c, int n_measures, int n_doy, int P, int Y,
                                   const int32_t *h_doy_map, bool intensity);

// pick_pg: the percentiles per group of the hot-word kernels (PG of k_hot_words and k_hot_pair) for P percentiles
int pick_pg(int P);

// k_hot_pair (compound.cu): percentile groups per CTA, CTAs per (cells, day-of-year block) and shared-memory bytes per CTA for P
// percentiles; false when P is outside 1 .. HDP_B200_MAX_PERCENTILES
bool hot_pair_plan(int P, int &pg, int &slices, int &groups_per_slice, size_t &smem);

// k_hot_pair over both measures' samples and thresholds in L: the compound hot-day words in L.hot
int run_hot_pair(const Layout &L, const WordPlan &plan, int64_t C, int P, cudaStream_t st, int unit, bool cold);

// k_intensity over the hot words in L: the intensity metrics f32 [3, P, D, Y, C] of measure m of L (its samples and thresholds).
// `seasons` i32 [2, Y + 1, 4]: the season tables of both hemispheres as intensity_season_table (intensity.h) accepts them.  `unit`:
// a plain unit code (0 - 2); `cold`: the words are cold-day bits and the intensity is the deficit below the threshold.
int run_intensity(const Layout &L, const WordPlan &plan, int m, int64_t C, int64_t T, int P, const int32_t *h_defs, int D,
                  const std::vector<int32_t> &seasons, int Y, const uint8_t *d_is_south, float *d_int, cudaStream_t st,
                  bool tables_resident, int unit, bool cold);

}  // namespace hdp
