// extent.cu - heatwave spatial extent (hdp_b200_extent): the weighted number of cells of each region that are on a heatwave day,
// for every day, percentile and definition.
//
// k_scan's EXTENT twins (scan.cuh, instantiated here) add +w / -w at the first day / the day after every in-season heatwave block
// of a cell to the difference array diff i64 [R, P, D, T + 1] in the workspace; k_extent_prefix then adds the inclusive prefix sum
// of every diff row to the caller's d_ext i64 [R, P, D, T].  All sums are of integers, so the result does not depend on the order
// of the reductions or on how the cells are split over calls.
#include "scan.cuh"

namespace hdp {

template int launch_scan<false, true>(const ScanConfig &, const ScanLaunch &);

constexpr int kPrefixThreads = 1024;

// One CTA per (r, p, d) row: ext[row, t] += sum_{u <= t} diff[row, u] for t < T, in tiles of kPrefixThreads days (a warp scan, then
// a scan of the warp totals, then the carry of the tiles before).  Unsigned arithmetic: the sums are exact two's complement.
__global__ void __launch_bounds__(kPrefixThreads)
k_extent_prefix(const int64_t *__restrict__ diff, int64_t T, int64_t *__restrict__ ext)
{
    __shared__ uint64_t warp_sum[kPrefixThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t *d = (const uint64_t *)diff + (int64_t)blockIdx.x * (T + 1);
    uint64_t *o = (uint64_t *)ext + (int64_t)blockIdx.x * T;
    uint64_t carry = 0;
    for (int64_t t0 = 0; t0 < T; t0 += kPrefixThreads) {
        const int64_t t = t0 + threadIdx.x;
        uint64_t v = t < T ? d[t] : 0ull;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const uint64_t u = __shfl_up_sync(0xffffffffu, v, k);
            if (lane >= k) v += u;
        }
        if (lane == 31) warp_sum[warp] = v;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = warp_sum[lane];
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) {
                const uint64_t u = __shfl_up_sync(0xffffffffu, w, k);
                if (lane >= k) w += u;
            }
            warp_sum[lane] = w;
        }
        __syncthreads();
        if (t < T) o[t] += carry + v + (warp > 0 ? warp_sum[warp - 1] : 0ull);
        carry += warp_sum[kPrefixThreads / 32 - 1];
        __syncthreads();                                              // warp_sum is refilled by the next tile
    }
}

size_t extent_diff_bytes(int64_t rows, int64_t T) { return align_up((size_t)rows * (size_t)(T + 1) * sizeof(int64_t)); }

int extent_prefix_launch(const int64_t *diff, int64_t rows, int64_t T, int64_t *ext, cudaStream_t st)
{
    if (rows == 0 || T == 0) return HDP_B200_OK;
    KernelTimer timer(kExtent, st);
    k_extent_prefix<<<(unsigned)rows, kPrefixThreads, 0, st>>>(diff, T, ext);
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

// The arguments hdp_b200_extent and hdp_b200_extent_host check alike: the region count, the output, the flags.
int extent_args(int R, const void *ext, int64_t T, int input_unit)
{
    if (R < 1 || (T > 0 && !ext) || (input_unit & HDP_B200_ONSET)) return HDP_B200_ERR_INVALID;
    if (R > HDP_B200_MAX_REGIONS) return HDP_B200_ERR_UNSUPPORTED;
    return HDP_B200_OK;
}

}  // namespace hdp

using namespace hdp;

extern "C" {

size_t hdp_b200_extent_workspace_bytes(int64_t C, int64_t T, int64_t ld_t, int64_t ld_c, int n_doy, int P, int D, int Y, int R,
                                       const int32_t *h_doy_map)
{
    (void)ld_t;
    if (C < 0 || T < 0 || P <= 0 || D <= 0 || R < 1 || R > HDP_B200_MAX_REGIONS) return 0;
    const size_t met = metric_pass_workspace_bytes(C, T, &ld_c, 1, n_doy, P, Y, h_doy_map, false);
    return met ? extent_diff_bytes((int64_t)R * P * D, T) + met : 0;
}

int hdp_b200_extent(const float *d_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                    const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                    const int32_t *h_defs, int D,
                    const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                    const uint8_t *d_is_south, const uint32_t *d_weight, const int32_t *d_region, int R,
                    int64_t *d_ext, uint16_t *d_out,
                    void *d_workspace, size_t workspace_bytes, void *stream, int input_unit)
{
    int rc = extent_args(R, d_ext, T, input_unit);
    if (rc != HDP_B200_OK) return rc;
    if (C < 0 || T < 0 || P <= 0 || D <= 0) return HDP_B200_ERR_INVALID;
    if (P > HDP_B200_MAX_PERCENTILES || D > HDP_B200_MAX_DEFINITIONS) return HDP_B200_ERR_UNSUPPORTED;
    const int64_t rows = (int64_t)R * P * D;
    const size_t diff_bytes = extent_diff_bytes(rows, T);
    if (!d_workspace || workspace_bytes < diff_bytes) return HDP_B200_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    ScanExtent ext;
    ext.diff = (int64_t *)d_workspace;
    ext.weight = d_weight;
    ext.region = d_region;
    ext.R = R;
    HDP_CUDA_TRY(cudaMemsetAsync(ext.diff, 0, diff_bytes, st));
    const Measure m = {d_measure, ld_t, ld_c, d_thr};
    rc = metric_pass(&m, 1, C, T, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y, d_is_south, d_out, nullptr,
                     (char *)d_workspace + diff_bytes, workspace_bytes - diff_bytes, stream, C, false, input_unit, &ext);
    if (rc != HDP_B200_OK) return rc;
    return extent_prefix_launch(ext.diff, rows, T, d_ext, st);
}

}  // extern "C"
