// common.cuh - shared host/device helpers for libhdp_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <atomic>
#include <stdint.h>
#include <stddef.h>

#include "hdp_b200.h"

namespace hdp {

// Number of kernels this library has launched (bench.py reports it as gpu_launches).
extern std::atomic<int64_t> g_launch_count;

inline int cuda_status(cudaError_t e) { return e == cudaSuccess ? HDP_B200_OK : (int)e; }

#define HDP_CUDA_TRY(expr)                                   \
    do {                                                     \
        cudaError_t _e = (expr);                             \
        if (_e != cudaSuccess) return (int)_e;               \
    } while (0)

// After every launch: count it and surface launch-configuration errors without synchronising.
#define HDP_LAUNCH_CHECK()                                   \
    do {                                                     \
        ::hdp::g_launch_count.fetch_add(1, std::memory_order_relaxed);                             \
        cudaError_t _e = cudaGetLastError();                 \
        if (_e != cudaSuccess) return (int)_e;               \
    } while (0)

// Optional per-kernel CUDA-event timing (hdp_b200_timing_enable / hdp_b200_timing_read).
enum KernelId { kNormalize = 1, kThrGeneric = 2, kHotWords = 3, kScan = 4, kUnpackMask = 5, kThrSeg = 6, kThrRanked = 7, kMeasure = 8, kThrCand = 9, kThrNet = 10, kSeam = 11, kIntensity = 12, kHotPair = 13 };
struct KernelTimer {
    bool on;
    cudaStream_t st;
    int id;
    cudaEvent_t start, stop;
    KernelTimer(int id, cudaStream_t st);
    ~KernelTimer();
};

constexpr size_t kAlign = 256;
inline size_t align_up(size_t v, size_t a = kAlign) { return (v + a - 1) / a * a; }

// Bump allocator over the caller-provided workspace.
struct Carver {
    char *base;
    size_t size;
    size_t off = 0;
    Carver(void *p, size_t n) : base((char *)p), size(n) {}
    template <typename T>
    T *take(size_t count) {
        size_t bytes = align_up(count * sizeof(T));
        T *r = (T *)(base ? base + off : nullptr);
        off += bytes;
        return r;
    }
    bool ok() const { return off <= size; }
};

#ifdef __CUDACC__
// 32-bit shared-state-space accesses: no generic -> shared conversion in front of every access
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ float lds_f32(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) { uint16_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_u16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory"); }
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void reds_or(uint32_t a, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t atoms_add(uint32_t a, uint32_t v) { uint32_t o; asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory"); return o; }
__device__ __forceinline__ uint4 lds_v4(uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory"); return v; }
#endif

#ifdef __CUDACC__
// hdp.measure's unit conversions (reference hdp/measure.py:10-41) as the kernels apply them to every sample they load
// (`input_unit` of the C ABI): 0 = already Celsius, 1 = Kelvin (temp -= 273.15), 2 = Fahrenheit ((temp - 32) / 1.8); float32
// arithmetic with separately rounded operations, bit-identical to the reference's NumPy float32 array arithmetic.
__device__ __forceinline__ float to_celsius_f(float v, int unit)
{
    if (unit == 1) return __fsub_rn(v, 273.15f);
    if (unit == 2) return __fdiv_rn(__fsub_rn(v, 32.0f), 1.8f);
    return v;
}
#endif
// Dense [n] float32 -> Celsius, out of place or in place (measure.cu).
int to_celsius_launch(const float *src, int64_t n, int unit, float *dst, cudaStream_t st);

// Copies the strided measure array into a time-major, cell-contiguous [T, C] buffer.
int normalize_layout(const float *src, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c, float *dst, cudaStream_t st);

// The whole of hdp_b200_thresholds (threshold.cu).  `carve_cells` sizes the workspace layout (>= C; the host pipeline passes its
// chunk capacity so that every chunk sees the tables at the same place) and `tables_resident` skips the table uploads when the
// previous call on this workspace and stream used identical tables.
int thresholds_launch(const float *d_temps, int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                      const int32_t *h_time_index, const int32_t *h_win_rows, int n_doy, int n_y, int W,
                      const double *h_q, int P, double *d_out,
                      void *d_workspace, size_t workspace_bytes, void *stream, int64_t carve_cells, bool tables_resident, int input_unit);

// One measure of a metric pass: samples [T, C] (day t of cell c at x[t * ld_t + c * ld_c]) and their thresholds [C, n_doy, P].
// A pass takes one or two; with two (hdp_b200_compound) a day counts only where both measures pass their own thresholds, and both
// threshold tables have the same n_doy and P.
struct Measure {
    const float *x;
    int64_t ld_t, ld_c;
    const double *thr;
};

// The whole of hdp_b200_metrics, hdp_b200_intensity and hdp_b200_compound (metric.cu) over n_measures (1 or 2) measures:
// k_hot_words (k_hot_pair for two), then k_scan on its hot words when d_out is given (u16 [4, P, D, Y, C], [6, ...] with HWO and
// HWE for HDP_B200_ONSET) and k_intensity when d_int is given (f32 [n_measures, 3, P, D, Y, C], one block per measure).
// carve_cells / tables_resident as above; input_unit = unit code, OR-ed with HDP_B200_COLD for the cold-spell pass and with
// HDP_B200_ONSET for the onset planes.
int metric_pass(const Measure *ms, int n_measures, int64_t C, int64_t T, int n_doy, int P, const int32_t *h_doy_map,
                const int32_t *h_defs, int D,
                const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                const uint8_t *d_is_south, uint16_t *d_out, float *d_int,
                void *d_workspace, size_t workspace_bytes, void *stream, int64_t carve_cells, bool tables_resident, int input_unit);

}  // namespace hdp
