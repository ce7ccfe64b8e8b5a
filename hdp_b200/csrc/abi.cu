// abi.cu - library-level entry points and the layout-normalising copy.
#include <atomic>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace hdp {

std::atomic<int64_t> g_launch_count{0};

// ---- per-kernel timing: event pairs recorded on the launching stream, read back on request ----
struct TimedLaunch { int id; cudaEvent_t start, stop; };
static std::atomic<bool> g_timing{false};
static std::vector<TimedLaunch> g_timed;
static std::mutex g_timed_mu;

// The timer owns its two events until the launch is bracketed; only complete pairs enter the list that
// hdp_b200_timing_read drains (a concurrent read can never see, or invalidate, a half-recorded launch).
KernelTimer::KernelTimer(int id_, cudaStream_t s) : on(g_timing.load(std::memory_order_relaxed)), st(s), id(id_), start(nullptr), stop(nullptr)
{
    if (!on) return;
    if (cudaEventCreate(&start) != cudaSuccess) { on = false; return; }
    if (cudaEventCreate(&stop) != cudaSuccess) { cudaEventDestroy(start); on = false; return; }
    cudaEventRecord(start, st);
}

KernelTimer::~KernelTimer()
{
    if (!on) return;
    cudaEventRecord(stop, st);
    std::lock_guard<std::mutex> lk(g_timed_mu);
    g_timed.push_back(TimedLaunch{id, start, stop});
}

// [C, T] (time-contiguous, ld_t == 1) -> [T, C]: 32x32 tiles through shared memory so that both the
// reads (along t) and the writes (along c) are coalesced.
__global__ void __launch_bounds__(256) k_transpose_ct(const float *__restrict__ src, int64_t C, int64_t T, int64_t ld_c,
                                                      float *__restrict__ dst)
{
    __shared__ float tile[32][33];
    const int64_t t0 = (int64_t)blockIdx.x * 32, c0 = (int64_t)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int64_t c = c0 + ty + 8 * i, t = t0 + tx;
        if (c < C && t < T) tile[ty + 8 * i][tx] = src[c * ld_c + t];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int64_t t = t0 + ty + 8 * i, c = c0 + tx;
        if (c < C && t < T) dst[t * C + c] = tile[tx][ty + 8 * i];
    }
}

// Any other stride pair: plain gather (correct, not fast; documented as the slow layout).
__global__ void __launch_bounds__(256) k_gather_strided(const float *__restrict__ src, int64_t C, int64_t T, int64_t ld_t,
                                                        int64_t ld_c, float *__restrict__ dst)
{
    int64_t n = C * T;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t t = i / C, c = i - t * C;
        dst[i] = src[t * ld_t + c * ld_c];
    }
}

int normalize_layout(const float *src, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c, float *dst, cudaStream_t st)
{
    if (C == 0 || T == 0) return HDP_B200_OK;
    KernelTimer timer(kNormalize, st);
    if (ld_t == 1 && (T + 31) / 32 < 2147483647LL && (C + 31) / 32 <= 65535) {
        dim3 grid((unsigned)((T + 31) / 32), (unsigned)((C + 31) / 32));
        k_transpose_ct<<<grid, 256, 0, st>>>(src, C, T, ld_c, dst);
    } else {
        int64_t blocks = (C * T + 255) / 256;
        if (blocks > 148 * 64) blocks = 148 * 64;
        k_gather_strided<<<(unsigned)blocks, 256, 0, st>>>(src, C, T, ld_t, ld_c, dst);
    }
    HDP_LAUNCH_CHECK();
    return HDP_B200_OK;
}

}  // namespace hdp

extern "C" {

int hdp_b200_abi_version(void) { return HDP_B200_ABI_VERSION; }

int64_t hdp_b200_launch_count(void) { return hdp::g_launch_count.load(std::memory_order_relaxed); }

void hdp_b200_timing_enable(int on)
{
    hdp::g_timing.store(on != 0);
}

int hdp_b200_timing_read(int *ids, float *ms, int cap)
{
    std::vector<hdp::TimedLaunch> done;
    {
        std::lock_guard<std::mutex> lk(hdp::g_timed_mu);
        done.swap(hdp::g_timed);
    }
    int n = 0;
    for (auto &t : done) {
        float v = -1.0f;
        if (cudaEventSynchronize(t.stop) == cudaSuccess) cudaEventElapsedTime(&v, t.start, t.stop);
        if (n < cap) { if (ids) ids[n] = t.id; if (ms) ms[n] = v; n++; }
        cudaEventDestroy(t.start);
        cudaEventDestroy(t.stop);
    }
    return n;
}

const char *hdp_b200_strerror(int code)
{
    switch (code) {
    case HDP_B200_OK: return "ok";
    case HDP_B200_ERR_INVALID:
        return "invalid argument (null pointer, negative size, quantile outside [0,1] or NaN, table entry out of range)";
    case HDP_B200_ERR_UNSUPPORTED:
        return "unsupported shape (more than 32 percentiles or definitions, a window of more than 32768 samples, "
               "a season longer than 65535 days, or - for the intensity metrics - two overlapping non-empty seasons in one "
               "hemisphere's table)";
    case HDP_B200_ERR_WORKSPACE: return "workspace missing or smaller than *_workspace_bytes()";
    case HDP_B200_ERR_NO_DEVICE: return "no CUDA device available";
    case HDP_B200_ERR_NOMEM: return "host allocation failed";
    default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown hdp_b200 error";
}

int hdp_b200_device_info(int *sm_count, int *cc_major, int *cc_minor)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return HDP_B200_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        cudaGetLastError();
        return HDP_B200_ERR_NO_DEVICE;
    }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return HDP_B200_OK;
}

}  // extern "C"
