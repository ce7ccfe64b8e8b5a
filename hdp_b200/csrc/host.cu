// host.cu - the *_host entry points: the same two paths with HOST buffers.
//
// Cells are independent in both paths (the reference parallelises over spatial Dask blocks,
// hdp/threshold.py:161, hdp/metric.py:444), so the host variants cut the cell axis into chunks of a few thousand
// cells and run them through a three-stage pipeline on three streams:
//
//     s_in :  H2D copy of chunk i+1 (samples, thresholds, hemisphere flags)
//     s_k  :  kernels of chunk i
//     s_out:  D2H copy of the results of chunk i-1
//
// with kSlots input and output buffers handed from stage to stage by events, so both PCIe directions and the SMs are
// busy at the same time and the call runs at the rate of its slowest stage (on B200 + PCIe Gen5: the H2D copy).
// Index tables are uploaded with the first chunk only and stay in the workspace (thresholds_launch / metric_pass
// `tables_resident`), so nothing blocks the host between chunks and the whole call is enqueued ahead of the GPU.
// Streams, events and device buffers live in a per-device context that is kept between calls (grown on demand;
// hdp_b200_host_release frees it): cudaMalloc / cudaFree of GB-sized buffers would otherwise cost as much as the copies.
// Pinned host buffers get the full PCIe rate.  PAGEABLE ones (what a NumPy caller has) cannot be read by the copy engines:
// the driver would stage them through one thread at ~11 GB/s, so they go through rings of pinned 32 MB blocks instead, filled
// (H2D) / emptied (D2H) by a small pool of worker threads while the engines move the previous blocks.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace hdp {

constexpr int kSlots = 3;
constexpr int kMaxDevices = 64;

struct DeviceBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {                      // grow-only
        if (bytes <= cap) return HDP_B200_OK;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        HDP_CUDA_TRY(cudaMalloc(&p, bytes));
        cap = bytes;
        return HDP_B200_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// ---- worker threads: parallel row copies between pageable memory and the pinned rings ----
class CopyPool {
public:
    static CopyPool &get() { static CopyPool *p = new CopyPool; return *p; }     // (never destroyed: no thread teardown at exit)
    // copies `rows` rows of `width` bytes (dst / src pitches in bytes), split over the pool; returns when done
    void copy2d(char *dst, size_t dpitch, const char *src, size_t spitch, size_t width, size_t rows) {
        if (rows == 0 || width == 0) return;
        if (rows == 1 && width >= ((size_t)4 << 20)) {                             // one long row: cut it into 1 MB pieces
            const size_t piece = (size_t)1 << 20, n = width / piece;
            copy2d(dst, piece, src, piece, piece, n);
            std::memcpy(dst + n * piece, src + n * piece, width - n * piece);
            return;
        }
        const int parts = (int)std::min<size_t>((size_t)n_threads_, std::max<size_t>(1, (rows * width) >> 20));   // >= 1 MB per part
        auto part = [=](int k) {
            const size_t r0 = rows * k / parts, r1 = rows * (k + 1) / parts;
            if (dpitch == width && spitch == width) { std::memcpy(dst + r0 * width, src + r0 * width, (r1 - r0) * width); return; }
            for (size_t r = r0; r < r1; r++) std::memcpy(dst + r * dpitch, src + r * spitch, width);
        };
        if (parts == 1) { part(0); return; }
        std::lock_guard<std::mutex> one_call(call_mu_);                             // one job at a time
        Job job;
        job.fn = part; job.parts = parts; job.next.store(0); job.active = 0;
        {
            std::lock_guard<std::mutex> lk(mu_);
            cur_ = &job;
            gen_++;
        }
        cv_.notify_all();
        for (;;) { const int k = job.next.fetch_add(1); if (k >= parts) break; part(k); }   // the caller works too
        std::unique_lock<std::mutex> lk(mu_);
        cur_ = nullptr;                                                             // late wakers find nothing
        done_.wait(lk, [&] { return job.active == 0; });                            // (a part is finished before its worker leaves)
    }
private:
    struct Job { std::function<void(int)> fn; int parts; std::atomic<int> next; int active; };
    CopyPool() {
        int n = 0;
        if (const char *e = std::getenv("HDP_B200_HOST_THREADS")) n = std::atoi(e);
        if (n <= 0) n = (int)std::min(8u, std::max(1u, std::thread::hardware_concurrency() / 2));
        n_threads_ = n;
        for (int i = 1; i < n; i++) std::thread([this] { run(); }).detach();
    }
    void run() {
        uint64_t seen = 0;
        for (;;) {
            Job *j;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                j = cur_;
                if (!j) continue;
                j->active++;
            }
            for (;;) { const int k = j->next.fetch_add(1); if (k >= j->parts) break; j->fn(k); }
            std::lock_guard<std::mutex> lk(mu_);
            if (--j->active == 0) done_.notify_all();
        }
    }
    int n_threads_ = 1;
    std::mutex mu_, call_mu_;
    std::condition_variable cv_, done_;
    Job *cur_ = nullptr;
    uint64_t gen_ = 0;
};

constexpr int kRingBlocks = 6;
constexpr size_t kRingBlockBytes = (size_t)32 << 20;

struct PinnedRing {
    char *blk[kRingBlocks] = {};
    cudaEvent_t ev[kRingBlocks] = {};
    int next = 0;
    int init() {
        for (int i = 0; i < kRingBlocks; i++) {
            if (!blk[i]) HDP_CUDA_TRY(cudaHostAlloc((void **)&blk[i], kRingBlockBytes, cudaHostAllocDefault));
            if (!ev[i]) HDP_CUDA_TRY(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
        }
        return HDP_B200_OK;
    }
    void release() {
        for (int i = 0; i < kRingBlocks; i++) {
            if (blk[i]) cudaFreeHost(blk[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
            blk[i] = nullptr; ev[i] = nullptr;
        }
    }
};

struct PendingOut { int slot; char *dst; size_t dpitch, width, rows; };

static bool is_pageable(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

struct HostCtx {
    std::mutex mu;                                   // one host call per device at a time
    bool ready = false;
    cudaStream_t s_in = nullptr, s_k = nullptr, s_out = nullptr;
    cudaEvent_t in_ready[kSlots] = {}, k_done[kSlots] = {}, out_done[kSlots] = {};
    DeviceBuf x[kSlots], aux[kSlots], south[kSlots], out[kSlots], out_f[kSlots], ws;
    PinnedRing ring_in, ring_out;                    // staging for pageable sources / destinations (allocated on first use)
    std::deque<PendingOut> pending;                  // D2H blocks on their way through ring_out

    // host -> device copy of `rows` rows of `width` bytes; pageable sources are staged through ring_in by the copy pool
    int h2d(char *dst, size_t dpitch, const char *src, size_t spitch, size_t width, size_t rows, bool pageable, cudaStream_t st) {
        if (rows == 0 || width == 0) return HDP_B200_OK;
        if (!pageable) {
            if (rows == 1) HDP_CUDA_TRY(cudaMemcpyAsync(dst, src, width, cudaMemcpyHostToDevice, st));
            else HDP_CUDA_TRY(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, cudaMemcpyHostToDevice, st));
            return HDP_B200_OK;
        }
        if (rows == 1 && width > kRingBlockBytes) {                                // one long row: block by block
            for (size_t o = 0; o < width; o += kRingBlockBytes) {
                const int rc = h2d(dst + o, 0, src + o, 0, std::min(kRingBlockBytes, width - o), 1, true, st);
                if (rc) return rc;
            }
            return HDP_B200_OK;
        }
        if (width > kRingBlockBytes) return HDP_B200_ERR_UNSUPPORTED;
        int rc = ring_in.init();
        if (rc) return rc;
        const size_t per = std::max<size_t>(1, kRingBlockBytes / width);
        for (size_t r0 = 0; r0 < rows; r0 += per) {
            const size_t nr = std::min(per, rows - r0);
            const int slot = ring_in.next++ % kRingBlocks;
            HDP_CUDA_TRY(cudaEventSynchronize(ring_in.ev[slot]));                  // the block's previous copy has left
            CopyPool::get().copy2d(ring_in.blk[slot], width, src + r0 * spitch, spitch, width, nr);
            if (nr == 1) HDP_CUDA_TRY(cudaMemcpyAsync(dst + r0 * dpitch, ring_in.blk[slot], width, cudaMemcpyHostToDevice, st));
            else HDP_CUDA_TRY(cudaMemcpy2DAsync(dst + r0 * dpitch, dpitch, ring_in.blk[slot], width, width, nr, cudaMemcpyHostToDevice, st));
            HDP_CUDA_TRY(cudaEventRecord(ring_in.ev[slot], st));
        }
        return HDP_B200_OK;
    }
    // finishes D2H blocks (waits for the copy engine, then the pool moves the block to the caller's memory) until at most
    // `keep` are still on their way
    int finish_out(size_t keep) {
        while (pending.size() > keep) {
            const PendingOut p = pending.front();
            pending.pop_front();
            HDP_CUDA_TRY(cudaEventSynchronize(ring_out.ev[p.slot]));
            CopyPool::get().copy2d(p.dst, p.dpitch, ring_out.blk[p.slot], p.width, p.width, p.rows);
        }
        return HDP_B200_OK;
    }
    // device -> host copy; pageable destinations are reached through ring_out (completed by finish_out)
    int d2h(char *dst, size_t dpitch, const char *src, size_t spitch, size_t width, size_t rows, bool pageable, cudaStream_t st) {
        if (rows == 0 || width == 0) return HDP_B200_OK;
        if (!pageable) {
            if (rows == 1) HDP_CUDA_TRY(cudaMemcpyAsync(dst, src, width, cudaMemcpyDeviceToHost, st));
            else HDP_CUDA_TRY(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, cudaMemcpyDeviceToHost, st));
            return HDP_B200_OK;
        }
        if (rows == 1 && width > kRingBlockBytes) {
            for (size_t o = 0; o < width; o += kRingBlockBytes) {
                const int rc = d2h(dst + o, 0, src + o, 0, std::min(kRingBlockBytes, width - o), 1, true, st);
                if (rc) return rc;
            }
            return HDP_B200_OK;
        }
        if (width > kRingBlockBytes) return HDP_B200_ERR_UNSUPPORTED;
        int rc = ring_out.init();
        if (rc) return rc;
        const size_t per = std::max<size_t>(1, kRingBlockBytes / width);
        for (size_t r0 = 0; r0 < rows; r0 += per) {
            const size_t nr = std::min(per, rows - r0);
            if ((rc = finish_out(kRingBlocks - 1))) return rc;                     // a free block
            const int slot = ring_out.next++ % kRingBlocks;
            if (nr == 1) HDP_CUDA_TRY(cudaMemcpyAsync(ring_out.blk[slot], src + r0 * spitch, width, cudaMemcpyDeviceToHost, st));
            else HDP_CUDA_TRY(cudaMemcpy2DAsync(ring_out.blk[slot], width, src + r0 * spitch, spitch, width, nr, cudaMemcpyDeviceToHost, st));
            HDP_CUDA_TRY(cudaEventRecord(ring_out.ev[slot], st));
            pending.push_back({slot, dst + r0 * dpitch, dpitch, width, nr});
        }
        return HDP_B200_OK;
    }

    int init() {
        if (ready) return HDP_B200_OK;
        HDP_CUDA_TRY(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
        HDP_CUDA_TRY(cudaStreamCreateWithFlags(&s_k, cudaStreamNonBlocking));
        HDP_CUDA_TRY(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
        for (int i = 0; i < kSlots; i++) {
            HDP_CUDA_TRY(cudaEventCreateWithFlags(&in_ready[i], cudaEventDisableTiming));
            HDP_CUDA_TRY(cudaEventCreateWithFlags(&k_done[i], cudaEventDisableTiming));
            HDP_CUDA_TRY(cudaEventCreateWithFlags(&out_done[i], cudaEventDisableTiming));
        }
        ready = true;
        return HDP_B200_OK;
    }
    // waits for everything this context has enqueued; returns the first error seen
    int drain() {
        int rc = finish_out(0);
        pending.clear();
        for (cudaStream_t s : {s_in, s_k, s_out}) {
            const cudaError_t e = cudaStreamSynchronize(s);
            if (e != cudaSuccess && rc == HDP_B200_OK) rc = (int)e;
        }
        return rc;
    }
    void release() {
        if (ready) {
            drain();
            cudaStreamDestroy(s_in); cudaStreamDestroy(s_k); cudaStreamDestroy(s_out);
            for (int i = 0; i < kSlots; i++) { cudaEventDestroy(in_ready[i]); cudaEventDestroy(k_done[i]); cudaEventDestroy(out_done[i]); }
            ready = false;
        }
        for (int i = 0; i < kSlots; i++) { x[i].release(); aux[i].release(); south[i].release(); out[i].release(); out_f[i].release(); }
        ws.release();
        ring_in.release(); ring_out.release();
    }
};

static HostCtx g_ctx[kMaxDevices];

static int current_ctx(HostCtx **ctx)
{
    int dev = 0;
    HDP_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) return HDP_B200_ERR_NO_DEVICE;
    *ctx = &g_ctx[dev];
    return HDP_B200_OK;
}

// Enqueues the copy of cells [c0, c0+nc) of a host measure array into a dense device buffer and reports the strides
// of the device copy.  Supported host layouts: cell-contiguous (ld_c == 1) and time-contiguous (ld_t == 1).
static int upload_cells(HostCtx *ctx, const float *h, bool pageable, int64_t T, int64_t ld_t, int64_t ld_c, int64_t c0, int64_t nc,
                        float *d, int64_t *d_ld_t, int64_t *d_ld_c, cudaStream_t st)
{
    if (ld_c == 1) {
        *d_ld_t = nc; *d_ld_c = 1;
        return ctx->h2d((char *)d, nc * sizeof(float), (const char *)(h + c0), ld_t * sizeof(float), nc * sizeof(float), T, pageable, st);
    }
    if (ld_t == 1) {
        *d_ld_t = 1; *d_ld_c = T;
        return ctx->h2d((char *)d, T * sizeof(float), (const char *)(h + c0 * ld_c), ld_c * sizeof(float), T * sizeof(float), nc, pageable, st);
    }
    return HDP_B200_ERR_UNSUPPORTED;
}

// Cells per chunk: small enough that the pipeline's fill and drain (one chunk each) stay near one percent of a CMIP-sized
// call, large enough that copy rows stay >= 2 KB and that a chunk's kernels (a k_scan launch takes >= 1.5 ms however few
// cells it has: every warp walks the whole series) stay shorter than its H2D copy; a multiple of 32 cells (warp = 32
// cells).  Measured on B200 / PCIe Gen5 (tools/e2e_breakdown.py): thresholds 1 024 .. 4 096 cells per chunk within 2 %,
// metrics 1 024 .. 4 096 within 2 %, 512 cells 17 % slower (kernel-bound).
static int64_t pick_chunk(int64_t C, size_t in_bytes_per_cell, size_t target_bytes)
{
    if (const char *e = std::getenv("HDP_B200_HOST_CHUNK_CELLS")) {
        const int64_t v = std::atoll(e);
        if (v > 0) return std::min<int64_t>(std::max<int64_t>(32, v / 32 * 32), std::max<int64_t>(C, 1));
    }
    int64_t chunk = (int64_t)target_bytes / (int64_t)std::max<size_t>(in_bytes_per_cell, 1);
    chunk = std::max<int64_t>(1024, chunk / 32 * 32);
    if (C > 4096) chunk = std::min(chunk, ((C + 3) / 4 + 31) / 32 * 32);       // at least 4 chunks once there is work to overlap
    return std::min(chunk, std::max<int64_t>(C, 1));
}

}  // namespace hdp

using namespace hdp;

// error inside the chunk loop: let the enqueued work finish (it reads and writes the caller's buffers), then report
#define HDP_HOST_TRY(expr)                                   \
    do {                                                     \
        const int _rc = (expr);                              \
        if (_rc != HDP_B200_OK) { ctx->drain(); return _rc; }\
    } while (0)
#define HDP_HOST_CUDA(expr) HDP_HOST_TRY(cuda_status(expr))

// hdp_b200_metrics_host and hdp_b200_intensity_host: metric_pass chunk by chunk; the u16 planes (h_out) and the f32 planes (h_int),
// whichever are given, go back to the host.
static int metric_pass_host(const float *h_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                            const double *h_thr, const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                            const int32_t *h_defs, int D,
                            const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                            const uint8_t *h_is_south, float *h_int, uint16_t *h_out, int input_unit)
{
    if (C < 0 || T <= 0 || n_doy <= 0 || P <= 0 || D <= 0 || Y < 0 || !h_doy_map) return HDP_B200_ERR_INVALID;
    if (C == 0 || Y == 0) return HDP_B200_OK;
    if (!h_measure || (!h_thr && !d_thr)) return HDP_B200_ERR_INVALID;
    if (ld_t <= 0 || ld_c <= 0) return HDP_B200_ERR_INVALID;
    if (ld_c != 1 && ld_t != 1) return HDP_B200_ERR_UNSUPPORTED;
    HostCtx *ctx = nullptr;
    int rc = current_ctx(&ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if ((rc = ctx->init())) return rc;

    const size_t thr_per_cell = (size_t)n_doy * P * sizeof(double);
    const size_t rows = (size_t)4 * P * D * Y;                                 // output rows of C cells each
    const size_t rows_f = (size_t)3 * P * D * Y;
    const int64_t chunk = pick_chunk(C, (size_t)T * sizeof(float) + thr_per_cell, (size_t)320 << 20);
    const int64_t dl_t = ld_c == 1 ? chunk : 1, dl_c = ld_c == 1 ? 1 : T;
    const size_t ws_bytes = h_int ? hdp_b200_intensity_workspace_bytes(chunk, T, dl_t, dl_c, n_doy, P, D, Y, h_doy_map)
                                  : hdp_b200_metrics_workspace_bytes(chunk, T, dl_t, dl_c, n_doy, P, D, Y, h_doy_map);
    if ((rc = ctx->ws.reserve(ws_bytes))) return rc;
    for (int i = 0; i < kSlots; i++) {
        if ((rc = ctx->x[i].reserve((size_t)chunk * T * sizeof(float)))) return rc;
        if (!d_thr && (rc = ctx->aux[i].reserve((size_t)chunk * thr_per_cell))) return rc;
        if ((rc = ctx->south[i].reserve((size_t)chunk))) return rc;
        if (h_out && (rc = ctx->out[i].reserve(rows * chunk * sizeof(uint16_t)))) return rc;
        if (h_int && (rc = ctx->out_f[i].reserve(rows_f * chunk * sizeof(float)))) return rc;
    }
    const bool page_x = is_pageable(h_measure), page_thr = !d_thr && is_pageable(h_thr), page_out = h_out && is_pageable(h_out);
    const bool page_int = h_int && is_pageable(h_int);
    const bool page_south = h_is_south && is_pageable(h_is_south);
    int64_t i = 0;
    for (int64_t c0 = 0; c0 < C; c0 += chunk, i++) {
        const int slot = (int)(i % kSlots);
        const int64_t nc = std::min(chunk, C - c0);
        int64_t a, b;
        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_in, ctx->k_done[slot], 0));
        HDP_HOST_TRY(upload_cells(ctx, h_measure, page_x, T, ld_t, ld_c, c0, nc, (float *)ctx->x[slot].p, &a, &b, ctx->s_in));
        if (!d_thr)                                                            // device-resident thresholds never cross PCIe again
            HDP_HOST_TRY(ctx->h2d((char *)ctx->aux[slot].p, 0, (const char *)(h_thr + (size_t)c0 * n_doy * P), 0, (size_t)nc * thr_per_cell, 1,
                                  page_thr, ctx->s_in));
        if (h_is_south)
            HDP_HOST_TRY(ctx->h2d((char *)ctx->south[slot].p, 0, (const char *)(h_is_south + c0), 0, (size_t)nc, 1, page_south, ctx->s_in));
        HDP_HOST_CUDA(cudaEventRecord(ctx->in_ready[slot], ctx->s_in));

        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_k, ctx->in_ready[slot], 0));
        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_k, ctx->out_done[slot], 0));
        const double *thr_chunk = d_thr ? d_thr + (size_t)c0 * n_doy * P : (const double *)ctx->aux[slot].p;
        const uint8_t *south_chunk = h_is_south ? (const uint8_t *)ctx->south[slot].p : nullptr;
        HDP_HOST_TRY(metric_pass((const float *)ctx->x[slot].p, nc, T, a, b, thr_chunk, n_doy, P, h_doy_map, h_defs, D,
                                 h_season_north, h_season_south, Y, south_chunk, h_out ? (uint16_t *)ctx->out[slot].p : nullptr,
                                 h_int ? (float *)ctx->out_f[slot].p : nullptr, ctx->ws.p, ws_bytes, ctx->s_k, chunk, i > 0, input_unit));
        HDP_HOST_CUDA(cudaEventRecord(ctx->k_done[slot], ctx->s_k));

        // device chunk is [rows, nc]; host array is [rows, C]
        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_out, ctx->k_done[slot], 0));
        if (h_out)
            HDP_HOST_TRY(ctx->d2h((char *)(h_out + c0), (size_t)C * sizeof(uint16_t), (const char *)ctx->out[slot].p, (size_t)nc * sizeof(uint16_t),
                                  (size_t)nc * sizeof(uint16_t), rows, page_out, ctx->s_out));
        if (h_int)
            HDP_HOST_TRY(ctx->d2h((char *)(h_int + c0), (size_t)C * sizeof(float), (const char *)ctx->out_f[slot].p, (size_t)nc * sizeof(float),
                                  (size_t)nc * sizeof(float), rows_f, page_int, ctx->s_out));
        HDP_HOST_CUDA(cudaEventRecord(ctx->out_done[slot], ctx->s_out));
    }
    return ctx->drain();
}

extern "C" {

void hdp_b200_host_release(void)
{
    for (HostCtx &c : g_ctx) {
        std::lock_guard<std::mutex> lock(c.mu);
        if (c.ready || c.ws.p || c.x[0].p) c.release();
    }
}

int hdp_b200_thresholds_host(const float *h_temps, int64_t C, int64_t T_b, int64_t ld_t, int64_t ld_c,
                             const int32_t *h_time_index, const int32_t *h_win_rows, int n_doy, int n_y, int W,
                             const double *h_q, int P, double *h_out, double *d_keep, int input_unit)
{
    if (C < 0 || T_b <= 0 || n_doy <= 0 || n_y <= 0 || W <= 0 || P <= 0) return HDP_B200_ERR_INVALID;
    if (C == 0) return HDP_B200_OK;
    if (!h_temps || !h_out) return HDP_B200_ERR_INVALID;
    if (ld_t <= 0 || ld_c <= 0) return HDP_B200_ERR_INVALID;              // pitches become size_t below: no reversed views
    if (ld_c != 1 && ld_t != 1) return HDP_B200_ERR_UNSUPPORTED;
    HostCtx *ctx = nullptr;
    int rc = current_ctx(&ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if ((rc = ctx->init())) return rc;

    const size_t out_per_cell = (size_t)n_doy * P * sizeof(double);
    const int64_t chunk = pick_chunk(C, (size_t)T_b * sizeof(float), (size_t)64 << 20);
    const int64_t dl_t = ld_c == 1 ? chunk : 1, dl_c = ld_c == 1 ? 1 : T_b;
    const size_t ws_bytes = hdp_b200_thresholds_workspace_bytes(chunk, T_b, dl_t, dl_c, n_doy, n_y, W, P, input_unit);
    if ((rc = ctx->ws.reserve(ws_bytes))) return rc;
    for (int i = 0; i < kSlots; i++) {
        if ((rc = ctx->x[i].reserve((size_t)chunk * T_b * sizeof(float)))) return rc;
        if (!d_keep && (rc = ctx->out[i].reserve((size_t)chunk * out_per_cell))) return rc;
    }
    const bool page_in = is_pageable(h_temps), page_out = is_pageable(h_out);
    int64_t i = 0;
    for (int64_t c0 = 0; c0 < C; c0 += chunk, i++) {
        const int slot = (int)(i % kSlots);
        const int64_t nc = std::min(chunk, C - c0);
        int64_t a, b;
        // stage 1: samples of this chunk (the slot's previous user must have been consumed by its kernels)
        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_in, ctx->k_done[slot], 0));
        HDP_HOST_TRY(upload_cells(ctx, h_temps, page_in, T_b, ld_t, ld_c, c0, nc, (float *)ctx->x[slot].p, &a, &b, ctx->s_in));
        HDP_HOST_CUDA(cudaEventRecord(ctx->in_ready[slot], ctx->s_in));
        // stage 2: kernels (the slot's previous results must have left for the host)
        // with d_keep the kernels write the chunk straight into its place in the caller's device-resident copy (which then feeds
        // hdp_b200_metrics_host without coming back over PCIe) and the D2H copy reads it from there: no slot to wait for
        double *d_chunk_out = d_keep ? d_keep + (size_t)c0 * n_doy * P : (double *)ctx->out[slot].p;
        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_k, ctx->in_ready[slot], 0));
        if (!d_keep) HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_k, ctx->out_done[slot], 0));
        HDP_HOST_TRY(thresholds_launch((const float *)ctx->x[slot].p, nc, T_b, a, b, h_time_index, h_win_rows, n_doy, n_y, W, h_q, P,
                                       d_chunk_out, ctx->ws.p, ws_bytes, ctx->s_k, chunk, i > 0, input_unit));
        HDP_HOST_CUDA(cudaEventRecord(ctx->k_done[slot], ctx->s_k));
        // stage 3: results
        HDP_HOST_CUDA(cudaStreamWaitEvent(ctx->s_out, ctx->k_done[slot], 0));
        HDP_HOST_TRY(ctx->d2h((char *)(h_out + (size_t)c0 * n_doy * P), 0, (const char *)d_chunk_out, 0, (size_t)nc * out_per_cell, 1,
                              page_out, ctx->s_out));
        HDP_HOST_CUDA(cudaEventRecord(ctx->out_done[slot], ctx->s_out));
    }
    return ctx->drain();
}

int hdp_b200_metrics_host(const float *h_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                          const double *h_thr, const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                          const int32_t *h_defs, int D,
                          const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                          const uint8_t *h_is_south, uint16_t *h_out, int input_unit)
{
    if (!h_out && C > 0 && Y > 0) return HDP_B200_ERR_INVALID;
    return metric_pass_host(h_measure, C, T, ld_t, ld_c, h_thr, d_thr, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y,
                            h_is_south, nullptr, h_out, input_unit);
}

int hdp_b200_intensity_host(const float *h_measure, int64_t C, int64_t T, int64_t ld_t, int64_t ld_c,
                            const double *h_thr, const double *d_thr, int n_doy, int P, const int32_t *h_doy_map,
                            const int32_t *h_defs, int D,
                            const int32_t *h_season_north, const int32_t *h_season_south, int Y,
                            const uint8_t *h_is_south, float *h_int, uint16_t *h_out, int input_unit)
{
    if (!h_int && C > 0 && Y > 0) return HDP_B200_ERR_INVALID;
    return metric_pass_host(h_measure, C, T, ld_t, ld_c, h_thr, d_thr, n_doy, P, h_doy_map, h_defs, D, h_season_north, h_season_south, Y,
                            h_is_south, h_int, h_out, input_unit);
}

}  // extern "C"
