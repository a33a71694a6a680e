// runtime.cu -- the library's host runtime (declared and described in runtime.h).  Host code only.
#include "runtime.h"

#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

namespace rmb {

thread_local std::string g_err;
std::mutex g_call_mutex;
thread_local int g_upload_share = 1;

void set_err(const char* what, const char* detail)
{
    g_err = what;
    if (detail) { g_err += ": "; g_err += detail; }
}

namespace {

// Device workspace cache: a call needs a few GB of scratch (operand images, candidate buffers); cudaMalloc / cudaFree
// of those cost tens of milliseconds per call and synchronise the device, so released blocks are kept for the next
// call (rmb200_release_workspace() or RMB200_NO_POOL=1 gives them back).
struct PoolEntry { void* p; size_t bytes; int dev; bool in_use; };
std::vector<PoolEntry> g_pool;
std::mutex g_pool_mutex;

bool pool_enabled()
{
    static const bool on = []() { const char* e = std::getenv("RMB200_NO_POOL"); return !(e && e[0] == '1'); }();
    return on;
}

void pool_trim_locked(int dev_only)
{
    for (size_t i = 0; i < g_pool.size();) {
        if (!g_pool[i].in_use && (dev_only < 0 || g_pool[i].dev == dev_only)) {
            cudaFree(g_pool[i].p);
            g_pool[i] = g_pool.back();
            g_pool.pop_back();
        } else i++;
    }
}

}  // namespace

cudaError_t pool_alloc(void** out, size_t bytes)
{
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    if (pool_enabled()) {
        int best = -1;
        for (size_t i = 0; i < g_pool.size(); i++) {
            const PoolEntry& e = g_pool[i];
            if (e.in_use || e.dev != dev || e.bytes < bytes || e.bytes > bytes + bytes / 4 + (1u << 20)) continue;
            if (best < 0 || e.bytes < g_pool[best].bytes) best = (int)i;
        }
        if (best >= 0) { g_pool[best].in_use = true; *out = g_pool[best].p; return cudaSuccess; }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e == cudaErrorMemoryAllocation) {           // give cached blocks back and try once more
        cudaGetLastError();
        pool_trim_locked(dev);
        e = cudaMalloc(out, bytes);
    }
    if (e == cudaSuccess && pool_enabled()) g_pool.push_back(PoolEntry{*out, bytes, dev, true});
    return e;
}

void pool_free(void* p)
{
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    for (auto& e : g_pool)
        if (e.p == p) { e.in_use = false; return; }
    cudaFree(p);
}

namespace {

// ---------------------------------------------------------------- host -> device uploads
// The reference's callers hand over ordinary (pageable) numpy / R memory (wrapper.pyx:208-224).  cudaMemcpy from
// pageable memory goes through the driver's single staging buffer at ~11 GB/s (measured: 62 ms for the 0.67 GB of a
// 151K-user cfg4 call); a PCIe 5 x16 link takes 55 GB/s from pinned memory.  Large pageable sources therefore go through
// our own pipeline: UP_THREADS host threads each copy their share of the rows into pinned bounce buffers (two per
// thread, UP_CHUNK bytes) and queue the DMA from there on their own stream -- the memcpy of one chunk overlaps the DMA
// of the previous one and the threads overlap each other.  Pinned (or registered) sources and small copies take the
// plain cudaMemcpyAsync path.  RMB200_UPLOAD_THREADS=0 switches the pipeline off.
constexpr size_t UP_CHUNK = 8u << 20;
constexpr int UP_MAX_THREADS = 16;
struct UploadLane {
    cudaStream_t st = nullptr;
    void* buf[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};      // recorded behind the DMA that reads buf[i]
    bool recorded[2] = {false, false};           // ... at least once: the buffer may still be in flight from an earlier upload
};
struct UploadPool {
    int dev = -1;
    UploadLane lane[UP_MAX_THREADS];
    cudaEvent_t done[UP_MAX_THREADS] = {};
    cudaEvent_t start = nullptr;
    int lanes = 0;
    bool ok = false;
};
UploadPool g_ups[MAX_DEVICES];   // one per device: calls are serialised by the library's mutex, and inside a multi-GPU call
                                 // every device has its own host thread

int upload_threads()
{
    int v = (int)std::thread::hardware_concurrency() / 2;      // measured on a 16-core box: 60 ms plain, 32 ms with 4 threads, 25 ms with 8
    if (v < 1) v = 1;
    if (const char* e = std::getenv("RMB200_UPLOAD_THREADS")) v = std::atoi(e);
    if (v > 1 && g_upload_share > 1) { v /= g_upload_share; if (v < 1) v = 1; }
    return v < 0 ? 0 : (v > UP_MAX_THREADS ? UP_MAX_THREADS : v);
}

void upload_pool_release(UploadPool& g_up)
{
    if (g_up.dev < 0) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(g_up.dev);
    for (int t = 0; t < UP_MAX_THREADS; t++) {
        UploadLane& L = g_up.lane[t];
        for (int b = 0; b < 2; b++) { if (L.buf[b]) cudaFreeHost(L.buf[b]); if (L.ev[b]) cudaEventDestroy(L.ev[b]); L.buf[b] = nullptr; L.ev[b] = nullptr; L.recorded[b] = false; }
        if (L.st) cudaStreamDestroy(L.st);
        L.st = nullptr;
        if (g_up.done[t]) cudaEventDestroy(g_up.done[t]);
        g_up.done[t] = nullptr;
    }
    if (g_up.start) cudaEventDestroy(g_up.start);
    g_up.start = nullptr;
    g_up.dev = -1; g_up.ok = false; g_up.lanes = 0;
    cudaSetDevice(cur);
}

bool upload_pool_ready(int dev, int nthreads)
{
    if (dev < 0 || dev >= MAX_DEVICES) return false;
    UploadPool& g_up = g_ups[dev];
    if (g_up.ok && g_up.dev == dev && g_up.lanes >= nthreads) return true;
    upload_pool_release(g_up);
    g_up.dev = dev;
    g_up.lanes = nthreads;
    for (int t = 0; t < nthreads; t++) {
        UploadLane& L = g_up.lane[t];
        if (cudaStreamCreateWithFlags(&L.st, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); upload_pool_release(g_up); return false; }
        for (int b = 0; b < 2; b++) {
            if (cudaHostAlloc(&L.buf[b], UP_CHUNK, cudaHostAllocDefault) != cudaSuccess ||
                cudaEventCreateWithFlags(&L.ev[b], cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); upload_pool_release(g_up); return false; }
        }
        if (cudaEventCreateWithFlags(&g_up.done[t], cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); upload_pool_release(g_up); return false; }
    }
    if (cudaEventCreateWithFlags(&g_up.start, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); upload_pool_release(g_up); return false; }
    g_up.ok = true;
    return true;
}

bool host_pointer_is_pageable(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}

// How many lanes copy `bytes` of host memory at `host` to or from the current device (stored in *dev): 0 -- the driver's
// plain copy -- unless the block is large and pageable and the device's lanes are ready for this thread's copy threads.
int lanes_for(const void* host, size_t bytes, int* dev)
{
    const int nt = upload_threads();
    cudaGetDevice(dev);
    size_t min_bytes = 32u << 20;
    if (const char* env = std::getenv("RMB200_UPLOAD_MIN_BYTES")) min_bytes = (size_t)std::atoll(env);      // developer / tests
    if (bytes < min_bytes || bytes == 0 || nt == 0 || !host_pointer_is_pageable(host) || !upload_pool_ready(*dev, nt)) return 0;
    return nt;
}

// Runs body(t, lane t) on nt threads, one per lane of device `dev`, behind what is already queued on `st` (e.g. kernels
// still reading the destination's previous contents); returns the first error.
template <typename Body>
cudaError_t run_lanes(int dev, int nt, cudaStream_t st, Body body)
{
    UploadPool& g_up = g_ups[dev];
    const cudaError_t e = cudaEventRecord(g_up.start, st);
    if (e != cudaSuccess) return e;
    cudaError_t errs[UP_MAX_THREADS];
    std::vector<std::thread> workers;
    for (int t = 0; t < nt; t++) {
        errs[t] = cudaSuccess;
        workers.emplace_back([&, t]() {
            cudaError_t er = cudaSetDevice(dev);
            UploadLane& L = g_up.lane[t];
            if (er == cudaSuccess) er = cudaStreamWaitEvent(L.st, g_up.start, 0);
            if (er == cudaSuccess) er = body(t, L);
            errs[t] = er;
        });
    }
    for (auto& w : workers) w.join();
    for (int t = 0; t < nt; t++) if (errs[t] != cudaSuccess) return errs[t];
    return cudaSuccess;
}

}  // namespace

cudaError_t upload_rows(void* dst, const void* src, size_t src_pitch, size_t row_bytes, size_t rows, cudaStream_t st)
{
    const size_t total = row_bytes * rows;
    // a contiguous source is a byte stream (chunks of UP_CHUNK bytes); a pitched one is cut at row boundaries
    const bool contiguous = (src_pitch == row_bytes) || rows == 1;
    int dev = 0;
    const int nt = (contiguous || row_bytes <= UP_CHUNK) ? lanes_for(src, total, &dev) : 0;
    if (nt == 0) {
        if (src_pitch == row_bytes) return cudaMemcpyAsync(dst, src, total, cudaMemcpyHostToDevice, st);
        return cudaMemcpy2DAsync(dst, row_bytes, src, src_pitch, row_bytes, rows, cudaMemcpyHostToDevice, st);
    }
    const size_t unit = contiguous ? 1 : row_bytes;                              // bytes per indivisible piece
    const size_t units = contiguous ? total : rows;
    const size_t rows_per_chunk = contiguous ? UP_CHUNK : UP_CHUNK / row_bytes;   // pieces per chunk
    const size_t nchunks = (units + rows_per_chunk - 1) / rows_per_chunk;
    cudaError_t e = run_lanes(dev, nt, st, [&](int t, UploadLane& L) {
        cudaError_t er = cudaSuccess;
        int b = 0;
        for (size_t c = (size_t)t; c < nchunks && er == cudaSuccess; c += (size_t)nt, b ^= 1) {
            const size_t r0 = c * rows_per_chunk, nr = (units - r0) < rows_per_chunk ? (units - r0) : rows_per_chunk;
            if (L.recorded[b]) er = cudaEventSynchronize(L.ev[b]);     // the DMA that last read this bounce buffer (this upload's or an earlier one's)
            if (er != cudaSuccess) break;
            const unsigned char* sp = static_cast<const unsigned char*>(src) + r0 * (contiguous ? 1 : src_pitch);
            if (contiguous) std::memcpy(L.buf[b], sp, nr);
            else for (size_t r = 0; r < nr; r++) std::memcpy(static_cast<unsigned char*>(L.buf[b]) + r * row_bytes, sp + r * src_pitch, row_bytes);
            er = cudaMemcpyAsync(static_cast<unsigned char*>(dst) + r0 * unit, L.buf[b], nr * unit, cudaMemcpyHostToDevice, L.st);
            if (er == cudaSuccess) { er = cudaEventRecord(L.ev[b], L.st); L.recorded[b] = true; }
        }
        return er;
    });
    if (e != cudaSuccess) return e;
    // `st` continues once every lane's copies have landed (the bounce buffers are reused only after their own events)
    UploadPool& g_up = g_ups[dev];
    for (int t = 0; t < nt; t++) {
        e = cudaEventRecord(g_up.done[t], g_up.lane[t].st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, g_up.done[t], 0);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

namespace {

// The mirror image of upload_rows for one contiguous block: device memory to ordinary (pageable) host memory through the
// lanes' pinned bounce buffers, every lane alternating between the DMA into one buffer and the memcpy out of the other.  The
// driver's own path stages through one buffer and copies out on one thread (12 GB/s measured); this reaches what the host's
// memory system gives several threads.  Work queued on `st` before the call is waited for; returns when the bytes are in dst.
cudaError_t download_bytes(void* dst, const void* src, size_t total, cudaStream_t st)
{
    int dev = 0;
    const int nt = lanes_for(dst, total, &dev);
    if (nt == 0) {
        const cudaError_t e = cudaMemcpyAsync(dst, src, total, cudaMemcpyDeviceToHost, st);
        return e != cudaSuccess ? e : cudaStreamSynchronize(st);
    }
    const size_t nchunks = (total + UP_CHUNK - 1) / UP_CHUNK;
    return run_lanes(dev, nt, st, [&](int t, UploadLane& L) {
        cudaError_t er = cudaSuccess;
        // (an earlier UPLOAD may still be reading the bounce buffers: its events come first)
        for (int b = 0; b < 2 && er == cudaSuccess; b++) if (L.recorded[b]) er = cudaEventSynchronize(L.ev[b]);
        auto span = [&](size_t c, size_t* off) { *off = c * UP_CHUNK; return (total - *off) < UP_CHUNK ? (total - *off) : UP_CHUNK; };
        auto fetch = [&](size_t c, int b) {
            size_t off; const size_t nb = span(c, &off);
            cudaError_t x = cudaMemcpyAsync(L.buf[b], static_cast<const unsigned char*>(src) + off, nb, cudaMemcpyDeviceToHost, L.st);
            if (x == cudaSuccess) { x = cudaEventRecord(L.ev[b], L.st); L.recorded[b] = true; }
            return x;
        };
        int b = 0;
        if (er == cudaSuccess && (size_t)t < nchunks) er = fetch((size_t)t, 0);
        for (size_t c = (size_t)t; c < nchunks && er == cudaSuccess; c += (size_t)nt, b ^= 1) {
            if (c + (size_t)nt < nchunks) er = fetch(c + (size_t)nt, b ^ 1);       // the next chunk's DMA runs under this chunk's memcpy
            if (er == cudaSuccess) er = cudaEventSynchronize(L.ev[b]);
            if (er != cudaSuccess) break;
            size_t off; const size_t nb = span(c, &off);
            std::memcpy(static_cast<unsigned char*>(dst) + off, L.buf[b], nb);
        }
        return er;
    });
}

}  // namespace

cudaError_t upload_bytes_pageable(void* dst, const void* src, size_t bytes, cudaStream_t st, int share)
{
    std::unique_lock<std::mutex> lk(g_call_mutex, std::try_to_lock);
    if (!lk.owns_lock()) return bytes ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
    g_upload_share = share > 1 ? share : 1;
    const cudaError_t e = bytes ? upload_rows(dst, src, bytes, bytes, 1, st) : cudaSuccess;
    g_upload_share = 1;
    return e;
}

cudaError_t download_bytes_pageable(void* dst, const void* src, size_t bytes, cudaStream_t st, int share)
{
    if (!bytes) return cudaSuccess;
    std::unique_lock<std::mutex> lk(g_call_mutex, std::try_to_lock);
    if (!lk.owns_lock()) {
        const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st);
        return e != cudaSuccess ? e : cudaStreamSynchronize(st);
    }
    g_upload_share = share > 1 ? share : 1;
    const cudaError_t e = download_bytes(dst, src, bytes, st);
    g_upload_share = 1;
    return e;
}

int use_device(int requested, int* dev)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        set_err("no CUDA device", "librecometrics_b200 has no CPU fallback");
        return RMB200_ERR_NO_DEVICE;
    }
    *dev = requested;
    if (*dev < 0) CK(cudaGetDevice(dev));
    if (*dev >= ndev) { set_err("bad argument", "device ordinal out of range"); return RMB200_ERR_BAD_ARG; }
    CK(cudaSetDevice(*dev));
    return RMB200_OK;
}

}  // namespace rmb

extern "C" const char* rmb200_last_error(void) { return rmb::g_err.c_str(); }

extern "C" void rmb200_release_workspace(void)
{
    std::lock_guard<std::mutex> call(rmb::g_call_mutex);      // not while a call is using them
    for (int d = 0; d < rmb::MAX_DEVICES; d++) rmb::upload_pool_release(rmb::g_ups[d]);
    std::lock_guard<std::mutex> lk(rmb::g_pool_mutex);
    rmb::pool_trim_locked(-1);
}
