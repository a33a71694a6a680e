// runtime.h -- the library's host runtime, shared by the evaluation call (api.cu) and the splitters (split.cu): the
// last-error text, the call mutex, the device workspace cache, the pageable-memory copy lanes, the device pick and the
// exception guard of the C entry points.  Definitions in runtime.cu.
#pragma once

#include "../../include/recometrics_b200.h"
#include <cuda_runtime.h>
#include <exception>
#include <mutex>
#include <new>
#include <string>

namespace rmb {

constexpr int MAX_DEVICES = 16;   // GPUs one call can be spread over

extern thread_local std::string g_err;   // what rmb200_last_error() returns
void set_err(const char* what, const char* detail = nullptr);

#define CK(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            rmb::set_err(#call, cudaGetErrorString(e_));                                 \
            cudaGetLastError();                                                          \
            return (e_ == cudaErrorMemoryAllocation) ? RMB200_ERR_OOM : RMB200_ERR_CUDA; \
        }                                                                                \
    } while (0)

#define TRY(expr) do { const int rc_ = (expr); if (rc_ != RMB200_OK) return rc_; } while (0)   // int return codes

// The body of a C entry point: a C++ exception (std::vector, std::thread, ...) becomes a status code and the last-error
// text instead of unwinding into the caller, where it would end the process.
template <typename F>
int guard(F&& body)
{
    try {
        return body();
    } catch (const std::bad_alloc&) {
        set_err("host allocation failed"); return RMB200_ERR_OOM;
    } catch (const std::exception& e) {
        set_err("unexpected C++ exception", e.what()); return RMB200_ERR_CUDA;
    } catch (...) {
        set_err("unexpected C++ exception"); return RMB200_ERR_CUDA;
    }
}

// Makes `requested` (< 0: the calling thread's current device) the calling thread's device and stores it in *dev.
// RMB200_ERR_NO_DEVICE when the process sees no CUDA device, RMB200_ERR_BAD_ARG for an ordinal out of range.
int use_device(int requested, int* dev);

// One call at a time per process: the SIGINT latch is process-wide, and the copy lanes belong to the holder.
extern std::mutex g_call_mutex;

cudaError_t pool_alloc(void** out, size_t bytes);
void pool_free(void* p);

struct DevBuf {
    void* p = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() { if (p) { pool_free(p); p = nullptr; } }
    cudaError_t alloc(size_t bytes)
    {
        release();
        if (bytes == 0) bytes = 16;
        return pool_alloc(&p, bytes);
    }
    template <typename U> U* as() const { return reinterpret_cast<U*>(p); }
};

extern thread_local int g_upload_share;   // a multi-GPU call divides the host's copy threads among its devices

// rows x row_bytes from host memory (row pitch src_pitch) to a packed device buffer on the current device, ordered on `st`
cudaError_t upload_rows(void* dst, const void* src, size_t src_pitch, size_t row_bytes, size_t rows, cudaStream_t st);

// One contiguous block between pageable host memory and the device for callers that do not hold the call mutex (the
// splitters): through the copy lanes when the mutex is free, else the driver's plain copy, so that a split running beside
// an evaluation call leaves the lanes to it.  `share`: divide the host's copy threads by this much.  The download returns
// when the bytes are in dst.
cudaError_t upload_bytes_pageable(void* dst, const void* src, size_t bytes, cudaStream_t st, int share);
cudaError_t download_bytes_pageable(void* dst, const void* src, size_t bytes, cudaStream_t st, int share);

}  // namespace rmb
