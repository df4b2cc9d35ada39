// common.cuh — error plumbing and small device helpers shared by every translation unit
// of libat_b200.so.
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "at_b200.h"

namespace at {

// Thread-local message returned by at_last_error().
char* error_buffer();
int set_error(int code, const char* fmt, ...);

#define AT_CUDA_TRY(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return ::at::set_error(_e == cudaErrorMemoryAllocation ? AT_ERR_NOMEM : AT_ERR_CUDA, \
                                   "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
                                   __FILE__, __LINE__);                                     \
    } while (0)

#define AT_LAUNCH_CHECK(name)                                                               \
    do {                                                                                    \
        cudaError_t _e = cudaGetLastError();                                                \
        if (_e != cudaSuccess)                                                              \
            return ::at::set_error(AT_ERR_CUDA, "launch of %s failed: %s (%s:%d)", name,    \
                                   cudaGetErrorString(_e), __FILE__, __LINE__);             \
    } while (0)

#define AT_REQUIRE(cond, ...)                                                               \
    do {                                                                                    \
        if (!(cond)) return ::at::set_error(AT_ERR_INVALID, __VA_ARGS__);                   \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Number of SMs of the current device (cached per device).
int sm_count();

// Device memory for the library's handles and temporaries, from a per-device cache of freed
// blocks.  cudaMalloc / cudaFree cost milliseconds each once several processes share a box (the
// driver maps and unmaps under a lock): the 15 buffers of one kNN index were 11 ms to allocate
// on an idle box and 150 ms with four ranks doing the same.  device_free waits for the device
// like cudaFree does (the block may still be in use by queued kernels) and keeps the block for
// the next request of the same size; at_device_cache_trim() returns everything to the driver.
cudaError_t device_alloc(void** p, size_t bytes);
void device_free(void* p);

// AT_ERR_INVALID unless the matrix is staged on `device` (on the current device).
int check_csr_device(const at_csr_t* csr, int device, const char* who);
int check_csr_on_current_device(const at_csr_t* csr, const char* who);

constexpr int kWarp = 32;

// Streaming (evict-first) 16-byte store: Y is written once and never re-read by the kernel.
__device__ __forceinline__ void st_stream_f4(float4* p, float4 v) { __stcs(p, v); }

// 16-byte read-only load through the non-coherent path.
__device__ __forceinline__ float4 ld_ro_f4(const float4* p) { return __ldg(p); }

}  // namespace at
