// spx_internal.h -- shared host-side helpers of libspx (error codes, thread-local last error).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/spx.h"

namespace spx {

int spx_set_error(int code, const char* fmt, ...);

#define SPX_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return ::spx::spx_set_error(SPX_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                        __FILE__, __LINE__);                                             \
    } while (0)

// NVTX range (SURVEY.md section 5, tracing row): names the H2D / kernel / D2H enqueue sections of the host pipeline, the
// ingest ring and the peer-output path in nsys / ncu timelines.  Header-only NVTX3: a no-op unless a tool is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name);
    ~NvtxRange();
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

#define SPX_TRY(expr)                 \
    do {                              \
        int _rc = (expr);             \
        if (_rc != SPX_OK) return _rc; \
    } while (0)

// SPX_E_NODEVICE without a CUDA device, SPX_E_INVALID unless 0 <= device < device count; else makes `device` current.
int check_device(int device);

// The byte size in environment variable `name` when it is set and at least `min` (>= 1), else `fallback`.
size_t env_bytes(const char* name, size_t fallback, long long min);

// Blocks of `kern` resident per SM at `threads` threads and `smem` bytes of dynamic shared memory on the current
// device (occ may be NULL); the first call per kernel and device raises the kernel's dynamic shared-memory limit to smem.
int kernel_setup(const void* kern, int threads, size_t smem, int* occ);

// K3 (features_kernel) over `batch` spectra of n bins `stride` apart, float32 (dtype 0) or float64 (dtype 1), on `st`;
// NULL user_opts: the reference's options
int features_launch(const void* in, int dtype, int n, int batch, long long stride, spx_features* out, int* peaks,
                    int peaks_cap, const spx_feature_opts* user_opts, cudaStream_t st);

}  // namespace spx
