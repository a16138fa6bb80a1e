// api_common.cuh — host plumbing of the C ABI, shared by its two translation units (gcs_b200_api.cu:
// the batch entry points, sketch_program.cu: the sketch-program entry points): the error path, the
// device scope of an entry point, one counted kernel launch and the dispatch on a kind.
#pragma once

#include <cuda_runtime.h>

#include <type_traits>

#include "../../include/gcs_b200.h"
#include "newton_core.cuh"

namespace gcsk {

// Sets gcs_b200_last_error() of the calling thread (printf-style) and returns `code`.
int fail(int code, const char* fmt, ...);

// Counts one kernel launch in gcs_b200_launch_count().
void count_launch();

// In a function that returns a GCS_* code: a CUDA error fails with GCS_E_CUDA, naming the call and
// where it was made.
#define CUDA_TRY(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return gcsk::fail(GCS_E_CUDA, "%s -> %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// In a function that returns a GCS_* code: passes on a failed GCS_* code.
#define RC_TRY(expr)                   \
    do {                               \
        const int rc_ = (expr);        \
        if (rc_ != GCS_OK) return rc_; \
    } while (0)

// Makes `device` current for the scope's lifetime and makes the caller's device current again when
// it ends, on every return path: no entry point changes the device its caller works on.  A failed
// switch sets rc to GCS_E_CUDA (gcs_b200_last_error() says why); the scope then restores nothing.
class DeviceScope {
public:
    explicit DeviceScope(int device)
    {
        int cur = -1;
        cudaError_t e = cudaGetDevice(&cur);
        if (e == cudaSuccess && cur != device) {
            e = cudaSetDevice(device);
            if (e == cudaSuccess) prev_ = cur;
        }
        rc = e == cudaSuccess ? GCS_OK : fail(GCS_E_CUDA, "making device %d current -> %s", device, cudaGetErrorString(e));
    }
    ~DeviceScope()
    {
        if (prev_ >= 0) cudaSetDevice(prev_);
    }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;

    int rc;

private:
    int prev_ = -1;  // the caller's device, when the scope switched away from it
};

// kernel<<<grid, block, smem, st>>>(args...), counted.  A grid beyond 31 bits launches nothing and
// returns too_large(), the caller's failure in its own words.
template <class... P, class TooLarge, class... A>
int launch_kernel(void (*kernel)(P...), long long grid, int block, size_t smem, cudaStream_t st, TooLarge&& too_large,
    const A&... args)
{
    if (grid > 0x7fffffffLL) return too_large();
    kernel<<<(unsigned)grid, block, smem, st>>>(args...);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

// The cooperative sibling of launch_kernel: cudaLaunchCooperativeKernel, counted.  Every block of
// the grid must be co-resident; a grid that is not fails here as a launch error (GCS_E_CUDA)
// instead of waiting at a grid barrier for blocks that never run.
template <class... P, class... A>
int launch_cooperative(void (*kernel)(P...), unsigned grid, int block, size_t smem, cudaStream_t st, const A&... args)
{
    void* params[] = { const_cast<A*>(&args)... };
    const cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kernel), dim3(grid), dim3(block), params, smem, st);
    count_launch();
    cudaGetLastError();  // the launch's error is e
    if (e != cudaSuccess)
        return fail(GCS_E_CUDA, "cudaLaunchCooperativeKernel(%u blocks of %d threads) -> %s", grid, block, cudaGetErrorString(e));
    return GCS_OK;
}

// f(std::integral_constant<int, kind>()): f sees a kind known at run time as a compile-time
// constant; a kind outside 1..4 is K5.  The host and the kernels' device lambdas share it; the
// pragma lets the one template call either.
#pragma nv_exec_check_disable
template <class F>
__host__ __device__ __forceinline__ auto with_kind(int kind, F&& f)
{
    switch (kind) {
    case GCS_KIND_PP: return f(std::integral_constant<int, GCS_KIND_PP>());
    case GCS_KIND_SDD: return f(std::integral_constant<int, GCS_KIND_SDD>());
    case GCS_KIND_PPL: return f(std::integral_constant<int, GCS_KIND_PPL>());
    case GCS_KIND_PLL: return f(std::integral_constant<int, GCS_KIND_PLL>());
    default: return f(std::integral_constant<int, GCS_KIND_ANG>());
    }
}

// a kind's input and output columns
__host__ __device__ __forceinline__ int in_cols(int kind)
{
    return with_kind(kind, [](auto K) { return Sys<decltype(K)::value>::kCols; });
}

__host__ __device__ __forceinline__ int out_cols(int kind)
{
    return with_kind(kind, [](auto K) { return Sys<decltype(K)::value>::kOut; });
}

}  // namespace gcsk
