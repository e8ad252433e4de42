// t3d_common.cuh -- shared device/host helpers for libt3d_sm100.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/t3d.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libt3d_sm100 is written for sm_100a (B200) only"
#endif

// ---------------------------------------------------------------- host side
void t3d_set_error(const char* fmt, ...);
void t3d_count_launch(int n = 1);

#define T3D_REQUIRE(cond, ...)                                   \
    do {                                                         \
        if (!(cond)) {                                           \
            t3d_set_error(__VA_ARGS__);                          \
            return T3D_ERR_BAD_ARG;                              \
        }                                                        \
    } while (0)

#define T3D_CUDA(expr)                                                               \
    do {                                                                             \
        cudaError_t e__ = (expr);                                                    \
        if (e__ != cudaSuccess) {                                                    \
            t3d_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),   \
                          __FILE__, __LINE__);                                       \
            return T3D_ERR_CUDA;                                                     \
        }                                                                            \
    } while (0)

#define T3D_LAUNCH_CHECK(name)                                                       \
    do {                                                                             \
        cudaError_t e__ = cudaGetLastError();                                        \
        if (e__ != cudaSuccess) {                                                    \
            t3d_set_error("launch of %s failed: %s", name, cudaGetErrorString(e__)); \
            return T3D_ERR_CUDA;                                                     \
        }                                                                            \
        t3d_count_launch();                                                          \
    } while (0)

int t3d_sm_count();   // cached per process (current device at first call; every device of a B200 box is the same part)
// Index of the calling thread's current CUDA device, for per-device one-time setup (cudaFuncSetAttribute is per
// device: a process that drives several GPUs must repeat it on each).
constexpr int kT3dMaxDevices = 64;
int t3d_device_slot();

// cudaFuncSetAttribute(Kernel, MaxDynamicSharedMemorySize, bytes) once per device.  The flag is keyed on the kernel
// itself (not on its type: instantiations with the same signature each need their own); benign race: idempotent.
template <auto Kernel>
int t3d_set_max_dynamic_smem(int bytes) {
    static bool done[kT3dMaxDevices] = {};
    bool& set = done[t3d_device_slot()];
    if (!set) {
        T3D_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        set = true;
    }
    return T3D_OK;
}

// Optional per-kernel CUDA-event timing (t3d_profile_begin / t3d_profile_end in include/t3d.h).
bool t3d_prof_before(const char* name, cudaStream_t st);
void t3d_prof_after(cudaStream_t st);

// T3D_LAUNCH("kernel_name", stream, kernel<<<grid, block, smem, stream>>>(args...));
#define T3D_LAUNCH(name, st, ...)                        \
    do {                                                 \
        const bool prof__ = t3d_prof_before(name, st);   \
        __VA_ARGS__;                                     \
        if (prof__) t3d_prof_after(st);                  \
        T3D_LAUNCH_CHECK(name);                          \
    } while (0)

static inline bool t3d_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline size_t t3d_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// -------------------------------------------------------------- device side
#ifdef __CUDACC__

// Streaming 128-bit global accesses: inputs are read once (no L1 allocation),
// outputs are written once (evict-first / cache-streaming).
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float ldg_stream_f1(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
// Halo data is shared with neighbouring tiles: keep the default (L1-allocating) path.
__device__ __forceinline__ float ldg_f1(const float* p) { return __ldg(p); }

__device__ __forceinline__ void stg_stream_f4(float* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void stg_stream_f1(float* p, float v) {
    asm volatile("st.global.cs.f32 [%0], %1;" :: "l"(p), "f"(v) : "memory");
}

// L2 residency control (createpolicy + .L2::cache_hint): scratch that one kernel writes and the next one reads is
// kept in the 126 MB L2 ("evict_last") while the streaming traffic around it passes through with normal priority.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void stg_f4_l2hint(float* p, float4 v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(policy) : "memory");
}
__device__ __forceinline__ float4 ldg_f4_l2hint(const float* p, uint64_t policy) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(policy));
    return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ float sgnf(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// cv2 INTER_NEAREST source index of destination index d: min(floor(d * scale), src - 1), scale = src / dst in fp64
// (utils/evaluate_depth_metrics.py:321-323).  Every nearest resample of the library goes through this one rule: the
// results are bit-exact against cv2 only while it matches cv2's.
__device__ __forceinline__ int nearest_src(int d, double scale, int src) {
    return min((int)floor(__dmul_rn((double)d, scale)), src - 1);
}

// gray = 0.299 c0 + 0.587 c1 + 0.114 c2, fp32, left to right, no FMA contraction
// (utils/loss.py:120; the rounding is an input to every thermal term).
__device__ __forceinline__ float gray3(float c0, float c1, float c2) {
    return __fadd_rn(__fadd_rn(__fmul_rn(0.299f, c0), __fmul_rn(0.587f, c1)), __fmul_rn(0.114f, c2));
}

#endif  // __CUDACC__
