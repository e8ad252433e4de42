// t3d_bilinear.cuh -- F.interpolate(mode='bilinear', align_corners=False) arithmetic, shared by every kernel that
// resamples: interp_bilinear_kernel (t3d_preprocess.cu), the tile loss kernel's fused taps (t3d_loss.cu) and the
// resampling marching kernel (t3d_loss_march.cu).  One definition with every rounding spelled out, so that "resample,
// then compute" and "resample while loading" produce the same bits at every call site.
#pragma once
#include <math.h>

// ATen: scale = in / out in fp32; src = max(scale * (dst + 0.5) - 0.5, 0); i0 = (int)src; i1 = i0 + (i0 < in - 1);
// l1 = src - i0; l0 = 1 - l1.  The scale * (dst + 0.5) - 0.5 step is one fused multiply-add (what nvcc made of the
// expression before it was spelled out); the host evaluates the same taps with the same roundings (the marching
// kernel's launcher sizes its shared-memory segments with it).
struct BTap { int i0, i1; float l0, l1; };
__host__ __device__ __forceinline__ float bscale(int in, int out) { return (float)in / (float)out; }
__host__ __device__ __forceinline__ BTap btap(int dst, int in, float scale) {
    const float f = fmaxf(fmaf(scale, (float)dst + 0.5f, -0.5f), 0.f);
    BTap t;
    t.i0 = (int)f; t.i1 = t.i0 + ((t.i0 < in - 1) ? 1 : 0);
    t.l1 = f - (float)t.i0; t.l0 = 1.f - t.l1;
    return t;
}

#ifdef __CUDACC__
// l0y (l0x v00 + l1x v01) + l1y (l0x v10 + l1x v11), each sum one fused multiply-add of the rounded other product.
// A zero weight times a non-finite value is NaN, as in ATen: callers read the i1 taps even when l1 == 0.
__device__ __forceinline__ float blerp(float v00, float v01, float v10, float v11, const BTap& ty, const BTap& tx) {
    const float a = __fmaf_rn(tx.l0, v00, __fmul_rn(tx.l1, v01));
    const float b = __fmaf_rn(tx.l0, v10, __fmul_rn(tx.l1, v11));
    return __fmaf_rn(ty.l0, a, __fmul_rn(ty.l1, b));
}
#endif
