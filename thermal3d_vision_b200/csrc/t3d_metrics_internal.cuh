// t3d_metrics_internal.cuh -- the per-pixel arithmetic of utils/metrics.py:48-59 (used by t3d_metrics.cu).
#pragma once
#include "t3d_common.cuh"
#include "t3d_select.cuh"

namespace t3d_metrics {

constexpr int kNPart = 8;                  // abs_rel, sq_rel, sq, log2, a1, a2, a3, (pad)
constexpr int kResampleMaxDim = 2048;      // H + W limit of the in-kernel nearest-neighbour index tables (8 KB)

__device__ __forceinline__ unsigned int key_of_bits(unsigned int b) { return b ^ ((unsigned int)((int)b >> 31) | 0x80000000u); }

__device__ __forceinline__ float np_maximum(float a, float b) { return (isnan(a) || isnan(b)) ? __int_as_float(0x7fc00000) : fmaxf(a, b); }

// Per-pixel terms of utils/metrics.py:48-59.  GENERAL == false (mask = gt > 0 & finite, so gt is a positive
// finite number): exactly one of gt/pred, pred/gt is >= 1, hence max(gt/pred, pred/gt) = max(gt,p) / min(gt,p)
// -- ONE IEEE division keeps the delta-counts exact -- and (log gt - log p)^2 = log(thresh)^2.  Non-positive or
// NaN predictions take the literal two-division form (same results as numpy: NaN / inf propagate).
template <bool GENERAL>
__device__ __forceinline__ void metric_terms(float gt, float z, float s, float accf[4], int cnt[3]) {
    if (isnan(gt)) return;                                                   // invalid pixel marker
    const float pr = __fmul_rn(z, s);                                        // pred *= scale   (:48)
    float th, dl;
    if (!GENERAL && pr > 0.f) {
        th = __fdiv_rn(fmaxf(gt, pr), fminf(gt, pr));                        // :51
        dl = 0.69314718f * __log2f(th);                                      // |log gt - log pred|
    } else {
        th = np_maximum(__fdiv_rn(gt, pr), __fdiv_rn(pr, gt));
        dl = __logf(gt) - __logf(pr);
    }
    cnt[0] += th < 1.25f; cnt[1] += th < 1.5625f; cnt[2] += th < 1.953125f;  // :52-54
    const float d = __fsub_rn(gt, pr);
    const float d2 = __fmul_rn(d, d);
    // IEEE divisions, as numpy: 1 / gt is subnormal for gt > 2^126 (an approximate reciprocal flushes it to 0) and
    // overflows for gt < 2^-128
    accf[0] += __fdiv_rn(fabsf(d), gt);                                      // :56  |gt - pred| / gt
    accf[1] += __fdiv_rn(d2, gt);                                            // :57
    accf[2] += d2;                                                           // :58
    accf[3] += dl * dl;                                                      // :59
}

// Fast form of the per-pixel terms for the common case (no caller mask: gt is a positive finite number or the
// NaN "invalid" marker; scaled prediction positive): branch-free, validity by select, counts by predicate.
// Same arithmetic as metric_terms<false>: ONE IEEE division max/min keeps the delta-counts exact.
__device__ __forceinline__ float lg2_fast(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

__device__ __forceinline__ void metric_terms_fast(float gt, float pr, float accf[4], int cnt[3]) {
    const bool valid = (gt == gt);                                           // NaN marks an unselected pixel
    const float g = valid ? gt : 1.0f, q = valid ? pr : 1.0f;               // -> th = 1, every term 0
    const float th = __fdiv_rn(fmaxf(g, q), fminf(g, q));                    // :51 (exactly one of the two ratios is >= 1)
    const float dl = 0.69314718f * lg2_fast(th);                             // |log gt - log pred|, th >= 1 is normal
    cnt[0] += (valid && th < 1.25f); cnt[1] += (valid && th < 1.5625f); cnt[2] += (valid && th < 1.953125f);   // :52-54
    const float d = g - q;
    const float d2 = d * d;
    accf[0] += __fdiv_rn(fabsf(d), g);                                       // :56  |gt - pred| / gt (IEEE, as metric_terms)
    accf[1] += __fdiv_rn(d2, g);                                             // :57
    accf[2] += d2;                                                           // :58
    accf[3] = fmaf(dl, dl, accf[3]);                                         // :59
}

// Division-free form of the same terms for g, q in [2^-120, 2^126) (valid pixels; invalid ones are passed as
// g = q = 1).  numpy: thresh = max(gt/pred, pred/gt) = fl(a / b), a = max, b = min
// (IEEE division is monotone), counted against T in {1.25, 1.5625, 1.953125} (:51-54).  For such T (in (1, 2), even
// mantissa) fl(a / b) < T  <=>  a / b < T - 2^-24 (the midpoint below T; a tie rounds to even = T)
// <=>  a - T b + 2^-24 b < 0, and that sign is computed EXACTLY by two FMAs: r = fma(-T, b, a) is exact whenever
// |a - T b| < b / 64 and ulp(b) / 64 >= 2^-149, and otherwise so much larger than 2^-24 b that its rounding cannot
// change the sign of the sum; fma(2^-24, b, r) rounds once, which never flips a sign (a negative sum that underflows
// is -0: sign bit set).  Exactness: a and T b are multiples of ulp(b) / 64 (T = k / 64), so r is one too, with at most
// 24 significant bits when |r| < b / 64 -- an fp32 number if that grid is not finer than the fp32 subnormal
// spacing 2^-149, i.e. ulp(b) >= 2^-143, b >= 2^-120.  Below that r is rounded and the sign can flip (the kernel
// sends such pixels to the literal formula; tests/test_metrics_nodiv_cpu.py restates both FMAs).
// -> the delta-counts are those of the correctly rounded quotient, without dividing.
// Above: g < 2^126 keeps 1 / g normal (rcp.approx.ftz flushes a subnormal reciprocal to 0).
// log: u = q / g to ~1 ulp (reciprocal + one Newton step), |log gt - log pred| = ln2 |lg2 u|; the caller folds
// ln2^2 into the sum of lg2(u)^2 (accl2).
__device__ __forceinline__ float rcp_fast(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// An unselected pixel (g = q = 1) adds 0 to every sum and 1 to every count: the caller subtracts their number.
__device__ __forceinline__ void metric_terms_nodiv(float g, float q, float accf[3], float& accl2, int cnt[3]) {
    const float a = fmaxf(g, q), b = fminf(g, q);
    const float c = 5.9604644775390625e-08f;                                 // 2^-24
    // a, b are positive normal numbers here, so the sum is finite and never -0: "< 0" is its sign bit (one shift-add
    // instead of compare + select + add)
    cnt[0] += (int)(__float_as_uint(fmaf(c, b, fmaf(-1.25f, b, a))) >> 31);        // :52
    cnt[1] += (int)(__float_as_uint(fmaf(c, b, fmaf(-1.5625f, b, a))) >> 31);      // :53
    cnt[2] += (int)(__float_as_uint(fmaf(c, b, fmaf(-1.953125f, b, a))) >> 31);    // :54
    const float rg = rcp_fast(g);
    float u = q * rg;
    u = fmaf(fmaf(-u, g, q), rg, u);                                         // Newton: u = q / g to ~1 ulp
    const float l2 = lg2_fast(u);
    accl2 = fmaf(l2, l2, accl2);                                             // :59 (in log2 units)
    const float d = g - q;
    const float d2 = d * d;
    accf[0] = fmaf(fabsf(d), rg, accf[0]);                                   // :56  |gt - pred| / gt
    accf[1] = fmaf(d2, rg, accf[1]);                                         // :57
    accf[2] += d2;                                                           // :58
}

}  // namespace t3d_metrics
