// t3d_preprocess_internal.cuh -- helpers shared by t3d_preprocess.cu (entry points, exact-histogram path,
// normalisation), t3d_preprocess_bracket.cu (percentiles without a per-pixel histogram atomic) and
// t3d_preprocess_fixed.cu (the fixed-window normalisation in one pass).
#pragma once
#include "t3d_common.cuh"

// ------------------------------------------------------------------ bilinear taps
struct Tap { int s0, s1; float c0, c1; };

// cv2 INTER_LINEAR tap for destination index d (resize.cpp, non-IPP path):
// f = (float)((d + 0.5) * scale - 0.5) rounded to fp32 BEFORE floor.
__device__ __forceinline__ Tap linear_tap(int d, int src_dim, double scale) {
    const double fd = __dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5);
    float f = __double2float_rn(fd);
    int s = __float2int_rd(f);
    f = __fsub_rn(f, (float)s);
    if (s < 0) { s = 0; f = 0.f; }
    if (s >= src_dim - 1) { s = src_dim - 1; f = 0.f; }
    Tap t;
    t.s0 = s; t.s1 = min(s + 1, src_dim - 1);
    t.c0 = __fsub_rn(1.0f, f); t.c1 = f;
    return t;
}

__device__ __forceinline__ uint16_t sat_u16(float v) {
    const int r = __float2int_rn(v);        // round half to even
    return (uint16_t)min(max(r, 0), 65535);
}

template <typename SrcT, bool DIV65535>
__device__ __forceinline__ float src_value(const SrcT* __restrict__ p) {
    const float v = (float)__ldg(p);
    return DIV65535 ? __fdiv_rn(v, 65535.0f) : v;
}

template <typename SrcT, bool DIV65535>
__device__ __forceinline__ float bilinear_at(const SrcT* __restrict__ src, int sw, const Tap& ty, const Tap& tx) {
    const SrcT* r0 = src + (size_t)ty.s0 * sw;
    const SrcT* r1 = src + (size_t)ty.s1 * sw;
    // horizontal pass then vertical pass, every product rounded separately (no FMA)
    const float h0 = __fadd_rn(__fmul_rn(src_value<SrcT, DIV65535>(r0 + tx.s0), tx.c0),
                               __fmul_rn(src_value<SrcT, DIV65535>(r0 + tx.s1), tx.c1));
    const float h1 = __fadd_rn(__fmul_rn(src_value<SrcT, DIV65535>(r1 + tx.s0), tx.c0),
                               __fmul_rn(src_value<SrcT, DIV65535>(r1 + tx.s1), tx.c1));
    return __fadd_rn(__fmul_rn(h0, ty.c0), __fmul_rn(h1, ty.c1));
}

// H54 -- the dataset's horizontal geometry.  640 -> 512 columns (data/dataset_loader.py:242 with the training size of
// train_thermal_dustr.py) is a 5:4 reduction: scale = 1.25 exactly, so cv2's x taps are periodic -- 4 outputs from 5
// inputs, weights {1/8, 3/8, 5/8, 7/8}, no border clamping -- and become compile-time constants: a lane's 8 output
// pixels read 10 consecutive source pixels (five 32-bit shared loads instead of sixteen 16-bit ones, no tap
// registers).  Same arithmetic, same order, same bits.  (The vertical 512 -> 384 is 4:3: its taps are not exactly
// periodic in floating point and stay in the table.)  DIV65535: the source values are divided by 65535 in fp32 first
// (the inference path, thermal_dustr_inference.py:42-52).
template <int K> struct W54 { static constexpr float f = (2 * (K & 3) + 1) * 0.125f; static constexpr float c = 1.0f - f; };

template <bool DIV65535 = false>
__device__ __forceinline__ void hpass54(uint32_t saddr, float h[8]) {
    unsigned int w[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w[i]) : "r"(saddr + 4u * i));
    float p[10];
#pragma unroll
    for (int i = 0; i < 5; ++i) { p[2 * i] = (float)(w[i] & 0xffffu); p[2 * i + 1] = (float)(w[i] >> 16); }
    if (DIV65535) {
#pragma unroll
        for (int i = 0; i < 10; ++i) p[i] = __fdiv_rn(p[i], 65535.0f);
    }
    // output u reads source pixels u + u / 4 and the next one
    h[0] = __fadd_rn(__fmul_rn(p[0], W54<0>::c), __fmul_rn(p[1], W54<0>::f));
    h[1] = __fadd_rn(__fmul_rn(p[1], W54<1>::c), __fmul_rn(p[2], W54<1>::f));
    h[2] = __fadd_rn(__fmul_rn(p[2], W54<2>::c), __fmul_rn(p[3], W54<2>::f));
    h[3] = __fadd_rn(__fmul_rn(p[3], W54<3>::c), __fmul_rn(p[4], W54<3>::f));
    h[4] = __fadd_rn(__fmul_rn(p[5], W54<0>::c), __fmul_rn(p[6], W54<0>::f));
    h[5] = __fadd_rn(__fmul_rn(p[6], W54<1>::c), __fmul_rn(p[7], W54<1>::f));
    h[6] = __fadd_rn(__fmul_rn(p[7], W54<2>::c), __fmul_rn(p[8], W54<2>::f));
    h[7] = __fadd_rn(__fmul_rn(p[8], W54<3>::c), __fmul_rn(p[9], W54<3>::f));
}

// ------------------------------------------------------------------ cp.async / shared-memory access
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst_saddr, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst_saddr), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ unsigned int lds_u16(uint32_t saddr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr));
    return v;
}

// np.percentile(method='linear') finish (numpy _quantile/_lerp): a, b fp32 order
// statistics, d = b - a in fp32, result fp64 two-sided lerp.
__device__ __forceinline__ double lerp_percentile(float a, float b, double g) {
    const float d = __fsub_rn(b, a);
    return (g < 0.5) ? __dadd_rn((double)a, __dmul_rn((double)d, g))
                     : __dsub_rn((double)b, __dmul_rn((double)d, __dsub_rn(1.0, g)));
}

__device__ __forceinline__ void percentile_ranks(int n, double q, unsigned int* k, double* g) {
    const double vi = __dmul_rn((double)(n - 1), __ddiv_rn(q, 100.0));
    const double fl = floor(vi);
    *k = (unsigned int)fl;
    *g = __dsub_rn(vi, fl);
}

// out = float( clip((double(x) - p2) / (p98 - p2), 0, 1) ), NaN propagates like np.clip
__device__ __forceinline__ float normalize_px(double x, double p2, double den) {
    const double q = __ddiv_rn(__dsub_rn(x, p2), den);
    if (isnan(q)) return __int_as_float(0x7fc00000);
    return __double2float_rn(fmin(fmax(q, 0.0), 1.0));
}

// ------------------------------------------------------------------ per-frame normalisation LUT
// Raw counts are integers, so clip((v - p2) / (p98 - p2), 0, 1) takes at most ceil(p98) - floor(p2) + 3
// distinct values per frame: the percentile kernel (one CTA per frame) tabulates them ONCE with the fp64
// formula (same function, same bits) and the normalisation kernel only looks them up.
constexpr int kLutMax = 4096;        // float2 entries (32 KB): covers p98 - p2 < 4093 counts, else the direct fp64 path

// all threads of the CTA; lutmeta[b] = {first value (floor(p2) - 1), entries} (entries == 0: no LUT)
__device__ __forceinline__ void build_norm_lut(int b, double p2, double p98, int rep3, float2* __restrict__ glut,
                                               int2* __restrict__ lutmeta) {
    const double den = __dsub_rn(p98, p2);
    const bool finite = (p2 == p2) && (p98 == p98) && fabs(p2) < 1.0e9 && fabs(p98) < 1.0e9;
    const int lom1 = finite ? (int)floor(p2) - 1 : 0, hip1 = finite ? (int)ceil(p98) + 1 : 0;
    const int range = hip1 - lom1 + 1;
    const bool use = finite && range <= kLutMax;
    if (use) {
        float2* l = glut + (size_t)b * kLutMax;
        for (int k = threadIdx.x; k < range; k += blockDim.x) {
            const float o = normalize_px((double)(lom1 + k), p2, den);
            l[k] = make_float2(o, rep3 ? gray3(o, o, o) : o);
        }
    }
    if (threadIdx.x == 0) lutmeta[b] = make_int2(lom1, use ? range : 0);
}

// ------------------------------------------------------------------ thermal-gradient statistics of the output image
// The normalisation kernels write partial sums per (frame, band of rows): grad_stats[b][band][4] (T3D_STATS_TILES).
constexpr int kNormBands = 24;       // CTAs per frame == statistic partials per frame (T3D_STATS_TILES)

// Half-resolution sums of a band (utils/loss.py:133-174: |Dx|, |Dy| of the 2x2 average-pooled gray image, zero-padded
// last column / row), for the multi-scale loss.  Thread = pooled column (W / 2 <= kNormThreads), the band's pooled rows
// (+ the one below) in registers; the right neighbour comes from a shuffle, across warps from shared memory.
constexpr int kS2MaxPool = 9;            // pooled rows of a band + 1 (bands of <= 16 rows)
template <typename Pooled>
__device__ __forceinline__ void half_res_band_sums(int y0, int y1, int H, int W, float (*edge)[kS2MaxPool],
                                                   Pooled pooled, float& tx2, float& ty2) {
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int h2 = H >> 1, w2 = W >> 1;
    const int I0 = y0 >> 1, I1 = min(y1, 2 * h2) >> 1;               // y0 is even: the band's own pooled rows [I0, I1)
    const int nown = I1 - I0, npool = nown + ((I1 < h2) ? 1 : 0);
    const int J = tid;
    float pv[kS2MaxPool];
#pragma unroll
    for (int r = 0; r < kS2MaxPool; ++r) pv[r] = (r < npool && J < w2) ? pooled(I0 + r, J) : 0.f;
    if (lane == 0) {
#pragma unroll
        for (int r = 0; r < kS2MaxPool; ++r) edge[wrp][r] = pv[r];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kS2MaxPool - 1; ++r) {
        float right = __shfl_down_sync(0xffffffffu, pv[r], 1);
        if (lane == 31) right = edge[wrp + 1][r];
        if (r < nown && J < w2) {
            if (J + 1 < w2) tx2 += fabsf(right - pv[r]);
            if (I0 + r + 1 < h2) ty2 += fabsf(pv[r + 1] - pv[r]);
        }
    }
}

// ------------------------------------------------------------------ percentile brackets (t3d_preprocess_bracket.cu)
constexpr int kBrBins = 2048;        // bins of each windowed histogram (p2 window, p98 window)
constexpr int kBrSlots = kBrBins + 32;  // + the below / above slot (t3d_preprocess_bracket.cu: kBrStride)

// ------------------------------------------------------------------ workspace of t3d_preprocess_train_u16
struct PreWs {
    uint16_t* resized;           // [B][dh*dw]
    unsigned int* meta;          // [2B+1]  per-frame vmin / vmax (exact-histogram path)
    uint2* gxt; uint4* gyt;      // bilinear taps
    unsigned int* bracket;       // [B][4]  lo2, hi2, lo98, hi98 (inclusive value windows)
    unsigned int* brhist;        // [B][2][kBrSlots], then one uint: frames that took the exact-select fallback
    float2* lut;                 // [B][kLutMax]
    int2* lutmeta;               // [B]
    size_t total;
};

static inline PreWs pre_ws_layout(void* base, int B, int dh, int dw) {
    PreWs w;
    size_t off = 0;
    char* p = reinterpret_cast<char*>(base);
    auto take = [&](size_t bytes) { char* r = p ? p + off : nullptr; off += t3d_align_up(bytes, 256); return r; };
    w.resized = reinterpret_cast<uint16_t*>(take((size_t)B * dh * dw * sizeof(uint16_t)));
    w.meta = reinterpret_cast<unsigned int*>(take((size_t)(2 * B + 1) * sizeof(unsigned int)));
    w.gxt = reinterpret_cast<uint2*>(take((size_t)dw * sizeof(uint2)));
    w.gyt = reinterpret_cast<uint4*>(take((size_t)dh * sizeof(uint4)));
    w.bracket = reinterpret_cast<unsigned int*>(take((size_t)B * 4 * sizeof(unsigned int)));
    w.brhist = reinterpret_cast<unsigned int*>(take(((size_t)B * 2 * kBrSlots + 1) * sizeof(unsigned int)));
    w.lut = reinterpret_cast<float2*>(take((size_t)B * kLutMax * sizeof(float2)));
    w.lutmeta = reinterpret_cast<int2*>(take((size_t)B * sizeof(int2)));
    w.total = off;
    return w;
}

// Percentiles without the full histogram (hist == NULL in t3d_preprocess_train_u16): sample -> value brackets
// around the p2 / p98 ranks -> one pass that resizes, counts the pixels below each bracket and histograms only
// the few percent inside -> exact order statistics, np.percentile lerp, normalisation LUT.
// `same` : source and destination sizes are equal (no resize; `resized` is not written, the raw frame is used).
// `shared`: other kernels run concurrently with the preprocessing (t3d_preprocess_train_u16's `shared`).
int t3d_launch_bracket_percentiles(const uint16_t* raw, int B, int sh, int sw, int dh, int dw, bool same,
                                   const PreWs& w, int rep3, double* percentiles, bool shared, int phase, cudaStream_t st);
