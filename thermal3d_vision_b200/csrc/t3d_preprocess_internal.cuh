// t3d_preprocess_internal.cuh -- helpers shared by t3d_preprocess.cu (entry points, exact-histogram path,
// normalisation) and t3d_preprocess_bracket.cu (percentiles without a per-pixel histogram atomic).
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
