// t3d_preprocess.cu -- 16-bit radiometric thermal -> normalised, contrast
// equalised, resized float thermal (sm_100a).
//
// Replaces /root/reference/utils/preprocessing.py:6-30 (enhance_thermal_contrast),
// :32-73 (enhance_thermal_fixed_range) and the cv2.resize calls around them
// (data/dataset_loader.py:237-249 train path, thermal_dustr_inference.py:25-60
// inference path, utils/evaluate_depth_metrics.py:320-323 nearest GT resample).
// Exact recipes: SURVEY.md Appendix B.  Outputs are bit-exact with
// numpy/OpenCV (IPP off): no FMA contraction in the interpolation, fp64 in
// the normalisation, integer histograms.
#include "t3d_preprocess_internal.cuh"
#include "t3d_select.cuh"
#include "t3d_bilinear.cuh"

namespace {

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

// ------------------------------------------------------------------ K1: resize kernels
// MODE 0: u16 -> u16 (train path, data/dataset_loader.py:242)
// MODE 1: u16 -> f32 with /65535 first (inference path, thermal_dustr_inference.py:42-52)
// MODE 2: f32 -> f32
template <int MODE>
__global__ void __launch_bounds__(256) resize_bilinear_kernel(const void* __restrict__ src_, void* __restrict__ dst_,
                                                              int B, int sh, int sw, int dh, int dw) {
    const double scx = (double)sw / (double)dw, scy = (double)sh / (double)dh;
    const size_t total = (size_t)B * dh * dw;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(idx % dw);
        const size_t t = idx / dw;
        const int y = (int)(t % dh);
        const int b = (int)(t / dh);
        const Tap tx = linear_tap(x, sw, scx), ty = linear_tap(y, sh, scy);
        if (MODE == 0) {
            const uint16_t* s = reinterpret_cast<const uint16_t*>(src_) + (size_t)b * sh * sw;
            reinterpret_cast<uint16_t*>(dst_)[idx] = sat_u16(bilinear_at<uint16_t, false>(s, sw, ty, tx));
        } else if (MODE == 1) {
            const uint16_t* s = reinterpret_cast<const uint16_t*>(src_) + (size_t)b * sh * sw;
            reinterpret_cast<float*>(dst_)[idx] = bilinear_at<uint16_t, true>(s, sw, ty, tx);
        } else {
            const float* s = reinterpret_cast<const float*>(src_) + (size_t)b * sh * sw;
            reinterpret_cast<float*>(dst_)[idx] = bilinear_at<float, false>(s, sw, ty, tx);
        }
    }
}

// cv2 INTER_NEAREST (nearest_src)
__global__ void __launch_bounds__(256) resize_nearest_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                             int B, int sh, int sw, int dh, int dw) {
    const double fx = (double)sw / (double)dw, fy = (double)sh / (double)dh;
    const size_t total = (size_t)B * dh * dw;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(idx % dw);
        const size_t t = idx / dw;
        const int y = (int)(t % dh);
        const int b = (int)(t / dh);
        const int sx = nearest_src(x, fx, sw), sy = nearest_src(y, fy, sh);
        dst[idx] = __ldg(src + ((size_t)b * sh + sy) * sw + sx);
    }
}

// ------------------------------------------------------------------ K2a: fused resize + privatised histogram (train path)
// One CTA owns up to 49 152 output pixels of one frame and a shared-memory
// histogram of all 65 536 values packed as 2 x u16 per word (128 KB): counts
// cannot overflow because a CTA sees < 65 536 pixels.  Non-zero bins are merged
// into the frame's global u32 histogram with atomics (integer adds: exact and
// order independent -> bit-exact, deterministic).
constexpr int kHistThreads = 256;
constexpr int kHistRows = 32;        // destination rows per CTA
constexpr int kWinBins = 16384;      // privatised window of the 65 536-bin histogram (2 x u16 counters per word)
constexpr int kWinWords = kWinBins / 2;
constexpr int kHistMaxW = 2044;      // widest destination row: x-tap table in shared memory and < 65 536 px per CTA

// all bilinear taps of one resize geometry, computed once per call (fp64 tap arithmetic is not cheap)
__global__ void build_taps_kernel(int sh, int sw, int dh, int dw, uint2* __restrict__ xt, uint4* __restrict__ yt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < dw) {
        const Tap t = linear_tap(i, sw, (double)sw / (double)dw);
        xt[i] = make_uint2((unsigned)t.s0 | ((unsigned)t.s1 << 16), __float_as_uint(t.c1));
    }
    if (i < dh) {
        const Tap t = linear_tap(i, sh, (double)sh / (double)dh);
        yt[i] = make_uint4((unsigned)t.s0, (unsigned)t.s1, __float_as_uint(t.c0), __float_as_uint(t.c1));
    }
}

// One CTA = kHistRows destination rows of one frame.  Thermal frames occupy a narrow band of the 16-bit range,
// so the CTA privatises only a 16 384-bin WINDOW of the histogram in shared memory (32 KB -> 6 CTAs per SM),
// centred on the values of a sample row; the rare values outside the window go straight to the frame's
// global histogram.  Integer adds only: exact and order independent -> bit-exact, deterministic.
// Warps take rows, lanes take columns with 4 independent pixels in flight.  The frame's [vmin, vmax] is
// published for the percentile kernel.
template <bool RESIZE>
__global__ void __launch_bounds__(kHistThreads, 6)
resize_hist_u16_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ resized,
                       unsigned int* __restrict__ hist, unsigned int* __restrict__ meta /* [B] min, [B] max */,
                       const uint2* __restrict__ gxt, const uint4* __restrict__ gyt,
                       int B, int sh, int sw, int dh, int dw, int chunks) {
    extern __shared__ unsigned int win[];       // kWinWords, then the x-tap table (RESIZE only)
    uint2* xt = reinterpret_cast<uint2*>(win + kWinWords);          // {s0 | s1 << 16, bits of f}
    __shared__ unsigned int s_lo, s_hi;
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int b = blockIdx.x / chunks, chunk = blockIdx.x - b * chunks;
    const int y0 = chunk * kHistRows, y1 = min(y0 + kHistRows, dh);
    const uint16_t* s = src + (size_t)b * sh * sw;
    unsigned int* gh = hist + (size_t)b * 65536;
    const int srow = (sw + 7) & ~7;
    const bool vec_rows = ((sw & 7) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15u) == 0);
    for (int i = tid; i < kWinWords; i += kHistThreads) win[i] = 0u;
    if (RESIZE) for (int x = tid; x < dw; x += kHistThreads) xt[x] = __ldg(gxt + x);
    if (tid == 0) { s_lo = 0xffffu; s_hi = 0u; }
    __syncthreads();
    auto ytap = [&](int y) -> Tap {
        const uint4 t = __ldg(gyt + y);
        Tap r; r.s0 = (int)t.x; r.s1 = (int)t.y; r.c0 = __uint_as_float(t.z); r.c1 = __uint_as_float(t.w);
        return r;
    };
    auto pixel = [&](const uint16_t* r0, const uint16_t* r1, const Tap& ty, int x) -> unsigned int {
        const uint2 t = xt[x];
        const int s0 = t.x & 0xffff, s1 = t.x >> 16;
        const float f = __uint_as_float(t.y), c0 = __fsub_rn(1.0f, f);
        const float h0 = __fadd_rn(__fmul_rn((float)__ldg(r0 + s0), c0), __fmul_rn((float)__ldg(r0 + s1), f));
        const float h1 = __fadd_rn(__fmul_rn((float)__ldg(r1 + s0), c0), __fmul_rn((float)__ldg(r1 + s1), f));
        return sat_u16(__fadd_rn(__fmul_rn(h0, ty.c0), __fmul_rn(h1, ty.c1)));
    };
    // window centre from a strided sample of the CTA's middle row
    {
        const int ym = (y0 + y1) >> 1, x = (int)(((long long)tid * dw) / kHistThreads);
        unsigned int v;
        if (RESIZE) {
            const Tap ty = ytap(ym);
            v = pixel(s + (size_t)ty.s0 * sw, s + (size_t)ty.s1 * sw, ty, x);
        } else {
            v = __ldg(s + (size_t)ym * sw + x);
        }
        const unsigned int lo = __reduce_min_sync(0xffffffffu, v), hi = __reduce_max_sync(0xffffffffu, v);
        if (lane == 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    }
    __syncthreads();
    const int centre = (int)((s_lo + s_hi) >> 1);
    const unsigned int wbase = (unsigned)min(max(centre - kWinBins / 2, 0), 65536 - kWinBins) & ~1u;
    __syncthreads();
    if (tid == 0) { s_lo = 0xffffu; s_hi = 0u; }
    __syncthreads();
    unsigned int vlo = 0xffffu, vhi = 0u;
    auto count = [&](unsigned int v) {
        vlo = min(vlo, v); vhi = max(vhi, v);
        const unsigned int d = v - wbase;
        if (d < (unsigned)kWinBins) atomicAdd(&win[d >> 1], (d & 1) ? 0x10000u : 1u);
        else atomicAdd(&gh[v], 1u);
    };
    // per-warp staging of the two source rows of an output row (coalesced 128-bit loads, then 2-byte LDS taps)
    uint16_t* stage = reinterpret_cast<uint16_t*>(xt + ((dw + 1) & ~1)) + (size_t)wrp * 2 * srow;   // 16-byte aligned; srow = sw rounded up to 8
    for (int y = y0 + wrp; y < y1; y += kHistThreads / 32) {
        if (RESIZE) {
            uint16_t* out_row = resized + ((size_t)b * dh + y) * dw;
            const Tap ty = ytap(y);
            const uint16_t* r0 = s + (size_t)ty.s0 * sw;
            const uint16_t* r1 = s + (size_t)ty.s1 * sw;
            __syncwarp();
            if (vec_rows) {
                for (int k = lane; k < (sw >> 3); k += 32) {
                    reinterpret_cast<uint4*>(stage)[k] = __ldg(reinterpret_cast<const uint4*>(r0) + k);
                    reinterpret_cast<uint4*>(stage + srow)[k] = __ldg(reinterpret_cast<const uint4*>(r1) + k);
                }
            } else {
                for (int k = lane; k < sw; k += 32) { stage[k] = __ldg(r0 + k); stage[srow + k] = __ldg(r1 + k); }
            }
            __syncwarp();
            const uint16_t* a0 = stage;
            const uint16_t* a1 = stage + srow;
            const float cy0 = ty.c0, cy1 = ty.c1;
            auto px = [&](int x) -> unsigned int {
                const uint2 t = xt[x];
                const int s0 = t.x & 0xffff, s1 = t.x >> 16;
                const float f = __uint_as_float(t.y), c0 = __fsub_rn(1.0f, f);
                const float h0 = __fadd_rn(__fmul_rn((float)a0[s0], c0), __fmul_rn((float)a0[s1], f));
                const float h1 = __fadd_rn(__fmul_rn((float)a1[s0], c0), __fmul_rn((float)a1[s1], f));
                return sat_u16(__fadd_rn(__fmul_rn(h0, cy0), __fmul_rn(h1, cy1)));
            };
            constexpr int U = 4;
            int x0 = lane;
            for (; x0 + 32 * (U - 1) < dw; x0 += 32 * U) {            // unguarded fast path
                unsigned int v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) v[u] = px(x0 + 32 * u);
#pragma unroll
                for (int u = 0; u < U; ++u) { out_row[x0 + 32 * u] = (uint16_t)v[u]; count(v[u]); }
            }
            for (; x0 < dw; x0 += 32) { const unsigned int v = px(x0); out_row[x0] = (uint16_t)v; count(v); }
        } else {
            const uint16_t* r0 = s + (size_t)y * sw;
            for (int x = lane; x < dw; x += 32) count(__ldg(r0 + x));
        }
    }
    vlo = __reduce_min_sync(0xffffffffu, vlo); vhi = __reduce_max_sync(0xffffffffu, vhi);
    if (lane == 0 && vlo <= vhi) { atomicMin(&s_lo, vlo); atomicMax(&s_hi, vhi); }
    __syncthreads();
    const unsigned int lo = s_lo, hi = s_hi;
    if (lo <= hi) {
        // sparse merge of the touched part of the window
        const int w0 = (int)max((int)(lo - wbase), 0) >> 1, w1 = min((int)((hi - wbase) >> 1), kWinWords - 1);
        if (hi >= wbase && lo < wbase + kWinBins)
            for (int i = w0 + tid; i <= w1; i += kHistThreads) {
                const unsigned int w = win[i];
                if (w & 0xffffu) atomicAdd(&gh[wbase + 2 * i], w & 0xffffu);
                if (w >> 16) atomicAdd(&gh[wbase + 2 * i + 1], w >> 16);
            }
        if (tid == 0) { atomicMin(&meta[b], lo); atomicMax(&meta[B + b], hi); }
    }
}

// K2b: p2 / p98 from the exact histogram: one CTA per frame scans only the frame's [vmin, vmax] bins.
__global__ void __launch_bounds__(1024) percentile_from_hist_kernel(const unsigned int* __restrict__ hist,
                                                                    const unsigned int* __restrict__ meta, int B, int n,
                                                                    double* __restrict__ out_p, int rep3,
                                                                    float2* __restrict__ glut, int2* __restrict__ lutmeta) {
    __shared__ unsigned int warp_tot[32];
    __shared__ float found[4];
    __shared__ double s_p[2];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const unsigned int vmin = min(meta[b], 65535u), vmax = min(meta[B + b], 65535u);
    const int range = (vmax >= vmin) ? (int)(vmax - vmin + 1) : 0;
    const int span = (range + 1023) / 1024;                      // consecutive bins per thread (<= 64)
    const unsigned int* h = hist + (size_t)b * 65536;
    const int first = (int)vmin + tid * span;
    unsigned int sum = 0;
    for (int k = 0; k < span; ++k) { const int v = first + k; if (v <= (int)vmax) sum += __ldg(h + v); }
    unsigned int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[wrp] = incl;
    __syncthreads();
    if (wrp == 0) {
        unsigned int w = warp_tot[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        warp_tot[lane] = wi - w;
    }
    __syncthreads();
    const unsigned int excl = warp_tot[wrp] + incl - sum;
    unsigned int k[2]; double g[2];
    percentile_ranks(n, 2.0, &k[0], &g[0]);
    percentile_ranks(n, 98.0, &k[1], &g[1]);
    const unsigned int ranks[4] = {k[0], min(k[0] + 1, (unsigned)n - 1), k[1], min(k[1] + 1, (unsigned)n - 1)};
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (ranks[r] >= excl && ranks[r] < excl + sum) {
            unsigned int c = excl;
            for (int q = 0; q < span; ++q) {
                c += __ldg(h + first + q);
                if (ranks[r] < c) { found[r] = (float)(first + q); break; }
            }
        }
    }
    __syncthreads();
    if (tid == 0) {
        s_p[0] = lerp_percentile(found[0], found[1], g[0]);
        s_p[1] = lerp_percentile(found[2], found[3], g[1]);
        out_p[2 * b] = s_p[0]; out_p[2 * b + 1] = s_p[1];
    }
    __syncthreads();
    build_norm_lut(b, s_p[0], s_p[1], rep3, glut, lutmeta);
}

// ------------------------------------------------------------------ channel collapse (utils/preprocessing.py:13-19)
// flag[b] = 1 iff np.allclose(c0, c1) and np.allclose(c0, c2)   (rtol 1e-5, atol 1e-8, fp32)
__device__ __forceinline__ bool is_close(float a, float b) {
    const bool fin = isfinite(b);
    const bool le = fabsf(__fsub_rn(a, b)) <= __fadd_rn(1e-8f, __fmul_rn(1e-5f, fabsf(b)));
    return (le && fin) || (a == b);
}

__global__ void __launch_bounds__(256) channels_close_kernel(const float* __restrict__ x, int n, int* __restrict__ flag) {
    // grid: (chunks, B); flag pre-set to 1; any violation clears it (idempotent store -> deterministic)
    const int b = blockIdx.y;
    const float* c0 = x + (size_t)b * 3 * n;
    bool ok = true;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float a = __ldg(c0 + i);
        ok = ok && is_close(a, __ldg(c0 + n + i)) && is_close(a, __ldg(c0 + 2 * (size_t)n + i));
    }
    if (!__all_sync(0xffffffffu, ok) && (threadIdx.x & 31) == 0) flag[b] = 0;
}

__global__ void set_int_kernel(int* p, int n, int v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// the plane enhance_thermal_contrast works on: channel 0, or fp32 gray (no FMA), or the raw array
__device__ __forceinline__ float plane_value(const float* __restrict__ img, int n, int channels, int collapse_to_c0, int i) {
    if (channels != 3 || collapse_to_c0) return __ldg(img + i);
    return gray3(__ldg(img + i), __ldg(img + n + i), __ldg(img + 2 * (size_t)n + i));
}

// ------------------------------------------------------------------ K2c: percentiles of arbitrary float data
// np.percentile(plane, (2, 98)) (utils/preprocessing.py:22) on float data, exact, in three small kernels -- the same
// scheme as the medians of t3d_metrics.cu:
//   F1 sample 4096 values (1024 jittered-stride quads), bracket each quantile's rank by two sample order statistics
//      9 sigma apart (monotone uint32 keys);
//   F2 one pass over the plane: count NaNs and the values below each bracket, collect the few percent inside;
//   F3 one CTA per image selects the exact order statistics among the candidates (radix select in shared memory) and
//      applies numpy's fp64 two-sided lerp.  If a bracket misses, or candidates overflow, that image falls back to a
//      full 3-pass radix select per rank over the plane: slower, same bits.
constexpr int kFSamp = 4096;
constexpr int kFCandCap = 32768;     // candidates per (image, window)
constexpr int kFCtaCand = 2048;      // staged per CTA per window
constexpr int kFThreads = 256;
constexpr int kFChunks = 24;

struct FpctWs {
    unsigned int* bracket;   // [B][4]  lo2, hi2, lo98, hi98 (keys, inclusive; lo > hi: no bracket)
    int* counters;           // [B][8]  n_nan, below2, below98, ncand2, ncand98, overflow, -, -
    unsigned int* cand;      // [B][2][kFCandCap]
    size_t total;
};
FpctWs fpct_ws(void* base, int B) {
    FpctWs w; size_t off = 0; char* p = reinterpret_cast<char*>(base);
    auto take = [&](size_t bytes) { char* r = p ? p + off : nullptr; off += t3d_align_up(bytes, 256); return r; };
    w.bracket = reinterpret_cast<unsigned int*>(take((size_t)B * 4 * sizeof(unsigned int)));
    w.counters = reinterpret_cast<int*>(take((size_t)B * 8 * sizeof(int)));
    w.cand = reinterpret_cast<unsigned int*>(take((size_t)B * 2 * kFCandCap * sizeof(unsigned int)));
    w.total = off;
    return w;
}

__global__ void __launch_bounds__(t3d_select::kThreads, 1)
fpct_sample_kernel(const float* __restrict__ x, int n, int channels, const int* __restrict__ close_flag,
                   unsigned int* __restrict__ bracket, float q_lo, float q_hi) {
    __shared__ float key[kFSamp];
    __shared__ t3d_select::Smem sm;
    __shared__ int s_valid;
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* img = x + (size_t)b * channels * n;
    const int collapse = (channels == 3) ? close_flag[b] : 0;
    const int count = (channels == 3) ? n : n * channels;
    const int m = min(count, kFSamp);
    if (tid == 0) s_valid = 0;
    __syncthreads();
    int nv = 0;
#pragma unroll
    for (int q = 0; q < kFSamp / t3d_select::kThreads; ++q) {
        const int k = q * t3d_select::kThreads + tid;
        float v = __int_as_float(0x7fc00000);                 // NaN = not part of the sample
        if (k < m) {
            int i = k;
            if (count > kFSamp) {
                const int l = k >> 2, qstride = (count >> 2) / (kFSamp >> 2);
                i = 4 * (l * qstride + (int)((((unsigned)l * 2654435761u) >> 8) % (unsigned)qstride)) + (k & 3);
            }
            v = plane_value(img, n, channels, collapse, i);
        }
        key[k] = v;
        nv += !isnan(v);
    }
    nv = __reduce_add_sync(0xffffffffu, nv);
    if ((tid & 31) == 0) atomicAdd(&s_valid, nv);
    __syncthreads();
    const int mv = s_valid;                                    // block-uniform
    auto get = [&](int i, float* v) { *v = key[i]; return !isnan(key[i]); };
    for (int w = 0; w < 2; ++w) {
        unsigned int lo = 1u, hi = 0u;                         // no bracket -> F3 falls back
        if (mv >= 64) {
            const float q = w ? q_hi : q_lo;                  // quantile as a fraction (0.02 / 0.98 for enhance_thermal_contrast)
            const int r = (int)(q * (float)(mv - 1) + 0.5f);
            const int d = (int)ceilf(9.0f * sqrtf((float)mv * q * (1.0f - q))) + 2;
            lo = t3d_select::float_key(t3d_select::select_rank(sm, kFSamp, (unsigned)max(r - d, 0), get));
            hi = t3d_select::float_key(t3d_select::select_rank(sm, kFSamp, (unsigned)min(r + d, mv - 1), get));
        }
        if (tid == 0) { bracket[4 * b + 2 * w] = lo; bracket[4 * b + 2 * w + 1] = hi; }
    }
}

__global__ void __launch_bounds__(kFThreads)
fpct_classify_kernel(const float* __restrict__ x, int n, int channels, const int* __restrict__ close_flag,
                     const unsigned int* __restrict__ bracket, int* __restrict__ counters, unsigned int* __restrict__ cand) {
    __shared__ unsigned int scand[2][kFCtaCand];
    __shared__ int scount[2], sbase[2], sred[3];
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const float* img = x + (size_t)b * channels * n;
    const int collapse = (channels == 3) ? close_flag[b] : 0;
    const int count = (channels == 3) ? n : n * channels;
    const uint4 br = __ldg(reinterpret_cast<const uint4*>(bracket) + b);
    const bool has2 = br.y >= br.x, has98 = br.w >= br.z;
    const unsigned int w2 = br.y - br.x, w98 = br.w - br.z;
    if (tid < 2) scount[tid] = 0;
    if (tid < 3) sred[tid] = 0;
    __syncthreads();
    int nan = 0, lt2 = 0, lt98 = 0;
    const int per = (count + gridDim.x - 1) / gridDim.x;
    const int i0 = blockIdx.x * per, i1 = min(i0 + per, count);
    for (int i = i0 + tid; i < i1; i += kFThreads) {
        const float v = plane_value(img, n, channels, collapse, i);
        if (isnan(v)) { ++nan; continue; }
        const unsigned int k = t3d_select::float_key(v);
        lt2 += k < br.x; lt98 += k < br.z;
        if (has2 && (k - br.x) <= w2) { const int slot = atomicAdd(&scount[0], 1); if (slot < kFCtaCand) scand[0][slot] = k; }
        if (has98 && (k - br.z) <= w98) { const int slot = atomicAdd(&scount[1], 1); if (slot < kFCtaCand) scand[1][slot] = k; }
    }
    nan = __reduce_add_sync(0xffffffffu, nan); lt2 = __reduce_add_sync(0xffffffffu, lt2); lt98 = __reduce_add_sync(0xffffffffu, lt98);
    if (lane == 0) { if (nan) atomicAdd(&sred[0], nan); if (lt2) atomicAdd(&sred[1], lt2); if (lt98) atomicAdd(&sred[2], lt98); }
    __syncthreads();
    int* c = counters + 8 * b;
    if (tid < 3 && sred[tid]) atomicAdd(&c[tid], sred[tid]);
    if (tid < 2) {
        const int k = scount[tid];
        if (k > kFCtaCand) { atomicExch(&c[5], 1); sbase[tid] = -1; }
        else {
            const int base = k ? atomicAdd(&c[3 + tid], k) : 0;
            if (base + k > kFCandCap) { atomicExch(&c[5], 1); sbase[tid] = -1; }
            else sbase[tid] = base;
        }
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int base = sbase[a], k = min(scount[a], kFCtaCand);
        if (base >= 0)
            for (int q = tid; q < k; q += kFThreads) cand[((size_t)b * 2 + a) * kFCandCap + base + q] = scand[a][q];
    }
}

// one CTA per image; out_p[b] = {p2, p98} as np.percentile(plane, (2, 98)) would return (fp64)
__global__ void __launch_bounds__(t3d_select::kThreads, 1)
fpct_select_kernel(const float* __restrict__ x, int n, int channels, const int* __restrict__ close_flag,
                   const int* __restrict__ counters, const unsigned int* __restrict__ cand, double* __restrict__ out_p,
                   double pct_lo, double pct_hi) {
    extern __shared__ unsigned int skeys[];                     // kFCandCap keys
    __shared__ t3d_select::Smem sm;
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* img = x + (size_t)b * channels * n;
    const int collapse = (channels == 3) ? close_flag[b] : 0;
    const int count = (channels == 3) ? n : n * channels;     // non-3-channel input: the whole array
    const int* c = counters + 8 * b;
    if (c[0] > 0) {                                             // np.percentile propagates NaN
        if (tid == 0) { out_p[2 * b] = __longlong_as_double(0x7ff8000000000000LL); out_p[2 * b + 1] = out_p[2 * b]; }
        return;
    }
    unsigned int k[2]; double g[2];
    percentile_ranks(count, pct_lo, &k[0], &g[0]);               // (2, 98) for enhance_thermal_contrast
    percentile_ranks(count, pct_hi, &k[1], &g[1]);
    float os[4];
    for (int w = 0; w < 2; ++w) {                               // block-uniform control flow throughout
        const unsigned int r0 = k[w], r1 = min(k[w] + 1, (unsigned)count - 1);
        const bool need1 = (g[w] != 0.0) && (r1 != r0);
        const int lt = c[1 + w], nc = c[3 + w];
        const bool ok = (c[5] == 0) && nc > 0 && nc <= kFCandCap && (int)r0 >= lt && (int)r1 < lt + nc;
        if (ok) {
            const unsigned int* src = cand + ((size_t)b * 2 + w) * kFCandCap;
            __syncthreads();
            for (int q = tid; q < nc; q += t3d_select::kThreads) skeys[q] = src[q];
            __syncthreads();
            auto get = [&](int i, float* v) { *v = t3d_select::key_float(skeys[i]); return true; };
            os[2 * w] = t3d_select::select_rank(sm, nc, r0 - (unsigned)lt, get);
            os[2 * w + 1] = need1 ? t3d_select::select_rank(sm, nc, r1 - (unsigned)lt, get) : os[2 * w];
        } else {                                                // fallback: full radix select over the plane
            auto get = [&](int i, float* v) { *v = plane_value(img, n, channels, collapse, i); return true; };
            os[2 * w] = t3d_select::select_rank(sm, count, r0, get);
            os[2 * w + 1] = need1 ? t3d_select::select_rank(sm, count, r1, get) : os[2 * w];
        }
    }
    if (tid == 0) {
        out_p[2 * b] = lerp_percentile(os[0], os[1], g[0]);
        out_p[2 * b + 1] = lerp_percentile(os[2], os[3], g[1]);
    }
}

// ------------------------------------------------------------------ K2d: clip-normalise in fp64, broadcast
// source is the resized u16 plane (train path); writes `rep` identical planes [B, rep, n]
__global__ void __launch_bounds__(256) normalize_u16_kernel(const uint16_t* __restrict__ src, const double* __restrict__ p,
                                                            float* __restrict__ dst, int n, int rep, int vec) {
    const int b = blockIdx.y;
    const double p2 = p[2 * b], den = __dsub_rn(p[2 * b + 1], p2);
    const uint16_t* s = src + (size_t)b * n;
    float* d = dst + (size_t)b * rep * n;
    const int n4 = vec ? (n >> 2) : 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        const ushort4 v = __ldg(reinterpret_cast<const ushort4*>(s) + i);
        const float4 o = make_float4(normalize_px((double)v.x, p2, den), normalize_px((double)v.y, p2, den),
                                     normalize_px((double)v.z, p2, den), normalize_px((double)v.w, p2, den));
        for (int r = 0; r < rep; ++r) stg_stream_f4(d + (size_t)r * n + 4 * (size_t)i, o);
    }
    if (blockIdx.x == 0) {
        for (int i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) {
            const float o = normalize_px((double)__ldg(s + i), p2, den);
            for (int r = 0; r < rep; ++r) d[(size_t)r * n + i] = o;
        }
    }
}

// Vector path of the train-path normalisation (W % 4 == 0), fused with the thermal-gradient statistics
// the loss needs (utils/loss.py:184-201,240-249): the frame's LUT over the integer values between floor(p2)
// and ceil(p98) (tabulated once per frame by the percentile kernel with the fp64 formula: same function, same
// bits, no per-pixel fp64 divide) is copied to shared memory, and the sums of |Dx gray|, |Dy gray| of the
// OUTPUT image are reduced per CTA into stats[b][band][0..1] (gray = 0.299 v + 0.587 v + 0.114 v in fp32
// when the output is replicated to 3 planes).
constexpr int kNormBands = 24;       // CTAs per frame == statistic partials per frame (T3D_STATS_TILES)
constexpr int kNormThreads = 256;
constexpr int kNormStageMax = 24 * 1024;  // staged band bytes: LUT 32 KB + band <= 56 KB per CTA, 4 CTAs per SM
// shapes whose bands the half-resolution pass handles: even bands of <= 16 rows, W / 2 columns <= one per thread,
// the band + two rows below fit the staging area
static bool norm_s2_supported(int H, int W) {
    const int rows_per = (H + kNormBands - 1) / kNormBands;
    return H >= 2 && W >= 8 && (W % 8) == 0 && (W / 2) <= kNormThreads && (rows_per % 2) == 0 && rows_per / 2 + 1 <= 9 /* kS2MaxPool */ &&
           (size_t)(rows_per + 2) * W * sizeof(uint16_t) <= (size_t)kNormStageMax;
}
constexpr int kNormWarps = kNormThreads / 32;

__device__ __forceinline__ float2 lds_f2(uint32_t saddr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(saddr));
    return v;
}

__device__ __forceinline__ uint2 lds_u2(uint32_t saddr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ unsigned int lds_h(uint32_t saddr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void cpa16(uint32_t dst_saddr, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst_saddr), "l"(src) : "memory");
}
__device__ __forceinline__ void cpa_commit_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

struct NormRow { float o[4], g[4]; };

// Frames whose p2..p98 range does not fit the LUT (> 4093 counts): direct fp64 evaluation, one pixel per thread.
template <int REP>
__device__ __noinline__ void normalize_band_direct(const uint16_t* __restrict__ s, float* __restrict__ d, int H, int W,
                                                   int y0, int y1, double p2, double den, bool do_stats, float& tx, float& ty) {
    const int n = H * W;
    auto val = [&](int i) { const float o = normalize_px((double)__ldg(s + i), p2, den); return make_float2(o, (REP == 3) ? gray3(o, o, o) : o); };
    for (int i = y0 * W + threadIdx.x; i < y1 * W; i += kNormThreads) {
        const int y = i / W, x = i - y * W;
        const float2 c = val(i);
#pragma unroll
        for (int r = 0; r < REP; ++r) d[(size_t)r * n + i] = c.x;
        if (do_stats) {
            if (x + 1 < W) tx += fabsf(val(i + 1).y - c.y);
            if (y + 1 < H) ty += fabsf(val(i + W).y - c.y);
        }
    }
}

// CTA = one band of rows of one frame; a warp takes a 128-column strip x a run of rows and marches down it:
// lane = 4 consecutive pixels (one 8-byte load per row, issued two rows ahead), the row below is looked up once
// and becomes the current row of the next iteration (two register sets, ping-pong), the right neighbour's gray
// comes from a shuffle (strip edge: one extra u16), outputs leave as 128-bit streaming stores.
// STAGED (W % 8 == 0, the band fits): the band's raw rows (+ the row below) and the LUT arrive in shared memory as
// ONE batch of cp.async copies -- a single exposed memory latency per CTA instead of one per marched row (the
// marches are short: 8 rows per warp at 384 rows), and the march itself then reads shared memory only.
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

template <int REP, bool STATS, bool STAGED, bool S2 = false>
__global__ void __launch_bounds__(kNormThreads, 4) normalize_stats_u16_kernel(const uint16_t* __restrict__ src,
                                                                           const double* __restrict__ p,
                                                                           float* __restrict__ dst, int H, int W,
                                                                           float* __restrict__ stats,
                                                                           const float2* __restrict__ glut,
                                                                           const int2* __restrict__ lutmeta, int nitems) {
    static_assert(!S2 || (STATS && STAGED), "half-resolution sums ride on the staged statistics variant");
    extern __shared__ float2 lut[];                 // {normalised value, its gray} for v in [floor(p2) - 1, ceil(p98) + 1]
    __shared__ float red[kNormWarps][4];
    __shared__ float edge[S2 ? kNormWarps + 1 : 1][kS2MaxPool];
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int n = H * W;
    // persistent over (frame, band) items: the grid is sized by the launcher (SMs x CTAs per SM), so the kernel
    // can be told to leave room on every SM for a concurrent kernel of another stream
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int b = item / kNormBands, band = item - b * kNormBands;
    __syncthreads();                                                  // previous item's LUT / red are no longer read
    const int2 lm = lutmeta[b];
    const int lom1 = lm.x, range = lm.y;
    const uint16_t* __restrict__ s = src + (size_t)b * n;
    float* __restrict__ d = dst + (size_t)b * REP * n;
    const int rows_per = (H + kNormBands - 1) / kNormBands;
    const int y0 = band * rows_per, y1 = min(y0 + rows_per, H);
    float tx = 0.f, ty = 0.f, tx2 = 0.f, ty2 = 0.f;
    if (range <= 0) {                                                 // block-uniform: no LUT for this frame
        const double p2 = p[2 * b], den = __dsub_rn(p[2 * b + 1], p2);
        normalize_band_direct<REP>(s, d, H, W, y0, y1, p2, den, STATS, tx, ty);
        if (S2) {
            auto gray = [&](int i) { const float o = normalize_px((double)__ldg(s + i), p2, den); return (REP == 3) ? gray3(o, o, o) : o; };
            half_res_band_sums(y0, y1, H, W, edge, [&](int I, int J) {
                const int i = 2 * I * W + 2 * J;
                return 0.25f * (((gray(i) + gray(i + 1)) + gray(i + W)) + gray(i + W + 1));
            }, tx2, ty2);
        }
    } else {
        const uint32_t sraw = (uint32_t)__cvta_generic_to_shared(lut) + (uint32_t)kLutMax * 8u;   // STAGED: rows [y0, yl)
        if (STAGED) {
            const uint32_t slut = (uint32_t)__cvta_generic_to_shared(lut);
            const char* gl = reinterpret_cast<const char*>(glut + (size_t)b * kLutMax);
            for (int k = tid; k < (range + 1) / 2; k += kNormThreads) cpa16(slut + 16u * k, gl + 16 * (size_t)k);
            const int yl = STATS ? min(y1 + (S2 ? 2 : 1), H) : y1;      // + the row(s) below: vertical differences
            const int nchunk = ((yl - y0) * W) >> 3;                  // the band is one contiguous block of the frame
            const char* gs = reinterpret_cast<const char*>(s + (size_t)y0 * W);
            for (int k = tid; k < nchunk; k += kNormThreads) cpa16(sraw + 16u * k, gs + 16 * (size_t)k);
            cpa_commit_wait_all();
        } else {
            const float4* g4 = reinterpret_cast<const float4*>(glut + (size_t)b * kLutMax);
            float4* l4 = reinterpret_cast<float4*>(lut);
            for (int k = tid; k < (range + 1) / 2; k += kNormThreads) l4[k] = __ldg(g4 + k);
        }
        __syncthreads();
        // lookup in the byte-address domain: addr = clamp(8 v + bias, first entry, last entry)
        const int a_lo = (int)(uint32_t)__cvta_generic_to_shared(lut), a_hi = a_lo + 8 * (range - 1), a_bias = a_lo - 8 * lom1;
        auto look = [&](unsigned int v8) -> float2 { return lds_f2((uint32_t)min(max((int)v8 + a_bias, a_lo), a_hi)); };
        auto lookup = [&](const uint2 q, NormRow& r) {
            const float2 a = look((q.x << 3) & 0x7fff8u), bq = look((q.x >> 13) & 0x7fff8u);
            const float2 c = look((q.y << 3) & 0x7fff8u), e = look((q.y >> 13) & 0x7fff8u);
            r.o[0] = a.x; r.o[1] = bq.x; r.o[2] = c.x; r.o[3] = e.x;
            r.g[0] = a.y; r.g[1] = bq.y; r.g[2] = c.y; r.g[3] = e.y;
        };
        const int nstrips = (W + 127) >> 7;
        const int RG = max(1, kNormWarps / nstrips);
        const int rpr = (y1 - y0 + RG - 1) / RG;
        const size_t rowb = (size_t)W * sizeof(uint16_t);
        for (int task = wrp; task < nstrips * RG; task += kNormWarps) {
            const int strip = task % nstrips, rg = task / nstrips;
            const int ya = y0 + rg * rpr, yb = min(ya + rpr, y1);
            const int x0 = (strip << 7) + 4 * lane;
            if (ya >= yb) continue;                                       // warp-uniform
            const bool active = x0 < W;
            const bool has_right = x0 + 4 < W;                            // a pixel right of this quad exists
            const bool edge_lane = STATS && active && has_right && lane == 31;   // right neighbour is in the next strip
            // rows [ya, ym) have a row below inside the image; row H - 1 (if it is ours) is the zero-padded one
            const int ym = STATS ? min(yb, H - 1) : ya;
            const int last = STATS ? min(yb, H - 1) : yb - 1;             // last row that is fetched
            const char* ld = reinterpret_cast<const char*>(s + (size_t)ya * W + (active ? x0 : 0));
            uint32_t lds_ = sraw + 2u * (uint32_t)((ya - y0) * W + (active ? x0 : 0));
            float* out = d + (size_t)ya * W + x0;
            auto fetch = [&](int y, uint2& q, unsigned int& hq) {          // raw quad (+ strip-edge pixel) of row y
                if (y <= last) {
                    if (STAGED) {
                        q = lds_u2(lds_);
                        if (edge_lane) hq = lds_h(lds_ + 8u);
                    } else {
                        q = __ldg(reinterpret_cast<const uint2*>(ld));
                        if (edge_lane) hq = __ldg(reinterpret_cast<const uint16_t*>(ld) + 4);
                    }
                }
                ld += rowb; lds_ += (uint32_t)rowb;
            };
            auto right_gray = [&](const NormRow& r, unsigned int hq) -> float {   // gray right of the quad (dx = 0 at the image edge)
                float gr = __shfl_down_sync(0xffffffffu, r.g[0], 1);
                if (edge_lane) gr = look((hq << 3) & 0x7fff8u).y;
                return has_right ? gr : r.g[3];
            };
            auto emit = [&](const NormRow& c) {
                if (active) {
                    const float4 o = make_float4(c.o[0], c.o[1], c.o[2], c.o[3]);
#pragma unroll
                    for (int r = 0; r < REP; ++r) stg_stream_f4(out + (size_t)r * n, o);
                }
                out += W;
            };
            auto dx_sum = [&](const NormRow& c, float gr) {
                return fabsf(c.g[1] - c.g[0]) + fabsf(c.g[2] - c.g[1]) + fabsf(c.g[3] - c.g[2]) + fabsf(gr - c.g[3]);
            };
            auto dy_sum = [&](const NormRow& c, const NormRow& nx) {
                return fabsf(nx.g[0] - c.g[0]) + fabsf(nx.g[1] - c.g[1]) + fabsf(nx.g[2] - c.g[2]) + fabsf(nx.g[3] - c.g[3]);
            };
            uint2 q0 = make_uint2(0u, 0u), q1 = q0, q2 = q0; unsigned int h0 = 0u, h1 = 0u, h2 = 0u;
            fetch(ya, q0, h0); fetch(ya + 1, q1, h1); fetch(ya + 2, q2, h2);
            NormRow A, Bq;
            lookup(q0, A);
            float grA = STATS ? right_gray(A, h0) : 0.f, grB = 0.f;
            float sx = 0.f, sy = 0.f;
            if (STATS) {
                // rows with a row below: A = row y, q1 = raw of row y + 1, q2 = raw of row y + 2
                int y = ya;
                for (; y + 1 < ym; y += 2) {
                    lookup(q1, Bq); grB = right_gray(Bq, h1); fetch(y + 3, q1, h1);
                    emit(A); sx += dx_sum(A, grA); sy += dy_sum(A, Bq);
                    lookup(q2, A); grA = right_gray(A, h2); fetch(y + 4, q2, h2);
                    emit(Bq); sx += dx_sum(Bq, grB); sy += dy_sum(Bq, A);
                }
                if (y < ym) {                                             // odd row count: one more row with a row below
                    lookup(q1, Bq); grB = right_gray(Bq, h1);
                    emit(A); sx += dx_sum(A, grA); sy += dy_sum(A, Bq);
                    A = Bq; grA = grB;
                    ++y;
                }
                if (y < yb) { emit(A); sx += dx_sum(A, grA); }            // the image's last row: dy = 0
                if (active) { tx += sx; ty += sy; }
            } else {
                int y = ya;
                for (; y + 1 < yb; y += 2) {
                    emit(A); lookup(q1, A); fetch(y + 3, q1, h1);
                    emit(A); lookup(q2, A); fetch(y + 4, q2, h2);
                }
                if (y < yb) emit(A);
            }
        }
        if (S2) {                                                         // the staged band + LUT are still in shared memory
            half_res_band_sums(y0, y1, H, W, edge, [&](int I, int J) {
                const uint32_t a = sraw + 2u * (uint32_t)((2 * I - y0) * W + 2 * J);
                unsigned int r0, r1;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r0) : "r"(a));
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r1) : "r"(a + 2u * (uint32_t)W));
                const float g00 = look((r0 << 3) & 0x7fff8u).y, g01 = look((r0 >> 13) & 0x7fff8u).y;
                const float g10 = look((r1 << 3) & 0x7fff8u).y, g11 = look((r1 >> 13) & 0x7fff8u).y;
                return 0.25f * (((g00 + g01) + g10) + g11);
            }, tx2, ty2);
        }
    }
    if (STATS) {
        tx = warp_sum(tx); ty = warp_sum(ty);
        if (S2) { tx2 = warp_sum(tx2); ty2 = warp_sum(ty2); }
        if (lane == 0) { red[wrp][0] = tx; red[wrp][1] = ty; red[wrp][2] = tx2; red[wrp][3] = ty2; }
        __syncthreads();
        if (tid < 4) {
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < kNormWarps; ++w) v += red[w][tid];
            stats[((size_t)b * kNormBands + band) * 4 + tid] = v;       // [2], [3]: the half-resolution sums (S2), else 0
        }
    }
    }   // items
}

// float source [B, channels, n] (drop-in enhance_thermal_contrast); rep output planes
__global__ void __launch_bounds__(256) normalize_f32_kernel(const float* __restrict__ x, int n, int channels,
                                                            const int* __restrict__ close_flag,
                                                            const double* __restrict__ p, float* __restrict__ dst,
                                                            int rep, int count) {
    const int b = blockIdx.y;
    const double p2 = p[2 * b], den = __dsub_rn(p[2 * b + 1], p2);
    const float* img = x + (size_t)b * channels * n;
    const int collapse = (channels == 3) ? close_flag[b] : 0;
    float* d = dst + (size_t)b * rep * count;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const float o = normalize_px((double)plane_value(img, n, channels, collapse, i), p2, den);
        for (int r = 0; r < rep; ++r) d[(size_t)r * count + i] = o;
    }
}

// ------------------------------------------------------------------ fixed range (utils/preprocessing.py:47-62), fp32 throughout
__global__ void __launch_bounds__(256) fixed_range_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n,
                                                          size_t plane, const int* __restrict__ close_flag,
                                                          int normalized) {
    // close_flag (3-channel input whose channels are np.allclose): every output plane is f(channel 0)
    const bool collapse = close_flag && close_flag[0];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float v = __ldg(x + (collapse ? i % plane : i));
        if (normalized) v = __fmul_rn(v, 65535.0f);
        // np.clip propagates NaN; fminf/fmaxf would not
        const float c = isnan(v) ? v : fminf(fmaxf(v, 21800.0f), 25000.0f);
        y[i] = __fdiv_rn(__fsub_rn(c, 21800.0f), 3200.0f);
    }
}

// ------------------------------------------------------------------ torch bilinear resample (align_corners=False)
// F.interpolate(x, size, mode='bilinear', align_corners=False) as train_thermal_dustr.py:234-271,465-481 applies
// it to the pseudo-GT pointmaps ([H,W,3] AoS -> permuted to NCHW there; here read and written in place as AoS)
// and confidences.  Taps and weights: btap / blerp (t3d_bilinear.cuh).
__global__ void __launch_bounds__(256) interp_bilinear_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                              int B, int C, int sh, int sw, int dh, int dw) {
    const float ry = bscale(sh, dh), rx = bscale(sw, dw);
    const size_t total = (size_t)B * dh * dw;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(idx % dw);
        const size_t t = idx / dw;
        const int y = (int)(t % dh);
        const int b = (int)(t / dh);
        const BTap ty = btap(y, sh, ry), tx = btap(x, sw, rx);
        const float* p = src + (size_t)b * sh * sw * C;
        for (int c = 0; c < C; ++c) {
            const float v00 = __ldg(p + ((size_t)ty.i0 * sw + tx.i0) * C + c), v01 = __ldg(p + ((size_t)ty.i0 * sw + tx.i1) * C + c);
            const float v10 = __ldg(p + ((size_t)ty.i1 * sw + tx.i0) * C + c), v11 = __ldg(p + ((size_t)ty.i1 * sw + tx.i1) * C + c);
            dst[idx * C + c] = blerp(v00, v01, v10, v11, ty, tx);
        }
    }
}

int grid_for(size_t n, int threads, int per_sm = 8) {
    const size_t need = (n + threads - 1) / threads;
    const size_t cap = (size_t)t3d_sm_count() * per_sm;
    return (int)(need < cap ? (need ? need : 1) : cap);
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int t3d_resize_bilinear(const void* src, void* dst, int mode, int B, int src_h, int src_w,
                        int dst_h, int dst_w, void* stream) {
    T3D_REQUIRE(src && dst, "NULL pointer");
    T3D_REQUIRE(B >= 1 && src_h >= 1 && src_w >= 1 && dst_h >= 1 && dst_w >= 1, "bad dims");
    T3D_REQUIRE(mode >= 0 && mode <= 2, "mode must be 0 (u16->u16), 1 (u16->/65535->f32) or 2 (f32->f32)");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int grid = grid_for((size_t)B * dst_h * dst_w, 256);
    if (mode == 0) T3D_LAUNCH("resize_bilinear_kernel", st, resize_bilinear_kernel<0><<<grid, 256, 0, st>>>(src, dst, B, src_h, src_w, dst_h, dst_w));
    else if (mode == 1) T3D_LAUNCH("resize_bilinear_kernel", st, resize_bilinear_kernel<1><<<grid, 256, 0, st>>>(src, dst, B, src_h, src_w, dst_h, dst_w));
    else T3D_LAUNCH("resize_bilinear_kernel", st, resize_bilinear_kernel<2><<<grid, 256, 0, st>>>(src, dst, B, src_h, src_w, dst_h, dst_w));
    return T3D_OK;
}

int t3d_resize_nearest_f32(const float* src, float* dst, int B, int src_h, int src_w, int dst_h, int dst_w,
                           void* stream) {
    T3D_REQUIRE(src && dst, "NULL pointer");
    T3D_REQUIRE(B >= 1 && src_h >= 1 && src_w >= 1 && dst_h >= 1 && dst_w >= 1, "bad dims");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("resize_nearest_kernel", st, resize_nearest_kernel<<<grid_for((size_t)B * dst_h * dst_w, 256), 256, 0, st>>>(src, dst, B, src_h, src_w, dst_h, dst_w));
    return T3D_OK;
}

size_t t3d_preprocess_workspace_bytes(int B, int dst_h, int dst_w) {
    if (B < 1 || dst_h < 1 || dst_w < 1) return 0;
    return pre_ws_layout(nullptr, B, dst_h, dst_w).total;
}

int t3d_preprocess_train_u16(const uint16_t* raw, int B, int src_h, int src_w, int dst_h, int dst_w,
                             float* out, int out_channels, unsigned int* hist, double* percentiles,
                             float* grad_stats, int stats_scales, int shared,
                             void* workspace, size_t workspace_bytes, int phase, void* stream) {
    T3D_REQUIRE(phase == T3D_PHASE_ALL || phase == T3D_PHASE_SAMPLE || phase == T3D_PHASE_REST, "bad phase %d", phase);
    T3D_REQUIRE(stats_scales == 1 || stats_scales == 2, "stats_scales must be 1 or 2, got %d", stats_scales);
    T3D_REQUIRE(phase == T3D_PHASE_ALL || hist == nullptr, "phases are a feature of the sampled-window path (hist == NULL)");
    T3D_REQUIRE(raw && out && percentiles && workspace, "NULL pointer");
    T3D_REQUIRE(B >= 1 && src_h >= 1 && src_w >= 1 && dst_h >= 1 && dst_w >= 1, "bad dims");
    T3D_REQUIRE(out_channels == 1 || out_channels == 3, "out_channels must be 1 or 3");
    T3D_REQUIRE((size_t)dst_h * dst_w < (1u << 30), "frame too large");
    T3D_REQUIRE(src_w <= 65535 && src_h <= 65535, "source frame too large (<= 65535 x 65535)");
    const PreWs w = pre_ws_layout(workspace, B, dst_h, dst_w);
    if (workspace_bytes < w.total) {
        t3d_set_error("workspace too small");
        return T3D_ERR_WORKSPACE;
    }
    T3D_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint16_t* resized = w.resized;
    const int npx = dst_h * dst_w;
    unsigned int* meta = w.meta;
    const bool same = (src_h == dst_h && src_w == dst_w);
    const int rep3 = (out_channels == 3);
    if (hist == nullptr) {
        // percentiles from sampled value windows: no per-pixel histogram atomic (t3d_preprocess_bracket.cu)
        if (int rc = t3d_launch_bracket_percentiles(raw, B, src_h, src_w, dst_h, dst_w, same, w, rep3, percentiles, shared != 0, phase, st)) return rc;
        if (phase == T3D_PHASE_SAMPLE) return T3D_OK;
    } else {
        // exact 65 536-bin histogram (an output) -> percentiles
        if (!same) {
            const int tn = max(dst_w, dst_h);
            T3D_LAUNCH("build_taps_kernel", st, build_taps_kernel<<<(tn + 255) / 256, 256, 0, st>>>(src_h, src_w, dst_h, dst_w, w.gxt, w.gyt));
        }
        T3D_CUDA(cudaMemsetAsync(hist, 0, (size_t)B * 65536 * sizeof(unsigned int), st));
        T3D_CUDA(cudaMemsetAsync(meta, 0xff, (size_t)B * sizeof(unsigned int), st));            // vmin = 0xffffffff
        T3D_CUDA(cudaMemsetAsync(meta + B, 0, (size_t)(B + 1) * sizeof(unsigned int), st));     // vmax = 0
        T3D_REQUIRE(dst_w <= kHistMaxW, "frame too wide for the histogram path (dst_w <= 2044)");
        const int chunks = (dst_h + kHistRows - 1) / kHistRows;       // kHistRows * dst_w < 65 536: u16 bins cannot overflow
        const size_t stage_bytes = same ? 0 : (size_t)(kHistThreads / 32) * 2 * ((src_w + 7) & ~7) * sizeof(uint16_t);
        const size_t hsmem = (size_t)kWinWords * 4 + (same ? 0 : (size_t)((dst_w + 1) & ~1) * sizeof(uint2)) + stage_bytes;
        T3D_REQUIRE(hsmem <= 200 * 1024, "source rows too wide for the shared-memory staging (src_w <= ~9000)");
        if (int rc = t3d_set_max_dynamic_smem<resize_hist_u16_kernel<true>>(200 * 1024)) return rc;
        if (int rc = t3d_set_max_dynamic_smem<resize_hist_u16_kernel<false>>(200 * 1024)) return rc;
        if (same)
            T3D_LAUNCH("resize_hist_u16_kernel", st, resize_hist_u16_kernel<false><<<B * chunks, kHistThreads, hsmem, st>>>(
                raw, resized, hist, meta, w.gxt, w.gyt, B, src_h, src_w, dst_h, dst_w, chunks));
        else
            T3D_LAUNCH("resize_hist_u16_kernel", st, resize_hist_u16_kernel<true><<<B * chunks, kHistThreads, hsmem, st>>>(
                raw, resized, hist, meta, w.gxt, w.gyt, B, src_h, src_w, dst_h, dst_w, chunks));
        T3D_LAUNCH("percentile_from_hist_kernel", st, percentile_from_hist_kernel<<<B, 1024, 0, st>>>(
            hist, meta, B, npx, percentiles, rep3, w.lut, w.lutmeta));
    }
    const uint16_t* nsrc = same ? raw : resized;
    const int vec = (dst_w % 4 == 0) && t3d_aligned16(out) && ((reinterpret_cast<uintptr_t>(nsrc) & 7u) == 0);
    if (vec) {
        constexpr int kLutBytes = kLutMax * 8, kStagedBytes = kLutMax * 8 + kNormStageMax;
#define T3D_NORM_ATTR(REP_, ST_) \
        if (int rc = t3d_set_max_dynamic_smem<normalize_stats_u16_kernel<REP_, ST_, false>>(kLutBytes)) return rc; \
        if (int rc = t3d_set_max_dynamic_smem<normalize_stats_u16_kernel<REP_, ST_, true>>(kStagedBytes)) return rc
        T3D_NORM_ATTR(1, true); T3D_NORM_ATTR(3, true); T3D_NORM_ATTR(1, false); T3D_NORM_ATTR(3, false);
#undef T3D_NORM_ATTR
        if (int rc = t3d_set_max_dynamic_smem<normalize_stats_u16_kernel<1, true, true, true>>(kStagedBytes)) return rc;
        if (int rc = t3d_set_max_dynamic_smem<normalize_stats_u16_kernel<3, true, true, true>>(kStagedBytes)) return rc;
        constexpr int kNormCtasPerSm = 32;
        const int nitems = B * kNormBands;
        const int grid = min(nitems, t3d_sm_count() * kNormCtasPerSm);
        // half-resolution sums too (stats_scales == 2) where the shape allows: two rows below the band
        const bool s2 = grad_stats && stats_scales == 2 && norm_s2_supported(dst_h, dst_w);
        if (s2) T3D_REQUIRE(t3d_aligned16(nsrc), "half-resolution statistics need 16-byte aligned frames");
        const int band_rows = (dst_h + kNormBands - 1) / kNormBands + (s2 ? 2 : 1);  // + the row(s) below (gradient statistics)
        const size_t stage_bytes = (size_t)band_rows * dst_w * sizeof(uint16_t);
        const bool staged = (dst_w % 8 == 0) && stage_bytes <= (size_t)kNormStageMax && t3d_aligned16(nsrc);
#define T3D_NORM_LAUNCH(REP_, ST_) do { \
            if (staged) T3D_LAUNCH("normalize_stats_u16_kernel", st, (normalize_stats_u16_kernel<REP_, ST_, true><<<grid, kNormThreads, kLutMax * 8 + stage_bytes, st>>>( \
                nsrc, percentiles, out, dst_h, dst_w, grad_stats, w.lut, w.lutmeta, nitems))); \
            else T3D_LAUNCH("normalize_stats_u16_kernel", st, (normalize_stats_u16_kernel<REP_, ST_, false><<<grid, kNormThreads, kLutMax * 8, st>>>( \
                nsrc, percentiles, out, dst_h, dst_w, grad_stats, w.lut, w.lutmeta, nitems))); } while (0)
        if (s2) {           // implies staged
            if (out_channels == 3) T3D_LAUNCH("normalize_stats_u16_kernel", st, (normalize_stats_u16_kernel<3, true, true, true><<<grid, kNormThreads, kLutMax * 8 + stage_bytes, st>>>(
                nsrc, percentiles, out, dst_h, dst_w, grad_stats, w.lut, w.lutmeta, nitems)));
            else T3D_LAUNCH("normalize_stats_u16_kernel", st, (normalize_stats_u16_kernel<1, true, true, true><<<grid, kNormThreads, kLutMax * 8 + stage_bytes, st>>>(
                nsrc, percentiles, out, dst_h, dst_w, grad_stats, w.lut, w.lutmeta, nitems)));
        }
        else if (out_channels == 3) { if (grad_stats) T3D_NORM_LAUNCH(3, true); else T3D_NORM_LAUNCH(3, false); }
        else { if (grad_stats) T3D_NORM_LAUNCH(1, true); else T3D_NORM_LAUNCH(1, false); }
#undef T3D_NORM_LAUNCH
    } else {
        T3D_REQUIRE(grad_stats == nullptr, "grad_stats needs dst_w %% 4 == 0 (t3d_preprocess_stats_tiles() == 0 here)");
        dim3 grid((unsigned)min((npx / 4 + 255) / 256 + 1, 64), (unsigned)B);
        T3D_LAUNCH("normalize_u16_kernel", st, normalize_u16_kernel<<<grid, 256, 0, st>>>(nsrc, percentiles, out, npx, out_channels, 0));
    }
    return T3D_OK;
}

int t3d_preprocess_fallback_count(const void* workspace, int B, int dst_h, int dst_w, unsigned int* count_host, void* stream) {
    T3D_REQUIRE(workspace && count_host, "NULL pointer");
    T3D_REQUIRE(B >= 1 && dst_h >= 1 && dst_w >= 1, "bad dims");
    const PreWs w = pre_ws_layout(const_cast<void*>(workspace), B, dst_h, dst_w);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_CUDA(cudaMemcpyAsync(count_host, w.brhist + (size_t)B * 2 * kBrSlots, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    T3D_CUDA(cudaStreamSynchronize(st));
    return T3D_OK;
}

int t3d_preprocess_stats_scales(int dst_h, int dst_w) {
    return (dst_h >= 1 && dst_w >= 4 && dst_w % 4 == 0) ? (norm_s2_supported(dst_h, dst_w) ? 2 : 1) : 0;
}

int t3d_preprocess_stats_tiles(int dst_h, int dst_w) {
    return (dst_h >= 1 && dst_w >= 4 && dst_w % 4 == 0) ? kNormBands : 0;
}

// np.percentile(plane, (pct_lo, pct_hi)) of B float planes: sampled brackets -> counting / collecting pass -> exact
// select among the candidates (full radix select as the fallback); percentiles [B][2] float64.
static int run_float_percentiles(const float* x, int B, int channels, int n, const int* close_flags, double pct_lo, double pct_hi,
                                 double* percentiles, const FpctWs& w, cudaStream_t st) {
    const int count = (channels == 3) ? n : n * channels;
    T3D_CUDA(cudaMemsetAsync(w.counters, 0, (size_t)B * 8 * sizeof(int), st));
    if (int rc = t3d_set_max_dynamic_smem<fpct_select_kernel>(kFCandCap * (int)sizeof(unsigned int))) return rc;
    T3D_LAUNCH("fpct_sample_kernel", st, fpct_sample_kernel<<<B, t3d_select::kThreads, 0, st>>>(
        x, n, channels, close_flags, w.bracket, (float)(pct_lo / 100.0), (float)(pct_hi / 100.0)));
    dim3 gc((unsigned)max(1, min(kFChunks, (count + 4095) / 4096)), (unsigned)B);
    T3D_LAUNCH("fpct_classify_kernel", st, fpct_classify_kernel<<<gc, kFThreads, 0, st>>>(x, n, channels, close_flags, w.bracket, w.counters, w.cand));
    T3D_LAUNCH("fpct_select_kernel", st, fpct_select_kernel<<<B, t3d_select::kThreads, kFCandCap * sizeof(unsigned int), st>>>(
        x, n, channels, close_flags, w.counters, w.cand, percentiles, pct_lo, pct_hi));
    return T3D_OK;
}

/* np.percentile(x[b], (pct_lo, pct_hi)) for B float32 arrays of n values (method 'linear', float64 results);
 * workspace as t3d_contrast_normalize_workspace_bytes(B). */
int t3d_percentiles_f32(const float* x, int B, int n, double pct_lo, double pct_hi, double* percentiles,
                        void* workspace, size_t workspace_bytes, void* stream) {
    T3D_REQUIRE(x && percentiles && workspace, "NULL pointer");
    T3D_REQUIRE(B >= 1 && n >= 1 && (double)n < 2.0e9, "bad dims");
    T3D_REQUIRE(pct_lo > 0.0 && pct_lo < pct_hi && pct_hi < 100.0, "percentiles must satisfy 0 < lo < hi < 100");
    const FpctWs w = fpct_ws(workspace, B);
    if (workspace_bytes < w.total) { t3d_set_error("workspace too small"); return T3D_ERR_WORKSPACE; }
    T3D_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15u) == 0, "workspace must be 16-byte aligned");
    return run_float_percentiles(x, B, 1, n, nullptr, pct_lo, pct_hi, percentiles, w, reinterpret_cast<cudaStream_t>(stream));
}

size_t t3d_contrast_normalize_workspace_bytes(int B) {
    if (B < 1) return 0;
    return fpct_ws(nullptr, B).total;
}

int t3d_contrast_normalize_f32(const float* x, int B, int channels, int n, float* out, int out_channels,
                               double* percentiles, int* close_flags, void* workspace, size_t workspace_bytes,
                               void* stream) {
    T3D_REQUIRE(x && out && percentiles && close_flags && workspace, "NULL pointer");
    T3D_REQUIRE(B >= 1 && channels >= 1 && n >= 1, "bad dims");
    T3D_REQUIRE((double)channels * n < 2.0e9, "image too large");
    const FpctWs w = fpct_ws(workspace, B);
    if (workspace_bytes < w.total) { t3d_set_error("workspace too small"); return T3D_ERR_WORKSPACE; }
    T3D_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15u) == 0, "workspace must be 16-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int count = (channels == 3) ? n : n * channels;
    if (channels == 3) {
        T3D_LAUNCH("set_int_kernel", st, set_int_kernel<<<(B + 255) / 256, 256, 0, st>>>(close_flags, B, 1));
        dim3 g((unsigned)min((n + 255) / 256, 32), (unsigned)B);
        T3D_LAUNCH("channels_close_kernel", st, channels_close_kernel<<<g, 256, 0, st>>>(x, n, close_flags));
    }
    if (int rc = run_float_percentiles(x, B, channels, n, close_flags, 2.0, 98.0, percentiles, w, st)) return rc;
    dim3 g2((unsigned)min((count + 255) / 256, 64), (unsigned)B);
    T3D_LAUNCH("normalize_f32_kernel", st, normalize_f32_kernel<<<g2, 256, 0, st>>>(x, n, channels, close_flags, percentiles, out, out_channels, count));
    return T3D_OK;
}

int t3d_channels_close(const float* x, int B, int n, int* close_flags, void* stream) {
    T3D_REQUIRE(x && close_flags, "NULL pointer");
    T3D_REQUIRE(B >= 1 && n >= 1, "bad dims");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("set_int_kernel", st, set_int_kernel<<<(B + 255) / 256, 256, 0, st>>>(close_flags, B, 1));
    dim3 g((unsigned)min((n + 255) / 256, 32), (unsigned)B);
    T3D_LAUNCH("channels_close_kernel", st, channels_close_kernel<<<g, 256, 0, st>>>(x, n, close_flags));
    return T3D_OK;
}

int t3d_fixed_range_normalize(const float* x, float* y, size_t n, size_t plane, const int* close_flag,
                              int normalized, void* stream) {
    T3D_REQUIRE(x && y, "NULL pointer");
    if (n == 0) return T3D_OK;
    T3D_REQUIRE(plane >= 1, "bad plane size");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("fixed_range_kernel", st, fixed_range_kernel<<<grid_for(n, 256), 256, 0, st>>>(x, y, n, plane, close_flag, normalized));
    return T3D_OK;
}

int t3d_interp_bilinear_f32(const float* src, float* dst, int B, int channels_last, int src_h, int src_w,
                            int dst_h, int dst_w, void* stream) {
    T3D_REQUIRE(src && dst, "NULL pointer");
    T3D_REQUIRE(B >= 1 && channels_last >= 1 && src_h >= 1 && src_w >= 1 && dst_h >= 1 && dst_w >= 1, "bad dims");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("interp_bilinear_kernel", st, interp_bilinear_kernel<<<grid_for((size_t)B * dst_h * dst_w, 256), 256, 0, st>>>(
        src, dst, B, channels_last, src_h, src_w, dst_h, dst_w));
    return T3D_OK;
}

}  // extern "C"
