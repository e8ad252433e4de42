// t3d_preprocess_fixed.cu -- 16-bit radiometric frames -> resized thermal on the Freiburg fixed window, in one pass
// (sm_100a).
//
// enhance_thermal_fixed_range (utils/preprocessing.py:32-73) needs no statistic of the whole frame: every output pixel
// is a function of its own bilinear taps.  So the percentile chain's four launches (sample, resize + classify,
// percentiles, normalise) and its u16 intermediate collapse into one kernel that reads the source rows once, resizes,
// clips to [21800, 25000], normalises and writes the planes.  Both paths of the reference, bit-exact:
//   train     (data/dataset_loader.py:237-249): cv2.resize to u16 (round-half-even), raw counts, normalized=False;
//   inference (thermal_dustr_inference.py:42-52): /65535 in fp32, float resize, normalized=True (x 65535 back).
// Tap arithmetic: SURVEY.md Appendix B (no FMA contraction); the window arithmetic is fp32 as the reference's.
#include <algorithm>

#include "t3d_preprocess_internal.cuh"

namespace {

constexpr float kFrLo = 21800.0f, kFrHi = 25000.0f, kFrSpan = 3200.0f;   // utils/preprocessing.py:53-54
constexpr int kFrThreads = 256;
constexpr int kFrWarps = kFrThreads / 32;
constexpr int kFrU = 8;                      // consecutive output pixels per lane (two 128-bit stores per plane)
constexpr int kFrStrip = 32 * kFrU;          // output columns per warp
constexpr int kFrStageMax = 96 * 1024;       // staged source rows per CTA: 2 CTAs per SM

// the fixed window of one resized value v: train: v rounded to u16 first; inference: v is a resize of x / 65535
template <bool INFER>
__device__ __forceinline__ float fixed_window(float v) {
    const float x = INFER ? __fmul_rn(v, 65535.0f) : (float)sat_u16(v);
    const float c = fminf(fmaxf(x, kFrLo), kFrHi);                    // finite: resized u16 data
    return __fdiv_rn(__fsub_rn(c, kFrLo), kFrSpan);
}

// Any shape and alignment, no statistics: one thread per output pixel.
template <bool INFER>
__global__ void __launch_bounds__(256) fixed_range_scalar_kernel(const uint16_t* __restrict__ raw, float* __restrict__ out,
                                                                 int B, int sh, int sw, int dh, int dw, int rep) {
    const double scx = (double)sw / (double)dw, scy = (double)sh / (double)dh;
    const size_t n = (size_t)dh * dw, total = (size_t)B * n;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(idx % dw);
        const size_t t = idx / dw;
        const int y = (int)(t % dh);
        const int b = (int)(t / dh);
        const float o = fixed_window<INFER>(bilinear_at<uint16_t, INFER>(raw + (size_t)b * sh * sw, sw,
                                                                          linear_tap(y, sh, scy), linear_tap(x, sw, scx)));
        float* d = out + (size_t)b * rep * n + (size_t)y * dw + x;
        for (int r = 0; r < rep; ++r) d[(size_t)r * n] = o;
    }
}

// Vector path (dst_w % 4 == 0, 16-byte aligned output).  Persistent grid over (frame, band) items with the band split
// of normalize_stats_u16_kernel (kNormBands bands of ceil(H / kNormBands) rows), so that the thermal-gradient partials
// land in the same [B][kNormBands][4] slots the loss reads.
//   STAGED: the band's source rows (+ those of the row(s) below it that the statistics need) arrive in shared memory as
//           ONE batch of cp.async copies -- they are one contiguous block of the frame; else they are read from global.
//   H54:    the 5:4 horizontal geometry with compile-time taps (hpass54), staged only.
// A warp takes a 256-column strip x a run of rows and marches down it: lane = 8 consecutive output pixels; the
// horizontal pass of a source row is evaluated once and kept in registers for the (up to two) output rows that use it;
// outputs leave as 128-bit streaming stores.  STATS: sums of |Dx gray|, |Dy gray| of the output image, gray computed as
// in the percentile chain's LUT (gray3(v, v, v) for 3 planes); s2: the half-resolution sums too (half_res_band_sums).
template <bool H54, bool STAGED, bool INFER, bool STATS>
__global__ void __launch_bounds__(kFrThreads, 2)
fixed_range_march_kernel(const uint16_t* __restrict__ raw, float* __restrict__ out, float* __restrict__ stats,
                         int sh, int sw, int dh, int dw, int rep, int s2, int nitems, int taps_off) {
    static_assert(!H54 || STAGED, "the compile-time taps read staged rows");
    extern __shared__ __align__(16) unsigned char fr_smem[];
    __shared__ float red[kFrWarps][4];
    __shared__ float edge[kFrWarps + 1][kS2MaxPool];
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const double scx = (double)sw / (double)dw, scy = (double)sh / (double)dh;
    const size_t n = (size_t)dh * dw;
    const int rows_per = (dh + kNormBands - 1) / kNormBands;
    const int nstrips = (dw + kFrStrip - 1) / kFrStrip;
    const int RG = max(1, kFrWarps / nstrips);
    const uint32_t sbase = smem_u32(fr_smem);
    const bool rep3 = rep == 3;
    // !H54: the x taps of every output column, once per CTA: {first source column, bits of the second weight}
    uint2* xtab = reinterpret_cast<uint2*>(fr_smem + taps_off);
    if (!H54) {
        for (int x = tid; x < dw; x += kFrThreads) {
            const Tap t = linear_tap(x, sw, scx);
            xtab[x] = make_uint2((unsigned)t.s0, __float_as_uint(t.c1));
        }
    }
    #pragma unroll 1
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int b = item / kNormBands, band = item - b * kNormBands;
        const int y0 = band * rows_per, y1 = min(y0 + rows_per, dh);
        const int yl = min(y1 + (STATS ? (s2 ? 2 : 1) : 0), dh);          // rows evaluated: + the row(s) below
        const uint16_t* __restrict__ frame = raw + (size_t)b * sh * sw;
        float* __restrict__ d = out + (size_t)b * rep * n;
        float tx = 0.f, ty = 0.f, tx2 = 0.f, ty2 = 0.f;
        __syncthreads();                                                  // the previous item's rows / red are no longer read
        if (y0 < y1) {                                                    // block-uniform
            const int sr0 = linear_tap(y0, sh, scy).s0;
            if (STAGED) {
                const int sr1 = linear_tap(yl - 1, sh, scy).s1;
                const int nchunk = ((sr1 - sr0 + 1) * sw) >> 3;
                const char* g = reinterpret_cast<const char*>(frame + (size_t)sr0 * sw);
                for (int k = tid; k < nchunk; k += kFrThreads) cp_async16(sbase + 16u * k, g + 16 * (size_t)k);
                cp_async_commit();
                cp_async_wait<0>();
                __syncthreads();
            }
            // source value (row r, column c): / 65535 in fp32 on the inference path
            auto sv = [&](int r, int c) -> float {
                const float v = STAGED ? (float)lds_u16(sbase + 2u * (uint32_t)((r - sr0) * sw + c)) : (float)__ldg(frame + (size_t)r * sw + c);
                return INFER ? __fdiv_rn(v, 65535.0f) : v;
            };
            auto hval = [&](int r, const Tap& t) { return __fadd_rn(__fmul_rn(sv(r, t.s0), t.c0), __fmul_rn(sv(r, t.s1), t.c1)); };
            auto gray = [&](float o) { return rep3 ? gray3(o, o, o) : o; };
            // one output pixel from scratch (strip edges, the half-resolution pass)
            auto pixel = [&](int y, int x) {
                const Tap ty_ = linear_tap(y, sh, scy), tx_ = linear_tap(x, sw, scx);
                return fixed_window<INFER>(__fadd_rn(__fmul_rn(hval(ty_.s0, tx_), ty_.c0), __fmul_rn(hval(ty_.s1, tx_), ty_.c1)));
            };
            const int rpr = (y1 - y0 + RG - 1) / RG;
            #pragma unroll 1
            for (int task = wrp; task < nstrips * RG; task += kFrWarps) {
                const int strip = task % nstrips, rg = task / nstrips;
                const int ya = y0 + rg * rpr, yb = min(ya + rpr, y1);
                if (ya >= yb) continue;                                   // warp-uniform
                const int x0 = strip * kFrStrip + kFrU * lane;
                const int nv = max(0, min(kFrU, dw - x0));                // valid pixels of this lane (0, 4 or 8)
                const bool has_right = lane < 31 && x0 + kFrU < dw;       // the pixel right of this lane's 8 is in the strip
                const uint32_t h54_off = 20u * (uint32_t)(min(x0, dw - kFrU) / kFrU);     // H54: the lane's 10 source pixels
                auto hrow = [&](int r, float h[kFrU]) {
                    if (H54) {
                        hpass54<INFER>(sbase + 2u * (uint32_t)((r - sr0) * sw) + h54_off, h);
                    } else {
#pragma unroll
                        for (int u = 0; u < kFrU; ++u) {        // linear_tap's s1 and c0, rebuilt from s0 and c1
                            const uint2 e = xtab[min(x0 + u, dw - 1)];
                            Tap t; t.s0 = (int)e.x; t.s1 = min(t.s0 + 1, sw - 1); t.c1 = __uint_as_float(e.y); t.c0 = __fsub_rn(1.0f, t.c1);
                            h[u] = hval(r, t);
                        }
                    }
                };
                const int yc = STATS ? min(yb + 1, dh) : yb;              // + the row below: vertical differences
                float hA[kFrU], hB[kFrU], gp[kFrU];
                int tagA = -1, tagB = -1;
                float sx = 0.f, sy = 0.f;
                #pragma unroll 1
                for (int y = ya; y < yc; ++y) {
                    const Tap t = linear_tap(y, sh, scy);
                    if (t.s0 != tagA) {
                        if (t.s0 == tagB) {
#pragma unroll
                            for (int u = 0; u < kFrU; ++u) hA[u] = hB[u];
                        } else hrow(t.s0, hA);
                        tagA = t.s0;
                    }
                    if (t.s1 != tagB) {
                        if (t.s1 == tagA) {
#pragma unroll
                            for (int u = 0; u < kFrU; ++u) hB[u] = hA[u];
                        } else hrow(t.s1, hB);
                        tagB = t.s1;
                    }
                    float o[kFrU];
#pragma unroll
                    for (int u = 0; u < kFrU; ++u) o[u] = fixed_window<INFER>(__fadd_rn(__fmul_rn(hA[u], t.c0), __fmul_rn(hB[u], t.c1)));
                    if (y < yb && nv > 0) {
                        float* p = d + (size_t)y * dw + x0;
                        for (int r = 0; r < rep; ++r, p += n) {
                            stg_stream_f4(p, make_float4(o[0], o[1], o[2], o[3]));
                            if (nv > 4) stg_stream_f4(p + 4, make_float4(o[4], o[5], o[6], o[7]));
                        }
                    }
                    if (STATS) {
                        float g[kFrU];
#pragma unroll
                        for (int u = 0; u < kFrU; ++u) g[u] = gray(o[u]);
                        if (y > ya) {                                     // row y - 1 (ours) has this row below it
#pragma unroll
                            for (int u = 0; u < kFrU; ++u) if (u < nv) sy += fabsf(g[u] - gp[u]);
                        }
                        if (y < yb) {
                            const float gr = __shfl_down_sync(0xffffffffu, g[0], 1);
#pragma unroll
                            for (int u = 0; u < kFrU - 1; ++u) if (u + 1 < nv) sx += fabsf(g[u + 1] - g[u]);
                            if (has_right) sx += fabsf(gr - g[kFrU - 1]);
                        }
#pragma unroll
                        for (int u = 0; u < kFrU; ++u) gp[u] = g[u];
                    }
                }
                tx += sx; ty += sy;
            }
            if (STATS) {                                                  // |Dx| across the strip edges
                for (int k = tid; k < (nstrips - 1) * (y1 - y0); k += kFrThreads) {
                    const int y = y0 + k / (nstrips - 1), x = (k % (nstrips - 1) + 1) * kFrStrip;
                    tx += fabsf(gray(pixel(y, x)) - gray(pixel(y, x - 1)));
                }
            }
            if (STATS && s2) {
                half_res_band_sums(y0, y1, dh, dw, edge, [&](int I, int J) {
                    const int y = 2 * I, x = 2 * J;
                    return 0.25f * (((gray(pixel(y, x)) + gray(pixel(y, x + 1))) + gray(pixel(y + 1, x))) + gray(pixel(y + 1, x + 1)));
                }, tx2, ty2);
            }
        }
        if (STATS) {
            tx = warp_sum(tx); ty = warp_sum(ty);
            tx2 = warp_sum(tx2); ty2 = warp_sum(ty2);
            if (lane == 0) { red[wrp][0] = tx; red[wrp][1] = ty; red[wrp][2] = tx2; red[wrp][3] = ty2; }
            __syncthreads();
            if (tid < 4) {
                float v = 0.f;
#pragma unroll
                for (int w = 0; w < kFrWarps; ++w) v += red[w][tid];
                stats[((size_t)b * kNormBands + band) * 4 + tid] = v;     // [2], [3]: the half-resolution sums (s2), else 0
            }
        }
    }   // items
}

template <bool H54, bool STAGED, bool INFER, bool STATS>
int launch_march(const uint16_t* raw, float* out, float* stats, int B, int sh, int sw, int dh, int dw, int rep, int s2,
                 size_t stage_bytes, cudaStream_t st) {
    constexpr auto kernel = fixed_range_march_kernel<H54, STAGED, INFER, STATS>;
    if (int rc = t3d_set_max_dynamic_smem<kernel>(kFrStageMax)) return rc;
    const int nitems = B * kNormBands;
    const int grid = min(nitems, t3d_sm_count() * 2);
    const size_t taps_off = t3d_align_up(stage_bytes, 16);
    const size_t smem = taps_off + (H54 ? 0 : (size_t)dw * sizeof(uint2));
    T3D_REQUIRE(smem <= (size_t)kFrStageMax, "dst_w too large for the x-tap table (<= 12288)");
    T3D_LAUNCH("fixed_range_march_kernel", st, (kernel<<<grid, kFrThreads, smem, st>>>(raw, out, stats, sh, sw, dh, dw, rep, s2,
                                                                                     nitems, (int)taps_off)));
    return T3D_OK;
}

template <bool INFER>
int launch_fixed(const uint16_t* raw, float* out, float* stats, int B, int sh, int sw, int dh, int dw, int rep, int s2,
                 cudaStream_t st) {
    // source rows a band spans: output rows (band + the 2 below) x scale, + 3 for the taps' floors and the second tap
    const int rows_per = (dh + kNormBands - 1) / kNormBands;
    const int span = min(sh, (int)ceil((double)(rows_per + 2) * sh / dh) + 3);
    const size_t smem = (size_t)span * sw * sizeof(uint16_t);      // + the x-tap table unless H54
    const bool staged = (sw % 8 == 0) && t3d_aligned16(raw) && smem + (size_t)dw * sizeof(uint2) <= (size_t)kFrStageMax;
    const bool h54 = staged && sw * 4 == dw * 5 && dw % kFrU == 0;
    if (h54) return stats ? launch_march<true, true, INFER, true>(raw, out, stats, B, sh, sw, dh, dw, rep, s2, smem, st)
                          : launch_march<true, true, INFER, false>(raw, out, stats, B, sh, sw, dh, dw, rep, s2, smem, st);
    if (staged) return stats ? launch_march<false, true, INFER, true>(raw, out, stats, B, sh, sw, dh, dw, rep, s2, smem, st)
                             : launch_march<false, true, INFER, false>(raw, out, stats, B, sh, sw, dh, dw, rep, s2, smem, st);
    return stats ? launch_march<false, false, INFER, true>(raw, out, stats, B, sh, sw, dh, dw, rep, s2, 0, st)
                 : launch_march<false, false, INFER, false>(raw, out, stats, B, sh, sw, dh, dw, rep, s2, 0, st);
}

}  // namespace

extern "C" {

int t3d_preprocess_fixed_range_u16(const uint16_t* raw, int B, int src_h, int src_w, int dst_h, int dst_w, int path,
                                   float* out, int out_channels, float* grad_stats, int stats_scales, void* stream) {
    T3D_REQUIRE(raw && out, "NULL pointer");
    T3D_REQUIRE(B >= 1 && src_h >= 1 && src_w >= 1 && dst_h >= 1 && dst_w >= 1, "bad dims");
    T3D_REQUIRE(path == T3D_PATH_TRAIN || path == T3D_PATH_INFERENCE, "path must be T3D_PATH_TRAIN or T3D_PATH_INFERENCE");
    T3D_REQUIRE(out_channels == 1 || out_channels == 3, "out_channels must be 1 or 3");
    T3D_REQUIRE(stats_scales == 1 || stats_scales == 2, "stats_scales must be 1 or 2, got %d", stats_scales);
    T3D_REQUIRE((size_t)dst_h * dst_w < (1u << 30), "frame too large");
    T3D_REQUIRE(src_w <= 65535 && src_h <= 65535, "source frame too large (<= 65535 x 65535)");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const bool infer = path == T3D_PATH_INFERENCE;
    const bool vec = (dst_w % 4 == 0) && t3d_aligned16(out);
    if (!vec) {
        T3D_REQUIRE(grad_stats == nullptr, "grad_stats needs dst_w %% 4 == 0 (t3d_preprocess_stats_tiles() == 0 here)");
        const size_t total = (size_t)B * dst_h * dst_w;
        const int grid = (int)std::min((total + 255) / 256, (size_t)t3d_sm_count() * 8);
        if (infer) T3D_LAUNCH("fixed_range_scalar_kernel", st, fixed_range_scalar_kernel<true><<<grid, 256, 0, st>>>(
            raw, out, B, src_h, src_w, dst_h, dst_w, out_channels));
        else T3D_LAUNCH("fixed_range_scalar_kernel", st, fixed_range_scalar_kernel<false><<<grid, 256, 0, st>>>(
            raw, out, B, src_h, src_w, dst_h, dst_w, out_channels));
        return T3D_OK;
    }
    // half-resolution sums too where t3d_preprocess_train_u16 writes them (the same shapes, the same slots)
    const int s2 = (grad_stats && stats_scales == 2 && t3d_preprocess_stats_scales(dst_h, dst_w) == 2) ? 1 : 0;
    return infer ? launch_fixed<true>(raw, out, grad_stats, B, src_h, src_w, dst_h, dst_w, out_channels, s2, st)
                 : launch_fixed<false>(raw, out, grad_stats, B, src_h, src_w, dst_h, dst_w, out_channels, s2, st);
}

}  // extern "C"
