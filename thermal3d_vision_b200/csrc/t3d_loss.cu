// t3d_loss.cu -- fused thermal-aware loss, forward + backward, for sm_100a.
//
// Replaces /root/reference/utils/loss.py:75-98 and :100-305 (and what autograd
// derives from them).  Math and the closed-form backward: SURVEY.md Appendix A.
//
// Kernels (all HBM-bound, no tensor cores -- nothing here is a contraction):
//   thermal_stats_kernel   per-image sums of |Dx gray|, |Dy gray| (scale 1, 2)
//   loss_tile_kernel       one pass over a 16x128 pixel tile of one view:
//                          128-bit loads of the AoS pointmaps, shared-memory
//                          halo planes (z, gt z, gray, edge weight), loss
//                          partial sums AND d/dpred, d/dconf written once
//   loss_finalize_kernel   deterministic fixed-order fp64 second stage
//   rescale / scale        device-conditional gradient rescaling (no host sync)
#include "t3d_loss_internal.cuh"
#include <type_traits>
#include <string.h>

namespace {

constexpr float kEps = 1e-5f;          // utils/loss.py:240
constexpr float kThermalFactor = 8.0f; // utils/loss.py:252
constexpr float kHuber = 0.1f;         // utils/loss.py:267
constexpr float kConfMin = 1e-5f, kConfMax = 10.0f;  // utils/loss.py:91-92
constexpr float kScale2Weight = 0.35f; // 0.7 / scale, utils/loss.py:288

// ------------------------------------------------------------------ stats
constexpr int kSTH = 16, kSTW = 256, kSThreads = 256;
constexpr int kSPW = kSTW + 4;  // row stride of the gray plane (2 halo cols + pad)

struct StatsArgs {
    const float* thermal[2];
    float* partials;  // [B*2][stiles][4]  (sum tx1, ty1, tx2, ty2)
    int B, H, W, tch, tiles_x, tiles_y;
    int replicated;   // tch == 3 and the planes are bit-identical: read plane 0, gray = gray3(v, v, v)
};
constexpr int kTchReplicated = 13;   // `tch` value of the gray loaders for that case

template <bool VEC>
__device__ __forceinline__ void load_gray_quad(const float* __restrict__ t, int tch, size_t plane,
                                               size_t idx, int nvalid, float g[4]) {
    // idx: offset of the first pixel inside channel 0 of this image; plane = H*W
    if (VEC) {
        float4 c0 = ldg_stream_f4(t + idx);
        if (tch == kTchReplicated) {
            g[0] = gray3(c0.x, c0.x, c0.x); g[1] = gray3(c0.y, c0.y, c0.y);
            g[2] = gray3(c0.z, c0.z, c0.z); g[3] = gray3(c0.w, c0.w, c0.w);
        } else if (tch == 3) {
            float4 c1 = ldg_stream_f4(t + plane + idx);
            float4 c2 = ldg_stream_f4(t + 2 * plane + idx);
            g[0] = gray3(c0.x, c1.x, c2.x); g[1] = gray3(c0.y, c1.y, c2.y);
            g[2] = gray3(c0.z, c1.z, c2.z); g[3] = gray3(c0.w, c1.w, c2.w);
        } else {
            g[0] = c0.x; g[1] = c0.y; g[2] = c0.z; g[3] = c0.w;
        }
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            g[e] = 0.f;
            if (e < nvalid) {
                float c0 = ldg_stream_f1(t + idx + e);
                g[e] = (tch == kTchReplicated) ? gray3(c0, c0, c0) :
                       (tch == 3) ? gray3(c0, ldg_stream_f1(t + plane + idx + e),
                                          ldg_stream_f1(t + 2 * plane + idx + e)) : c0;
            }
        }
    }
}

__device__ __forceinline__ float load_gray_px(const float* __restrict__ t, int tch, size_t plane, size_t idx) {
    float c0 = ldg_f1(t + idx);
    if (tch == kTchReplicated) return gray3(c0, c0, c0);
    return (tch == 3) ? gray3(c0, ldg_f1(t + plane + idx), ldg_f1(t + 2 * plane + idx)) : c0;
}

template <bool MULTI, bool VEC>
__global__ void __launch_bounds__(kSThreads, 4) thermal_stats_kernel(const StatsArgs a) {
    __shared__ __align__(16) float sg[kSTH + 2][kSPW];
    __shared__ float red[kSThreads / 32][4];

    const int tid = threadIdx.x;
    const int tiles = a.tiles_x * a.tiles_y;
    const int img = blockIdx.x / tiles;
    const int tile = blockIdx.x - img * tiles;
    const int tyi = tile / a.tiles_x, txi = tile - tyi * a.tiles_x;
    const int i0 = tyi * kSTH, j0 = txi * kSTW;
    const int b = img >> 1, view = img & 1;
    const int H = a.H, W = a.W;
    const size_t plane = (size_t)H * W;
    const float* __restrict__ t = a.thermal[view] + (size_t)b * a.tch * plane;
    const int ltch = a.replicated ? kTchReplicated : a.tch;
    constexpr int HALO = MULTI ? 2 : 1;

    // main quads
    constexpr int QPR = kSTW / 4;  // quads per tile row
    for (int q = tid; q < kSTH * QPR; q += kSThreads) {
        const int r = q / QPR, cq = q - r * QPR;
        const int i = i0 + r, j = j0 + 4 * cq;
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (i < H && j < W) load_gray_quad<VEC>(t, ltch, plane, (size_t)i * W + j, min(4, W - j), g);
        *reinterpret_cast<float4*>(&sg[r][4 * cq]) = make_float4(g[0], g[1], g[2], g[3]);
    }
    // halo: HALO rows below, HALO cols to the right
    constexpr int NB = HALO * (kSTW + HALO), NR = HALO * kSTH;
    for (int h = tid; h < NB + NR; h += kSThreads) {
        int r, c;
        if (h < NB) { r = kSTH + h / (kSTW + HALO); c = h % (kSTW + HALO); }
        else        { int k = h - NB; r = k / HALO; c = kSTW + k % HALO; }
        const int i = i0 + r, j = j0 + c;
        sg[r][c] = (i < H && j < W) ? load_gray_px(t, ltch, plane, (size_t)i * W + j) : 0.f;
    }
    __syncthreads();

    float s[4] = {0.f, 0.f, 0.f, 0.f};
    for (int p = tid; p < kSTH * kSTW; p += kSThreads) {
        const int r = p / kSTW, c = p - r * kSTW;
        const int i = i0 + r, j = j0 + c;
        if (i < H && j < W) {
            const float g0 = sg[r][c];
            if (j < W - 1) s[0] += fabsf(sg[r][c + 1] - g0);
            if (i < H - 1) s[1] += fabsf(sg[r + 1][c] - g0);
        }
    }
    if (MULTI) {
        const int h2 = H >> 1, w2 = W >> 1;
        for (int p = tid; p < (kSTH / 2) * (kSTW / 2); p += kSThreads) {
            const int R = p / (kSTW / 2), C = p - R * (kSTW / 2);
            const int I = (i0 >> 1) + R, J = (j0 >> 1) + C;
            if (I < h2 && J < w2) {
                const int r = 2 * R, c = 2 * C;
                auto pool = [&](int rr, int cc) {
                    return 0.25f * (((sg[rr][cc] + sg[rr][cc + 1]) + sg[rr + 1][cc]) + sg[rr + 1][cc + 1]);
                };
                const float g0 = pool(r, c);
                if (J < w2 - 1) s[2] += fabsf(pool(r, c + 2) - g0);
                if (I < h2 - 1) s[3] += fabsf(pool(r + 2, c) - g0);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] = warp_sum(s[k]);
    if ((tid & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) red[tid >> 5][k] = s[k];
    }
    __syncthreads();
    if (tid < 4) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < kSThreads / 32; ++w) v += red[w][tid];
        a.partials[(((size_t)view * a.B + b) * tiles + tile) * 4 + tid] = v;   // [view][b][tile][4]
    }
}

// Fast path of the statistics (W % 4 == 0, 16-byte aligned planes): a warp marches down a 128-pixel strip of a
// 32-row band, 4 pixels per lane, 128-bit loads, vertical neighbours in registers, horizontal ones from shuffles
// (the strip's right edge: one 8-byte load); the half-resolution sums ride along on row pairs.  No shared memory.
// MODE 0: one plane, 1: three planes, 2: three bit-identical planes (plane 0 is read, gray = gray3(v, v, v)).
constexpr int kSMWarps = 4;
// rows per work item (a multiple of 4): shorter marches = finer load balance, more halo rows
constexpr int kStatsMarchRows = 32;
struct SRow { float g[4], e0, e1; };     // gray of the lane's quad and of the two pixels right of it

template <bool MULTI, int MODE>
__global__ void __launch_bounds__(kSMWarps * 32, (MODE == 1) ? 3 : 6) thermal_stats_march_kernel(const StatsArgs a, int nbands, int nstrips, int rows) {
    const int lane = threadIdx.x & 31;
    const int per_img = nbands * nstrips;
    const int item = blockIdx.x * kSMWarps + (threadIdx.x >> 5);
    if (item >= a.B * 2 * per_img) return;
    const int img = item / per_img, t = item - img * per_img;
    const int band = t / nstrips, strip = t - band * nstrips;
    const int b = img >> 1, view = img & 1;
    const int H = a.H, W = a.W, h2 = H >> 1;
    const size_t plane = (size_t)H * W;
    const float* __restrict__ th = a.thermal[view] + (size_t)b * a.tch * plane;
    const int ra = band * rows, rb = min(ra + rows, H);
    const int x0 = strip * 128 + 4 * lane;
    const bool active = x0 < W, has_right = x0 + 4 < W;
    const bool edge_lane = active && has_right && lane == 31;       // the pixels right of the quad belong to the next strip
    const float* __restrict__ px = th + (active ? x0 : 0);

    auto gray = [&](float c0, float c1, float c2) { return MODE == 0 ? c0 : gray3(c0, c1, c2); };
    struct Raw { float4 c0, c1, c2; float2 h0, h1, h2; };
    auto fetch = [&](int y, Raw& r) {                                // issue the loads of row y (nothing if outside the image)
        if (y < H && active) {
            const float* p = px + (size_t)y * W;
            r.c0 = ldg_stream_f4(p);
            if (MODE == 1) { r.c1 = ldg_stream_f4(p + plane); r.c2 = ldg_stream_f4(p + 2 * plane); }
            if (edge_lane) {
                r.h0 = __ldg(reinterpret_cast<const float2*>(p + 4));
                if (MODE == 1) { r.h1 = __ldg(reinterpret_cast<const float2*>(p + plane + 4)); r.h2 = __ldg(reinterpret_cast<const float2*>(p + 2 * plane + 4)); }
            }
        }
    };
    auto finish = [&](const Raw& r, SRow& o) {                       // gray values + right neighbours of a fetched row
        if (MODE == 1) {
            o.g[0] = gray(r.c0.x, r.c1.x, r.c2.x); o.g[1] = gray(r.c0.y, r.c1.y, r.c2.y);
            o.g[2] = gray(r.c0.z, r.c1.z, r.c2.z); o.g[3] = gray(r.c0.w, r.c1.w, r.c2.w);
        } else {
            o.g[0] = gray(r.c0.x, r.c0.x, r.c0.x); o.g[1] = gray(r.c0.y, r.c0.y, r.c0.y);
            o.g[2] = gray(r.c0.z, r.c0.z, r.c0.z); o.g[3] = gray(r.c0.w, r.c0.w, r.c0.w);
        }
        o.e0 = __shfl_down_sync(0xffffffffu, o.g[0], 1);
        o.e1 = MULTI ? __shfl_down_sync(0xffffffffu, o.g[1], 1) : 0.f;
        if (edge_lane) {
            if (MODE == 1) { o.e0 = gray(r.h0.x, r.h1.x, r.h2.x); o.e1 = gray(r.h0.y, r.h1.y, r.h2.y); }
            else { o.e0 = gray(r.h0.x, r.h0.x, r.h0.x); o.e1 = gray(r.h0.y, r.h0.y, r.h0.y); }
        }
        if (!has_right) { o.e0 = o.g[3]; o.e1 = o.g[3]; }           // zero-padded last column: dx == 0
    };
    auto dx_sum = [&](const SRow& c) { return fabsf(c.g[1] - c.g[0]) + fabsf(c.g[2] - c.g[1]) + fabsf(c.g[3] - c.g[2]) + fabsf(c.e0 - c.g[3]); };
    auto dy_sum = [&](const SRow& c, const SRow& n) { return fabsf(n.g[0] - c.g[0]) + fabsf(n.g[1] - c.g[1]) + fabsf(n.g[2] - c.g[2]) + fabsf(n.g[3] - c.g[3]); };
    auto pool = [&](float a0, float a1, float b0, float b1) { return 0.25f * (((a0 + a1) + b0) + b1); };
    struct Pooled { float c0, c1, cr; };
    auto pool_rows = [&](const SRow& u, const SRow& v) {
        Pooled p;
        p.c0 = pool(u.g[0], u.g[1], v.g[0], v.g[1]); p.c1 = pool(u.g[2], u.g[3], v.g[2], v.g[3]);
        p.cr = has_right ? pool(u.e0, u.e1, v.e0, v.e1) : p.c1;     // zero-padded last pooled column
        return p;
    };

    float s[4] = {0.f, 0.f, 0.f, 0.f};
    // rows ra, ra+1 first; then per pair (y, y+1): rows y+2, y+3 were fetched two pairs ago (four rows of loads in
    // flight per lane), are finished now, and the pair is evaluated
    Raw qa0 = {}, qa1 = {}, qb0 = {}, qb1 = {};
    SRow r0, r1, r2, r3;
    r1 = SRow{{0.f, 0.f, 0.f, 0.f}, 0.f, 0.f}; r2 = r1; r3 = r1;
    const int y_end = rb + 2;                                        // rows rb, rb+1: the pooled row below the band
    fetch(ra, qa0); fetch(ra + 1, qa1);
    fetch(ra + 2, qb0); fetch(ra + 3, qb1);
    finish(qa0, r0);
    if (ra + 1 < H) finish(qa1, r1);
    if (ra + 4 < y_end) { fetch(ra + 4, qa0); fetch(ra + 5, qa1); }
    Pooled pc = {0.f, 0.f, 0.f};
    if (MULTI && (ra >> 1) < h2) pc = pool_rows(r0, r1);
    // one row pair (y, y+1) held in (c0, c1); (n0, n1) receive rows y+2, y+3 from the fetched (f0, f1), which are
    // refilled with rows y+6, y+7.  INTERIOR: every row up to y+3 exists and pooled row y/2 + 1 does -- no guards.
    auto pair = [&](int y, Raw& f0, Raw& f1, const SRow& c0, const SRow& c1, SRow& n0, SRow& n1, auto interior_tag) {
        constexpr bool INTERIOR = decltype(interior_tag)::value;
        const bool has2 = INTERIOR || y + 2 < H, has3 = INTERIOR || y + 3 < H;
        if (has2) finish(f0, n0);
        if (has3) finish(f1, n1);
        if (y + 6 < y_end) { fetch(y + 6, f0); fetch(y + 7, f1); }
        // scale 1: rows y and y+1 (zero-padded last row: dy == 0)
        s[0] += dx_sum(c0);
        if (INTERIOR || y + 1 < H) s[1] += dy_sum(c0, c1);
        if (INTERIOR || y + 1 < rb) {
            s[0] += dx_sum(c1);
            if (has2) s[1] += dy_sum(c1, n0);
        }
        if (MULTI) {
            const int I = y >> 1;
            if (INTERIOR || I < h2) {
                s[2] += fabsf(pc.c1 - pc.c0) + fabsf(pc.cr - pc.c1);
                if (INTERIOR || I + 1 < h2) {                        // rows y+2, y+3 exist
                    const Pooled pn = pool_rows(n0, n1);
                    s[3] += fabsf(pn.c0 - pc.c0) + fabsf(pn.c1 - pc.c1);
                    pc = pn;
                }
            }
        }
    };
    if (rb + 2 <= H && ((rb - ra) & 3) == 0) {                       // rows rb, rb+1 exist (so does pooled row rb / 2)
        for (int y = ra; y < rb; y += 4) {
            pair(y, qb0, qb1, r0, r1, r2, r3, std::true_type{});
            pair(y + 2, qa0, qa1, r2, r3, r0, r1, std::true_type{});
        }
    } else {
        for (int y = ra; y < rb; y += 4) {                           // ra even, rb even or == H
            pair(y, qb0, qb1, r0, r1, r2, r3, std::false_type{});
            if (y + 2 < rb) pair(y + 2, qa0, qa1, r2, r3, r0, r1, std::false_type{});
        }
    }
    if (!active) { s[0] = 0.f; s[1] = 0.f; s[2] = 0.f; s[3] = 0.f; }
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] = warp_sum(s[k]);
    if (lane == 0)
        *reinterpret_cast<float4*>(a.partials + (((size_t)view * a.B + b) * per_img + t) * 4) = make_float4(s[0], s[1], s[2], s[3]);
}

// out_stats[B][2][2][2] = means (public API of t3d_thermal_grad_stats)
__global__ void thermal_stats_finalize_kernel(const float* __restrict__ partials, int stiles, int B,
                                              int H, int W, int multi, float* __restrict__ out) {
    const int img = blockIdx.x;      // 2 b + view
    const int k = threadIdx.x;  // 0..3
    if (k >= 4) return;
    double s = 0.0;
    const size_t base = ((size_t)(img & 1) * B + (img >> 1)) * stiles;
    for (int t = 0; t < stiles; ++t) s += (double)partials[(base + t) * 4 + k];
    const double n1 = (double)H * W, n2 = (double)(H >> 1) * (W >> 1);
    double m = (k < 2) ? s / n1 : ((multi && n2 > 0) ? s / n2 : 0.0);
    out[(size_t)img * 4 + k] = (float)m;
}

// ------------------------------------------------------------------ fused loss tile kernel
constexpr int kTH = 16, kTW = 128, kThreads = 256;
constexpr int kPW = kTW + 8;          // raw plane row stride: col j -> c = j - j0 + 4
constexpr int kQPT = kTH * kTW / 4 / kThreads;  // quads per thread (2)
constexpr int kP2H = kTH / 2 + 2, kP2W = kTW / 2 + 4;  // pooled planes: (I,J) -> R = I-I0+1, C = J-J0+1
constexpr int kNTerms = 8;            // basic, E1, S1, D1, E2, S2, D2, (pad)

struct LossArgs {
    const float* pred[2]; const float* gt[2]; const float* conf[2]; const float* thermal[2];
    float* dpred[2]; float* dconf[2];
    const float* stats[2];        // per view: [B][stiles][4]
    float* partials;              // [B*2][tiles][kNTerms]
    int B, H, W, tch, tiles_x, tiles_y, stiles;
    float alpha;
    float kb;                     // grad_scale / (3 H W)
    float kc;                     // grad_scale / (H W)
    float kE[2], kS[2], kD[2];    // grad_scale * lambda_s * weight / n_s
    float conf_max;               // upper clamp of the confidence: 10 (utils/loss.py:91), +inf with T3D_LOSS_CONF_MIN_ONLY
    // GT (and GT confidence) at another resolution: bilinear taps fused into the loads (train_thermal_dustr.py:234-271)
    int gt_h, gt_w;               // size of the gt arrays; 0 = the prediction's size (read directly)
    int conf_h, conf_w;           // size of the conf arrays; 0 = the prediction's size
};

// one channel-last value of F.interpolate(mode='bilinear', align_corners=False): taps btap, weights blerp
// (t3d_bilinear.cuh), as interp_bilinear_kernel (t3d_preprocess.cu)
__device__ __forceinline__ float bsample(const float* __restrict__ img, int sw, int C, int c, const BTap& ty, const BTap& tx) {
    const float v00 = __ldg(img + ((size_t)ty.i0 * sw + tx.i0) * C + c), v01 = __ldg(img + ((size_t)ty.i0 * sw + tx.i1) * C + c);
    const float v10 = __ldg(img + ((size_t)ty.i1 * sw + tx.i0) * C + c), v11 = __ldg(img + ((size_t)ty.i1 * sw + tx.i1) * C + c);
    return blerp(v00, v01, v10, v11, ty, tx);
}

template <bool MULTI>
constexpr size_t loss_smem_bytes() {
    constexpr int HALO = MULTI ? 2 : 1;
    size_t raw = (size_t)3 * (kTH + 2 * HALO) * kPW + (size_t)(kTH + 1) * kPW;
    size_t pooled = MULTI ? (size_t)3 * kP2H * kP2W + (size_t)kP2H * kP2W : 0;
    return (raw + pooled) * sizeof(float);
}

struct Acc3 { float E, S, D; };

// One forward-difference term (x or y) at one position (SURVEY.md Appendix A):
//   s = zb - za, a = |s|, b = |gb - ga|;  E += a(1-w), S += a^2 w, D += huber(|a-b|)
//   q = sgn(s) [kE (1-w) + kS 2 a w + kD rho'(|a-b|) sgn(a-b)]
// valid == false is the zero-padded last column / row (or outside the image): all zero.
template <bool ACC>
__device__ __forceinline__ float diff_term(bool valid, float za, float zb, float ga, float gb, float w,
                                           float kE, float kS, float kD, Acc3& acc) {
    if (!valid) return 0.f;
    const float s = zb - za;
    const float a = fabsf(s);
    const float b = fabsf(gb - ga);
    const float e = a - b;
    const float d = fabsf(e);
    const bool quad = d < kHuber;                     // strict, utils/loss.py:275
    if (ACC) {
        acc.E += a * (1.f - w);
        acc.S += a * a * w;
        acc.D += quad ? 0.5f * d * d : kHuber * (d - 0.5f * kHuber);
    }
    const float dh = quad ? e : copysignf(kHuber, e);  // rho'(d) * sgn(e); e == 0 -> 0
    return sgnf(s) * (kE * (1.f - w) + kS * 2.f * a * w + kD * dh);
}

__device__ __forceinline__ float edge_weight_of(float tx, float ty, float inv_mx, float inv_my, float m) {
    // utils/loss.py:240-256: exp(-8 clamp(tx/mean,0,m)) * exp(-8 clamp(ty/mean,0,m))
    // tx, ty >= 0 so only the upper clamp acts; the select form lets NaN through like torch.clamp
    const float ax = tx * inv_mx, ay = ty * inv_my;
    const float cx = (ax > m) ? m : ax;
    const float cy = (ay > m) ? m : ay;
    return expf(-kThermalFactor * cx) * expf(-kThermalFactor * cy);
}

template <bool MULTI, bool VEC, bool BWD>
__global__ void __launch_bounds__(kThreads, MULTI ? 2 : 3) loss_tile_kernel(const LossArgs a) {
    constexpr int HALO = MULTI ? 2 : 1;
    constexpr int ROWS = kTH + 2 * HALO;
    extern __shared__ __align__(16) float smem[];
    float (*sz)[kPW]  = reinterpret_cast<float (*)[kPW]>(smem);
    float (*sgz)[kPW] = reinterpret_cast<float (*)[kPW]>(smem + ROWS * kPW);
    float (*sg)[kPW]  = reinterpret_cast<float (*)[kPW]>(smem + 2 * ROWS * kPW);
    float (*swt)[kPW] = reinterpret_cast<float (*)[kPW]>(smem + 3 * ROWS * kPW);   // w(i,j): row i -> i-i0+1
    float* pooled_base = smem + 3 * ROWS * kPW + (kTH + 1) * kPW;
    float (*pz)[kP2W]  = reinterpret_cast<float (*)[kP2W]>(pooled_base);
    float (*pgz)[kP2W] = reinterpret_cast<float (*)[kP2W]>(pooled_base + kP2H * kP2W);
    float (*pg)[kP2W]  = reinterpret_cast<float (*)[kP2W]>(pooled_base + 2 * kP2H * kP2W);
    float (*pw)[kP2W]  = reinterpret_cast<float (*)[kP2W]>(pooled_base + 3 * kP2H * kP2W);
    __shared__ float red[kThreads / 32][kNTerms];
    __shared__ float s_inv[4];

    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int tiles = a.tiles_x * a.tiles_y;
    const int img = blockIdx.x / tiles;
    const int tile = blockIdx.x - img * tiles;
    const int tyi = tile / a.tiles_x, txi = tile - tyi * a.tiles_x;
    const int i0 = tyi * kTH, j0 = txi * kTW;
    const int b = img >> 1, view = img & 1;
    const int H = a.H, W = a.W;
    const size_t plane = (size_t)H * W;
    const bool thermal_on = a.tch != 0;

    const float* __restrict__ pred = a.pred[view] + (size_t)b * plane * 3;
    const bool gt_rs = a.gt_h != 0, conf_rs = a.conf_h != 0;        // block-uniform: bilinear taps instead of direct reads
    const float* __restrict__ gt = a.gt[view] + (size_t)b * (gt_rs ? (size_t)a.gt_h * a.gt_w : plane) * 3;
    const float* __restrict__ conf = a.conf[view] ? a.conf[view] + (size_t)b * (conf_rs ? (size_t)a.conf_h * a.conf_w : plane) : nullptr;
    const float gsy = gt_rs ? (float)a.gt_h / (float)H : 1.f, gsx = gt_rs ? (float)a.gt_w / (float)W : 1.f;
    const float csy = conf_rs ? (float)a.conf_h / (float)H : 1.f, csx = conf_rs ? (float)a.conf_w / (float)W : 1.f;
    const float* __restrict__ th = thermal_on ? a.thermal[view] + (size_t)b * a.tch * plane : nullptr;
    float* __restrict__ dpred = BWD ? a.dpred[view] + (size_t)b * plane * 3 : nullptr;
    float* __restrict__ dconf = (BWD && a.dconf[view]) ? a.dconf[view] + (size_t)b * plane : nullptr;

    // 1/(mean + eps) of the thermal gradients of this image (fixed-order sum of the stats partials)
    if (thermal_on && tid < 4) {
        double s = 0.0;
        const float* sp = a.stats[view] + (size_t)b * a.stiles * 4 + tid;
        for (int t = 0; t < a.stiles; ++t) s += (double)sp[(size_t)t * 4];
        const double n = (tid < 2) ? (double)H * W : (double)(H >> 1) * (W >> 1);
        const float mean = (n > 0) ? (float)(s / n) : 0.f;
        s_inv[tid] = 1.0f / (mean + kEps);
    }

    // ---------------- phase 1: load own quads, basic term, fill planes
    float gq[kQPT][12];   // basic-term gradient of this thread's quads (AoS order)
    float sum_basic = 0.f;
#pragma unroll
    for (int k = 0; k < kQPT; ++k) {
        const int r = wrp + (kThreads / 32) * k;
        const int i = i0 + r, j = j0 + 4 * lane;
        float zq[4] = {0.f, 0.f, 0.f, 0.f}, gzq[4] = {0.f, 0.f, 0.f, 0.f}, grq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 12; ++e) gq[k][e] = 0.f;
        if (i < H && j < W) {
            const int nvalid = VEC ? 4 : min(4, W - j);
            const size_t pix = (size_t)i * W + j;
            float p[12], g[12], c[4];
            if (VEC) {
                const float4* pp = reinterpret_cast<const float4*>(pred + pix * 3);
                const float4* gp = reinterpret_cast<const float4*>(gt + pix * 3);
                float4 p0 = ldg_stream_f4((const float*)(pp)), p1 = ldg_stream_f4((const float*)(pp + 1)),
                       p2 = ldg_stream_f4((const float*)(pp + 2));
                float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0, g2 = g0;
                if (!gt_rs) { g0 = ldg_stream_f4((const float*)(gp)); g1 = ldg_stream_f4((const float*)(gp + 1)); g2 = ldg_stream_f4((const float*)(gp + 2)); }
                p[0] = p0.x; p[1] = p0.y; p[2] = p0.z; p[3] = p0.w; p[4] = p1.x; p[5] = p1.y;
                p[6] = p1.z; p[7] = p1.w; p[8] = p2.x; p[9] = p2.y; p[10] = p2.z; p[11] = p2.w;
                g[0] = g0.x; g[1] = g0.y; g[2] = g0.z; g[3] = g0.w; g[4] = g1.x; g[5] = g1.y;
                g[6] = g1.z; g[7] = g1.w; g[8] = g2.x; g[9] = g2.y; g[10] = g2.z; g[11] = g2.w;
                if (conf && !conf_rs) {
                    float4 cc = ldg_stream_f4(conf + pix);
                    c[0] = cc.x; c[1] = cc.y; c[2] = cc.z; c[3] = cc.w;
                } else { c[0] = c[1] = c[2] = c[3] = 1.f; }
            } else {
#pragma unroll
                for (int e = 0; e < 12; ++e) {
                    const bool ok = e < nvalid * 3;
                    p[e] = ok ? ldg_stream_f1(pred + pix * 3 + e) : 0.f;
                    g[e] = (ok && !gt_rs) ? ldg_stream_f1(gt + pix * 3 + e) : 0.f;
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) c[e] = (conf && !conf_rs && e < nvalid) ? ldg_stream_f1(conf + pix + e) : 1.f;
            }
            if (gt_rs || conf_rs) {                            // taps of this row / these 4 columns
                const BTap gty = btap(i, a.gt_h, gsy), cty = btap(i, a.conf_h, csy);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (e >= nvalid) continue;
                    if (gt_rs) {
                        const BTap gtx = btap(j + e, a.gt_w, gsx);
#pragma unroll
                        for (int ch = 0; ch < 3; ++ch) g[3 * e + ch] = bsample(gt, a.gt_w, 3, ch, gty, gtx);
                    }
                    if (conf_rs && conf) c[e] = bsample(conf, a.conf_w, 1, 0, cty, btap(j + e, a.conf_w, csx));
                }
            }
            if (thermal_on) load_gray_quad<VEC>(th, a.tch, plane, pix, nvalid, grq);
            float dc[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float dx = p[3 * e] - g[3 * e], dy = p[3 * e + 1] - g[3 * e + 1], dz = p[3 * e + 2] - g[3 * e + 2];
                const float l = ((fabsf(dx) + fabsf(dy)) + fabsf(dz)) / 3.0f;             // utils/loss.py:82
                const float craw = c[e];
                const float cc = (craw < kConfMin) ? kConfMin : ((craw > a.conf_max) ? a.conf_max : craw);   // :91, NaN passes
                const bool ok = e < nvalid;
                if (ok) sum_basic += cc * l - a.alpha * logf(cc);                          // :95
                zq[e] = p[3 * e + 2];
                gzq[e] = g[3 * e + 2];
                if (BWD) {
                    const float kc3 = cc * a.kb;
                    gq[k][3 * e] = sgnf(dx) * kc3;
                    gq[k][3 * e + 1] = sgnf(dy) * kc3;
                    gq[k][3 * e + 2] = sgnf(dz) * kc3;
                    const bool inside = (craw >= kConfMin) && (craw <= a.conf_max);       // clamp grad mask (inclusive)
                    dc[e] = inside ? (l - a.alpha / cc) * a.kc : 0.f;
                }
            }
            if (BWD && dconf) {
                if (VEC) stg_stream_f4(dconf + pix, make_float4(dc[0], dc[1], dc[2], dc[3]));
                else {
#pragma unroll
                    for (int e = 0; e < 4; ++e) if (e < nvalid) stg_stream_f1(dconf + pix + e, dc[e]);
                }
            }
        }
        if (thermal_on) {
            *reinterpret_cast<float4*>(&sz[r + HALO][4 + 4 * lane]) = make_float4(zq[0], zq[1], zq[2], zq[3]);
            *reinterpret_cast<float4*>(&sgz[r + HALO][4 + 4 * lane]) = make_float4(gzq[0], gzq[1], gzq[2], gzq[3]);
            *reinterpret_cast<float4*>(&sg[r + HALO][4 + 4 * lane]) = make_float4(grq[0], grq[1], grq[2], grq[3]);
        }
    }

    Acc3 acc1 = {0.f, 0.f, 0.f}, acc2 = {0.f, 0.f, 0.f};

    if (thermal_on) {
        // ---------------- halo ring (z, gt z, gray): HALO rows above/below, HALO cols left/right
        constexpr int RW = kTW + 2 * HALO;                   // ring row width
        constexpr int NTOPBOT = 2 * HALO * RW, NSIDE = 2 * HALO * kTH;
        for (int h = tid; h < NTOPBOT + NSIDE; h += kThreads) {
            int r, c;  // plane coordinates
            if (h < NTOPBOT) {
                const int rr = h / RW, cc = h - rr * RW;
                r = (rr < HALO) ? rr : (kTH + rr);            // rows 0..HALO-1 and kTH+HALO..kTH+2HALO-1
                c = 4 - HALO + cc;
            } else {
                const int k = h - NTOPBOT;
                const int rr = k / (2 * HALO), cc = k - rr * (2 * HALO);
                r = HALO + rr;
                c = (cc < HALO) ? (4 - HALO + cc) : (4 + kTW + cc - HALO);
            }
            const int i = i0 + r - HALO, j = j0 + c - 4;
            float zv = 0.f, gzv = 0.f, gv = 0.f;
            if (i >= 0 && i < H && j >= 0 && j < W) {
                const size_t pix = (size_t)i * W + j;
                zv = ldg_f1(pred + pix * 3 + 2);
                gzv = gt_rs ? bsample(gt, a.gt_w, 3, 2, btap(i, a.gt_h, gsy), btap(j, a.gt_w, gsx)) : ldg_f1(gt + pix * 3 + 2);
                gv = load_gray_px(th, a.tch, plane, pix);
            }
            sz[r][c] = zv; sgz[r][c] = gzv; sg[r][c] = gv;
        }
        __syncthreads();

        // ---------------- phase 2: edge weights w(i,j) for rows i0-1..i0+TH-1, cols j0-1..j0+TW-1
        const float m = (view == 0) ? 0.4f : 0.5f;            // utils/loss.py:253-256
        const float inv_mx1 = s_inv[0], inv_my1 = s_inv[1];
        auto w_at = [&](int r, int c) -> float {               // plane coords of (i,j)
            const int i = i0 + r - HALO, j = j0 + c - 4;
            if (i < 0 || i >= H || j < 0 || j >= W) return 0.f;
            const float g0 = sg[r][c];
            const float tx = (j < W - 1) ? fabsf(sg[r][c + 1] - g0) : 0.f;
            const float ty = (i < H - 1) ? fabsf(sg[r + 1][c] - g0) : 0.f;
            return edge_weight_of(tx, ty, inv_mx1, inv_my1, m);
        };
#pragma unroll
        for (int k = 0; k < kQPT; ++k) {
            const int r = wrp + (kThreads / 32) * k;
            float4 wv;
            wv.x = w_at(r + HALO, 4 + 4 * lane);     wv.y = w_at(r + HALO, 5 + 4 * lane);
            wv.z = w_at(r + HALO, 6 + 4 * lane);     wv.w = w_at(r + HALO, 7 + 4 * lane);
            *reinterpret_cast<float4*>(&swt[r + 1][4 + 4 * lane]) = wv;
        }
        if (tid < kTW + 1) swt[0][3 + tid] = w_at(HALO - 1, 3 + tid);              // row i0-1
        else if (tid < kTW + 1 + kTH) { const int r = tid - (kTW + 1); swt[r + 1][3] = w_at(r + HALO, 3); }  // col j0-1

        if (MULTI) {
            // pooled planes for cells I0-1..I0+TH/2, J0-1..J0+TW/2 (utils/loss.py:159-174, floor division)
            const int h2 = H >> 1, w2 = W >> 1;
            const int I0 = i0 >> 1, J0 = j0 >> 1;
            for (int p = tid; p < kP2H * (kTW / 2 + 2); p += kThreads) {
                const int R = p / (kTW / 2 + 2), C = p - R * (kTW / 2 + 2);
                const int I = I0 + R - 1, J = J0 + C - 1;
                float vz = 0.f, vgz = 0.f, vg = 0.f;
                if (I >= 0 && I < h2 && J >= 0 && J < w2) {
                    const int r = 2 * R, c = 2 * C + 2;   // raw plane coords of (2I, 2J)
                    vz  = 0.25f * (((sz[r][c] + sz[r][c + 1]) + sz[r + 1][c]) + sz[r + 1][c + 1]);
                    vgz = 0.25f * (((sgz[r][c] + sgz[r][c + 1]) + sgz[r + 1][c]) + sgz[r + 1][c + 1]);
                    vg  = 0.25f * (((sg[r][c] + sg[r][c + 1]) + sg[r + 1][c]) + sg[r + 1][c + 1]);
                }
                pz[R][C] = vz; pgz[R][C] = vgz; pg[R][C] = vg;
            }
            __syncthreads();
            const float inv_mx2 = s_inv[2], inv_my2 = s_inv[3];
            for (int p = tid; p < (kTH / 2 + 1) * (kTW / 2 + 1); p += kThreads) {
                const int R = p / (kTW / 2 + 1), C = p - R * (kTW / 2 + 1);
                const int I = I0 + R - 1, J = J0 + C - 1;
                float w = 0.f;
                if (I >= 0 && I < h2 && J >= 0 && J < w2) {
                    const float g0 = pg[R][C];
                    const float tx = (J < w2 - 1) ? fabsf(pg[R][C + 1] - g0) : 0.f;
                    const float ty = (I < h2 - 1) ? fabsf(pg[R + 1][C] - g0) : 0.f;
                    w = edge_weight_of(tx, ty, inv_mx2, inv_my2, m);
                }
                pw[R][C] = w;
            }
        }
        __syncthreads();

        // ---------------- phase 3: stencil terms + gather gradient for own pixels
#pragma unroll
        for (int k = 0; k < kQPT; ++k) {
            const int r0 = wrp + (kThreads / 32) * k;
            const int i = i0 + r0, j = j0 + 4 * lane;
            if (i >= H || j >= W) continue;
            const int r = r0 + HALO, c = 4 + 4 * lane;
            const float kE = a.kE[0], kS = a.kS[0], kD = a.kD[0];
            // row i: cols c-1 .. c+4
            float zr[6], gr[6];
            {
                const float4 zc = *reinterpret_cast<const float4*>(&sz[r][c]);
                const float4 gc = *reinterpret_cast<const float4*>(&sgz[r][c]);
                zr[0] = sz[r][c - 1]; zr[1] = zc.x; zr[2] = zc.y; zr[3] = zc.z; zr[4] = zc.w; zr[5] = sz[r][c + 4];
                gr[0] = sgz[r][c - 1]; gr[1] = gc.x; gr[2] = gc.y; gr[3] = gc.z; gr[4] = gc.w; gr[5] = sgz[r][c + 4];
            }
            const float4 zu = *reinterpret_cast<const float4*>(&sz[r - 1][c]);
            const float4 gu = *reinterpret_cast<const float4*>(&sgz[r - 1][c]);
            const float4 zd = *reinterpret_cast<const float4*>(&sz[r + 1][c]);
            const float4 gd = *reinterpret_cast<const float4*>(&sgz[r + 1][c]);
            const float4 wc = *reinterpret_cast<const float4*>(&swt[r0 + 1][c]);
            const float4 wu = *reinterpret_cast<const float4*>(&swt[r0][c]);
            const float wl = swt[r0 + 1][c - 1];
            const float zup[4] = {zu.x, zu.y, zu.z, zu.w}, gup[4] = {gu.x, gu.y, gu.z, gu.w};
            const float zdn[4] = {zd.x, zd.y, zd.z, zd.w}, gdn[4] = {gd.x, gd.y, gd.z, gd.w};
            const float wcur[4] = {wc.x, wc.y, wc.z, wc.w}, wup[4] = {wu.x, wu.y, wu.z, wu.w};

            Acc3 dummy = {0.f, 0.f, 0.f};
            // q_x(i, j-1)
            float qx_prev = diff_term<false>(j > 0, zr[0], zr[1], gr[0], gr[1], wl, kE, kS, kD, dummy);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int jj = j + e;
                const bool in = VEC ? true : (jj < W);
                float dz = 0.f;
                if (in) {
                    const float qx = diff_term<true>(jj < W - 1, zr[e + 1], zr[e + 2], gr[e + 1], gr[e + 2],
                                                     wcur[e], kE, kS, kD, acc1);
                    const float qy = diff_term<true>(i < H - 1, zr[e + 1], zdn[e], gr[e + 1], gdn[e],
                                                     wcur[e], kE, kS, kD, acc1);
                    const float qyu = diff_term<false>(i > 0, zup[e], zr[e + 1], gup[e], gr[e + 1],
                                                       wup[e], kE, kS, kD, dummy);
                    dz = -qx + qx_prev - qy + qyu;
                    qx_prev = qx;
                }
                if (BWD) gq[k][3 * e + 2] += dz;
            }
            if (MULTI) {
                const int h2 = H >> 1, w2 = W >> 1;
                const int I = i >> 1;
                if (I < h2) {
                    const int R = I - (i0 >> 1) + 1;
                    const bool own_row = (i & 1) == 0;       // count each pooled cell once
                    const float kE2 = a.kE[1], kS2 = a.kS[1], kD2 = a.kD[1];
#pragma unroll
                    for (int cidx = 0; cidx < 2; ++cidx) {
                        const int J = (j >> 1) + cidx;
                        if (J >= w2) continue;
                        const int C = J - (j0 >> 1) + 1;
                        const float z0 = pz[R][C], g0 = pgz[R][C], w0 = pw[R][C];
                        Acc3 acc_tmp = {0.f, 0.f, 0.f};
                        const float qx = diff_term<true>(J < w2 - 1, z0, pz[R][C + 1], g0, pgz[R][C + 1], w0, kE2, kS2, kD2, acc_tmp);
                        const float qy = diff_term<true>(I < h2 - 1, z0, pz[R + 1][C], g0, pgz[R + 1][C], w0, kE2, kS2, kD2, acc_tmp);
                        const float qxl = diff_term<false>(J > 0, pz[R][C - 1], z0, pgz[R][C - 1], g0, pw[R][C - 1], kE2, kS2, kD2, dummy);
                        const float qyu = diff_term<false>(I > 0, pz[R - 1][C], z0, pgz[R - 1][C], g0, pw[R - 1][C], kE2, kS2, kD2, dummy);
                        if (own_row) { acc2.E += acc_tmp.E; acc2.S += acc_tmp.S; acc2.D += acc_tmp.D; }
                        const float dz2 = 0.25f * (-qx + qxl - qy + qyu);
                        if (BWD) {
                            if (VEC || j + 2 * cidx < W) gq[k][3 * (2 * cidx) + 2] += dz2;
                            if (VEC || j + 2 * cidx + 1 < W) gq[k][3 * (2 * cidx + 1) + 2] += dz2;
                        }
                    }
                }
            }
        }
    }

    // ---------------- store d/dpred (one write per element)
    if (BWD) {
#pragma unroll
        for (int k = 0; k < kQPT; ++k) {
            const int r = wrp + (kThreads / 32) * k;
            const int i = i0 + r, j = j0 + 4 * lane;
            if (i >= H || j >= W) continue;
            const size_t pix = (size_t)i * W + j;
            if (VEC) {
                float* o = dpred + pix * 3;
                stg_stream_f4(o, make_float4(gq[k][0], gq[k][1], gq[k][2], gq[k][3]));
                stg_stream_f4(o + 4, make_float4(gq[k][4], gq[k][5], gq[k][6], gq[k][7]));
                stg_stream_f4(o + 8, make_float4(gq[k][8], gq[k][9], gq[k][10], gq[k][11]));
            } else {
                const int nvalid = min(4, W - j);
#pragma unroll
                for (int e = 0; e < 12; ++e) if (e < nvalid * 3) stg_stream_f1(dpred + pix * 3 + e, gq[k][e]);
            }
        }
    }

    // ---------------- block reduction -> one partial vector per tile
    float v[kNTerms] = {sum_basic, acc1.E, acc1.S, acc1.D, acc2.E, acc2.S, acc2.D, 0.f};
#pragma unroll
    for (int t = 0; t < kNTerms - 1; ++t) v[t] = warp_sum(v[t]);
    if (lane == 0) {
#pragma unroll
        for (int t = 0; t < kNTerms; ++t) red[wrp][t] = v[t];
    }
    __syncthreads();
    if (tid < kNTerms) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) s += red[w][tid];
        a.partials[((size_t)img * tiles + tile) * kNTerms + tid] = s;
    }
}

// ------------------------------------------------------------------ second stage
struct FinalizeArgs {
    const float* partials2;  // multi-scale split path: [B*2][tiles2][4] = E2, S2, D2, 0 (else NULL)
    int tiles2;
    const float* partials;   // [B*2][tiles][kNTerms]
    float* out_sample; float* out_batch; double* out_f64;
    unsigned int* counter;
    int B, H, W, tiles, multi, thermal_on;
    float ew, sw, dw;
};

__global__ void __launch_bounds__(128) loss_finalize_kernel(const FinalizeArgs a) {
    __shared__ double tot[2][kNTerms];
    __shared__ bool is_last;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    // 16 (view, term) sums.  Thread t owns the tiles t, t + 128, ... of each view (two 128-bit loads per
    // partial), then a fixed butterfly per warp and a fixed order over the 4 warps: deterministic.
    __shared__ double wsum[4][2][kNTerms];
    double acc[2][kNTerms];
#pragma unroll
    for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int k = 0; k < kNTerms; ++k) acc[v][k] = 0.0;
#pragma unroll
    for (int view = 0; view < 2; ++view) {
        const float4* p = reinterpret_cast<const float4*>(a.partials + ((size_t)(2 * b + view) * a.tiles) * kNTerms);
        for (int t = tid; t < a.tiles; t += 128) {
            const float4 lo = p[2 * t], hi = p[2 * t + 1];
            acc[view][0] += (double)lo.x; acc[view][1] += (double)lo.y; acc[view][2] += (double)lo.z; acc[view][3] += (double)lo.w;
            acc[view][4] += (double)hi.x; acc[view][5] += (double)hi.y; acc[view][6] += (double)hi.z; acc[view][7] += (double)hi.w;
        }
    }
#pragma unroll
    for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int k = 0; k < kNTerms - 1; ++k) {          // term 7 is padding
            const double r = warp_sum(acc[v][k]);
            if (lane == 0) wsum[wrp][v][k] = r;
        }
    __syncthreads();
    if (tid < 2 * kNTerms) {
        const int v = tid / kNTerms, k = tid - v * kNTerms;
        tot[v][k] = (k < kNTerms - 1) ? ((wsum[0][v][k] + wsum[1][v][k]) + (wsum[2][v][k] + wsum[3][v][k])) : 0.0;
    }
    __syncthreads();
    if (a.partials2) {                 // scale-2 sums of the split multi-scale path: lane t owns tiles t, t + 32, ...
        const int v = wrp >> 1;        // of one view (2 warps per view: 6 (view, term) sums over 4 warps), fixed butterfly
        const float4* p2 = reinterpret_cast<const float4*>(a.partials2 + ((size_t)(2 * b + v) * a.tiles2) * 4);
        double s2[3] = {0.0, 0.0, 0.0};
        if ((wrp & 1) == 0)
            for (int t = lane; t < a.tiles2; t += 32) { const float4 x = p2[t]; s2[0] += (double)x.x; s2[1] += (double)x.y; s2[2] += (double)x.z; }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double r = warp_sum(s2[k]);
            if ((wrp & 1) == 0 && lane == 0) tot[v][4 + k] = r;
        }
    }
    __syncthreads();
    if (tid == 0) {
        const double N = (double)a.H * a.W;
        const double n2 = (double)(a.H >> 1) * (a.W >> 1);
        const double basic = tot[0][0] / N + tot[1][0] / N;                 // utils/loss.py:95-98
        double edge = 0, smooth = 0, detail = 0;
        if (a.thermal_on) {
            edge = (tot[0][1] + tot[1][1]) / N;
            smooth = (tot[0][2] + tot[1][2]) / N;
            detail = (tot[0][3] + tot[1][3]) / N;
            if (a.multi) {                                                   // 0/0 -> NaN like the reference
                edge += (double)kScale2Weight * ((tot[0][4] + tot[1][4]) / n2);
                smooth += (double)kScale2Weight * ((tot[0][5] + tot[1][5]) / n2);
                detail += (double)kScale2Weight * ((tot[0][6] + tot[1][6]) / n2);
            }
        }
        const double total = basic + (double)a.ew * edge + (double)a.sw * smooth + (double)a.dw * detail;  // :295
        const float tf = (float)total;
        const bool valid = isfinite(tf) && tf > 0.f;                        // train_thermal_dustr.py:320
        float* o = a.out_sample + (size_t)b * T3D_LOSS_OUT_STRIDE;
        o[0] = tf; o[1] = (float)basic; o[2] = (float)edge; o[3] = (float)smooth; o[4] = (float)detail;
        o[5] = valid ? 1.f : 0.f; o[6] = 0.f; o[7] = 0.f;
        if (a.out_f64) {
            double* d = a.out_f64 + (size_t)b * T3D_LOSS_OUT_STRIDE;
            d[0] = total; d[1] = basic; d[2] = edge; d[3] = smooth; d[4] = detail; d[5] = valid ? 1.0 : 0.0;
            d[6] = 0; d[7] = 0;
        }
        __threadfence();
        const unsigned int done = atomicAdd(a.counter, 1u);
        is_last = (done == (unsigned)a.B - 1);
    }
    __syncthreads();
    if (is_last) {
        // batch stage: mean over valid samples; fixed-shape tree over a fixed sample->thread map (deterministic)
        __shared__ double bs[128][6];
        __threadfence();
        double s[6] = {0, 0, 0, 0, 0, 0};
        for (int i = tid; i < a.B; i += 128) {
            const float* o = a.out_sample + (size_t)i * T3D_LOSS_OUT_STRIDE;
            const float4 v0 = __ldcg(reinterpret_cast<const float4*>(o));
            const float4 v1 = __ldcg(reinterpret_cast<const float4*>(o) + 1);
            if (v1.y != 0.f) {
                s[0] += (double)v0.x; s[1] += (double)v0.y; s[2] += (double)v0.z; s[3] += (double)v0.w;
                s[4] += (double)v1.x; s[5] += 1.0;
            }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) bs[tid][k] = s[k];
        __syncthreads();
        for (int stride = 64; stride > 0; stride >>= 1) {
            if (tid < stride) {
#pragma unroll
                for (int k = 0; k < 6; ++k) bs[tid][k] += bs[tid + stride][k];
            }
            __syncthreads();
        }
        if (tid == 0) {
            const double nv = bs[0][5];
            for (int k = 0; k < 5; ++k) a.out_batch[k] = (nv > 0) ? (float)(bs[0][k] / nv) : 0.f;
            a.out_batch[5] = (float)nv; a.out_batch[6] = (float)a.B; a.out_batch[7] = 0.f;
            *a.counter = 0u;
        }
    }
}

// ------------------------------------------------------------------ gradient rescaling
struct ScaleArgs {
    float* dpred[2]; float* dconf[2];
    const float* out_sample; const float* out_batch; const float* grad_output;
    int B; size_t plane;
};

// mode 0: per-sample validity fix-up; mode 1: uniform *grad_output
template <int MODE>
__global__ void __launch_bounds__(256) scale_grads_kernel(const ScaleArgs a) {
    float uniform = 1.f;
    if (MODE == 0) { if (a.out_batch[5] == (float)a.B) return; }
    else { uniform = *a.grad_output; if (uniform == 1.0f) return; }
    const float nv = (MODE == 0) ? a.out_batch[5] : 1.f;
    const size_t per_sample[2] = {a.plane * 3, a.plane};
#pragma unroll
    for (int which = 0; which < 4; ++which) {
        float* base = (which < 2) ? a.dpred[which] : a.dconf[which - 2];
        if (!base) continue;
        const size_t n = per_sample[which >> 1];
        const size_t total = n * a.B;
        for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
             idx += (size_t)gridDim.x * blockDim.x) {
            float f = uniform;
            if (MODE == 0) {
                const int b = (int)(idx / n);
                const bool valid = a.out_sample[(size_t)b * T3D_LOSS_OUT_STRIDE + 5] != 0.f;
                f = (valid && nv > 0.f) ? (float)a.B / nv : 0.f;
            }
            // invalid samples may hold NaN/Inf gradients: force exact zeros there
            base[idx] = (f == 0.f) ? 0.f : base[idx] * f;
        }
    }
}

// ------------------------------------------------------------------ v1 loss (utils/loss.py:4-72)
// basic + (edge_weight + smoothness_weight) * sum_views [ mean_{H x (W-1)} |Dx z| exp(-10 |Dx gray|)
//                                                       + mean_{(H-1) x W} |Dy z| exp(-10 |Dy gray|) ]
// (the reference computes the same expression twice, as "edge" and as "smoothness").  Dead code in the
// reference's training loop; kept for API completeness -> simple one-thread-per-pixel kernel.
struct V1Args {
    const float* pred[2]; const float* gt[2]; const float* conf[2]; const float* thermal[2];
    float* dpred[2]; float* dconf[2];
    float* partials;      // [B*2][blocks][kNTerms]
    int B, H, W, tch, blocks;
    float alpha, kb, kc, kx, ky;      // kx = gscale (ew+sw) / (H (W-1)), ky = gscale (ew+sw) / ((H-1) W)
    float sx, sy;                     // N / (H (W-1)), N / ((H-1) W): the second stage divides by N
};

template <bool BWD>
__global__ void __launch_bounds__(256) loss_v1_kernel(const V1Args a) {
    __shared__ float red[8][2];
    const int img = blockIdx.y, b = img >> 1, view = img & 1;
    const int H = a.H, W = a.W;
    const size_t plane = (size_t)H * W;
    const int idx = blockIdx.x * 256 + threadIdx.x;
    const float* pred = a.pred[view] + (size_t)b * plane * 3;
    const float* gt = a.gt[view] + (size_t)b * plane * 3;
    const float* conf = a.conf[view] ? a.conf[view] + (size_t)b * plane : nullptr;
    const float* th = a.tch ? a.thermal[view] + (size_t)b * a.tch * plane : nullptr;
    float sum_b = 0.f, sum_e = 0.f;
    if (idx < (int)plane) {
        const int i = idx / W, j = idx - i * W;
        const float px = pred[(size_t)idx * 3], py = pred[(size_t)idx * 3 + 1], pz = pred[(size_t)idx * 3 + 2];
        const float dx = px - gt[(size_t)idx * 3], dy = py - gt[(size_t)idx * 3 + 1], dz = pz - gt[(size_t)idx * 3 + 2];
        const float l = ((fabsf(dx) + fabsf(dy)) + fabsf(dz)) / 3.0f;
        const float craw = conf ? conf[idx] : 1.0f;
        const float cc = (craw < kConfMin) ? kConfMin : ((craw > kConfMax) ? kConfMax : craw);
        sum_b = cc * l - a.alpha * logf(cc);
        float gz = sgnf(dz) * cc * a.kb;
        if (th) {
            auto G = [&](int q) { return load_gray_px(th, a.tch, plane, (size_t)q); };
            auto Z = [&](int q) { return pred[(size_t)q * 3 + 2]; };
            const float g0 = G(idx);
            if (j < W - 1) {
                const float s = Z(idx + 1) - pz, e = expf(-fabsf(G(idx + 1) - g0) * 10.f);
                sum_e += fabsf(s) * e * a.sx;
                gz -= sgnf(s) * e * a.kx;
            }
            if (i < H - 1) {
                const float s = Z(idx + W) - pz, e = expf(-fabsf(G(idx + W) - g0) * 10.f);
                sum_e += fabsf(s) * e * a.sy;
                gz -= sgnf(s) * e * a.ky;
            }
            if (j > 0) gz += sgnf(pz - Z(idx - 1)) * expf(-fabsf(g0 - G(idx - 1)) * 10.f) * a.kx;
            if (i > 0) gz += sgnf(pz - Z(idx - W)) * expf(-fabsf(g0 - G(idx - W)) * 10.f) * a.ky;
        }
        if (BWD) {
            float* o = a.dpred[view] + ((size_t)b * plane + idx) * 3;
            o[0] = sgnf(dx) * cc * a.kb; o[1] = sgnf(dy) * cc * a.kb; o[2] = gz;
            if (a.dconf[view]) {
                const bool inside = (craw >= kConfMin) && (craw <= kConfMax);
                a.dconf[view][(size_t)b * plane + idx] = inside ? (l - a.alpha / cc) * a.kc : 0.f;
            }
        }
    }
    sum_b = warp_sum(sum_b); sum_e = warp_sum(sum_e);
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = sum_b; red[threadIdx.x >> 5][1] = sum_e; }
    __syncthreads();
    if (threadIdx.x < kNTerms) {
        float v = 0.f;
        if (threadIdx.x < 3) for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x == 0 ? 0 : 1];   // [0] basic, [1] = [2] = edge
        a.partials[((size_t)img * a.blocks + blockIdx.x) * kNTerms + threadIdx.x] = v;
    }
}

// ------------------------------------------------------------------ host helpers
struct WsLayout {
    size_t stats_partials, loss_partials, counter, total;
    size_t s2_partials, s2_dzp;        // multi-scale only (appended: the other offsets do not depend on `multi`)
    int stiles_x, stiles_y, tiles_x, tiles_y, s2_tiles_x, s2_tiles_y;
    int sm_bands, sm_strips;           // work items per image-view of the marching statistics kernel
};

WsLayout ws_layout(int B, int H, int W, int multi = 0) {
    WsLayout L;
    L.stiles_x = (W + kSTW - 1) / kSTW; L.stiles_y = (H + kSTH - 1) / kSTH;
    L.tiles_x = (W + kTW - 1) / kTW;    L.tiles_y = (H + kTH - 1) / kTH;
    size_t off = 0;
    L.counter = off;        off += 256;
    L.sm_bands = (H + kStatsMarchRows - 1) / kStatsMarchRows; L.sm_strips = (W + 127) / 128;
    const size_t stats_tiles = (size_t)max(L.stiles_x * L.stiles_y, L.sm_bands * L.sm_strips);
    L.stats_partials = off; off += t3d_align_up((size_t)B * 2 * stats_tiles * 4 * sizeof(float), 256);
    // sized for the tile kernel (16-row tiles) and the marching kernel (>= 8-row bands)
    L.loss_partials = off;  off += t3d_align_up((size_t)B * 2 * L.tiles_x * ((H + 7) / 8) * kNTerms * sizeof(float), 256);
    t3d_scale2_tiles(H, W, &L.s2_tiles_x, &L.s2_tiles_y);
    L.s2_partials = L.s2_dzp = off;
    if (multi) {
        L.s2_partials = off; off += t3d_align_up((size_t)B * 2 * L.s2_tiles_x * L.s2_tiles_y * 4 * sizeof(float), 256);
        L.s2_dzp = off;      off += t3d_align_up((size_t)B * 2 * (H >> 1) * (W >> 1) * sizeof(float), 256);
    }
    L.total = off;
    return L;
}

inline float __int_as_float_host(unsigned int u) { float f; memcpy(&f, &u, sizeof(f)); return f; }

// optional event recorded right behind the main (marching / tile) kernel of the next loss call of this thread
thread_local cudaEvent_t g_main_done_event = nullptr;

int check_dims(int B, int H, int W) {
    T3D_REQUIRE(B >= 1 && H >= 1 && W >= 1, "bad dims B=%d H=%d W=%d", B, H, W);
    T3D_REQUIRE((double)B * 2.0 * H * W < 2.0e9, "problem too large for 32-bit tile indexing");
    return T3D_OK;
}

template <bool MULTI>
int launch_stats_march(const StatsArgs& sa, int nbands, int nstrips, cudaStream_t st) {
    const int items = sa.B * 2 * nbands * nstrips;
    const int grid = (items + kSMWarps - 1) / kSMWarps;
    if (sa.replicated) T3D_LAUNCH("thermal_stats_march_kernel", st, (thermal_stats_march_kernel<MULTI, 2><<<grid, kSMWarps * 32, 0, st>>>(sa, nbands, nstrips, kStatsMarchRows)));
    else if (sa.tch == 3) T3D_LAUNCH("thermal_stats_march_kernel", st, (thermal_stats_march_kernel<MULTI, 1><<<grid, kSMWarps * 32, 0, st>>>(sa, nbands, nstrips, kStatsMarchRows)));
    else T3D_LAUNCH("thermal_stats_march_kernel", st, (thermal_stats_march_kernel<MULTI, 0><<<grid, kSMWarps * 32, 0, st>>>(sa, nbands, nstrips, kStatsMarchRows)));
    return T3D_OK;
}

template <bool MULTI, bool VEC>
int launch_stats(const StatsArgs& sa, cudaStream_t st) {
    const int grid = sa.B * 2 * sa.tiles_x * sa.tiles_y;
    T3D_LAUNCH("thermal_stats_kernel", st, thermal_stats_kernel<MULTI, VEC><<<grid, kSThreads, 0, st>>>(sa));
    return T3D_OK;
}

// *stiles_out = partial sums per image-view this run leaves in `partials` ([view][b][stiles][4])
int run_stats(const float* t1, const float* t2, int tch, int B, int H, int W, int multi,
              float* partials, const WsLayout& L, cudaStream_t st, int replicated, int* stiles_out) {
    StatsArgs sa;
    sa.replicated = (replicated && tch == 3) ? 1 : 0;
    sa.thermal[0] = t1; sa.thermal[1] = t2; sa.partials = partials;
    sa.B = B; sa.H = H; sa.W = W; sa.tch = tch; sa.tiles_x = L.stiles_x; sa.tiles_y = L.stiles_y;
    const bool vec = (W % 4 == 0) && t3d_aligned16(t1) && t3d_aligned16(t2);
    if (vec) {
        *stiles_out = L.sm_bands * L.sm_strips;
        return multi ? launch_stats_march<true>(sa, L.sm_bands, L.sm_strips, st) : launch_stats_march<false>(sa, L.sm_bands, L.sm_strips, st);
    }
    *stiles_out = L.stiles_x * L.stiles_y;
    return multi ? launch_stats<true, false>(sa, st) : launch_stats<false, false>(sa, st);
}

template <bool MULTI, bool VEC, bool BWD>
int launch_loss(const LossArgs& la, cudaStream_t st) {
    static bool attr_done[kT3dMaxDevices] = {};   // per device; benign race: idempotent
    bool& attr_set = attr_done[t3d_device_slot()];
    constexpr size_t smem = loss_smem_bytes<MULTI>();
    if (!attr_set) {
        T3D_CUDA(cudaFuncSetAttribute(loss_tile_kernel<MULTI, VEC, BWD>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    const int grid = la.B * 2 * la.tiles_x * la.tiles_y;
    T3D_LAUNCH("loss_tile_kernel", st, loss_tile_kernel<MULTI, VEC, BWD><<<grid, kThreads, smem, st>>>(la));
    return T3D_OK;
}

int loss_impl(bool bwd, const float* pred1, const float* pred2, const float* gt1, const float* gt2,
              const float* conf1, const float* conf2, const float* thermal1, const float* thermal2,
              int tch, const float* ustats1, const float* ustats2, int ustats_tiles, float* dpred1, float* dpred2, float* dconf1, float* dconf2,
              int B, int H, int W, int flags, float alpha, float ew, float sw, float dw, float gscale,
              float* out_sample, float* out_batch, double* out_f64,
              void* workspace, size_t ws_bytes, void* stream,
              int gt_h = 0, int gt_w = 0, int conf_h = 0, int conf_w = 0) {
    if (int rc = check_dims(B, H, W)) return rc;
    T3D_REQUIRE((flags & ~(T3D_LOSS_MULTI_SCALE | T3D_LOSS_CONF_MIN_ONLY | T3D_LOSS_STATS_TWO_SCALES)) == 0, "unknown loss flags 0x%x", flags);
    if (gt_h == H && gt_w == W) gt_h = gt_w = 0;                    // same size: direct reads
    if (conf_h == H && conf_w == W) conf_h = conf_w = 0;
    T3D_REQUIRE((gt_h == 0) == (gt_w == 0) && gt_h >= 0 && (conf_h == 0) == (conf_w == 0) && conf_h >= 0, "bad gt / conf size");
    const bool resampled = gt_h != 0 || conf_h != 0;
    const int multi = (flags & T3D_LOSS_MULTI_SCALE) ? 1 : 0;
    const bool conf_min_only = (flags & T3D_LOSS_CONF_MIN_ONLY) != 0;
    T3D_REQUIRE(pred1 && pred2 && gt1 && gt2, "pred/gt pointers must not be NULL");
    T3D_REQUIRE(out_sample && out_batch && workspace, "output / workspace pointers must not be NULL");
    const bool thermal_on = thermal1 != nullptr && thermal2 != nullptr;   // utils/loss.py:116
    const int replicated = (tch == (3 | T3D_THERMAL_REPLICATED));
    if (replicated) tch = 3;
    if (thermal_on) T3D_REQUIRE(tch == 1 || tch == 3, "thermal_channels must be 1, 3 or 3 | T3D_THERMAL_REPLICATED, got %d", tch);
    if (bwd) T3D_REQUIRE(dpred1 && dpred2, "dpred pointers must not be NULL");
    const WsLayout L = ws_layout(B, H, W, multi);
    if (ws_bytes < L.total) {
        t3d_set_error("workspace too small: %zu < %zu", ws_bytes, L.total);
        return T3D_ERR_WORKSPACE;
    }
    T3D_REQUIRE(t3d_aligned16(workspace), "workspace must be 16-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char* ws = reinterpret_cast<char*>(workspace);
    float* stats_partials = reinterpret_cast<float*>(ws + L.stats_partials);
    float* loss_partials = reinterpret_cast<float*>(ws + L.loss_partials);
    unsigned int* counter = reinterpret_cast<unsigned int*>(ws + L.counter);

    T3D_CUDA(cudaMemsetAsync(counter, 0, 2 * sizeof(unsigned int), st));   // [0] finalize ticket, [1] work queue
    // thermal-gradient statistics: supplied by the caller (fused into the preprocessing) or computed here
    const bool user_stats = thermal_on && (!multi || (flags & T3D_LOSS_STATS_TWO_SCALES)) && ustats1 && ustats2 && ustats_tiles > 0;
    const float* stats_v[2] = {stats_partials, stats_partials};
    int stiles = 0;
    if (user_stats) { stats_v[0] = ustats1; stats_v[1] = ustats2; stiles = ustats_tiles; }
    else if (thermal_on) {
        if (int rc = run_stats(thermal1, thermal2, tch, B, H, W, multi, stats_partials, L, st, replicated, &stiles)) return rc;
        stats_v[1] = stats_partials + (size_t)B * stiles * 4;
    }

    LossArgs la;
    la.pred[0] = pred1; la.pred[1] = pred2; la.gt[0] = gt1; la.gt[1] = gt2;
    la.conf[0] = conf1; la.conf[1] = conf2;
    la.thermal[0] = thermal_on ? thermal1 : nullptr; la.thermal[1] = thermal_on ? thermal2 : nullptr;
    la.dpred[0] = dpred1; la.dpred[1] = dpred2; la.dconf[0] = dconf1; la.dconf[1] = dconf2;
    la.stats[0] = stats_v[0]; la.stats[1] = stats_v[1]; la.partials = loss_partials;
    la.B = B; la.H = H; la.W = W; la.tch = thermal_on ? tch : 0;
    la.tiles_x = L.tiles_x; la.tiles_y = L.tiles_y; la.stiles = stiles;
    la.alpha = alpha;
    la.conf_max = conf_min_only ? __int_as_float_host(0x7f800000u) : kConfMax;
    la.gt_h = gt_h; la.gt_w = gt_w; la.conf_h = conf_h; la.conf_w = conf_w;
    const double N = (double)H * W, n2 = (double)(H / 2) * (W / 2);
    la.kb = (float)((double)gscale / (3.0 * N));
    la.kc = (float)((double)gscale / N);
    la.kE[0] = (float)((double)gscale * ew / N); la.kS[0] = (float)((double)gscale * sw / N);
    la.kD[0] = (float)((double)gscale * dw / N);
    const double l2 = (n2 > 0) ? (double)kScale2Weight / n2 : 0.0;
    la.kE[1] = (float)((double)gscale * ew * l2); la.kS[1] = (float)((double)gscale * sw * l2);
    la.kD[1] = (float)((double)gscale * dw * l2);

    bool vec = (W % 4 == 0) && t3d_aligned16(pred1) && t3d_aligned16(pred2) && (gt_h != 0 || (t3d_aligned16(gt1) &&
               t3d_aligned16(gt2))) && (conf_h != 0 || (t3d_aligned16(conf1) && t3d_aligned16(conf2))) &&
               t3d_aligned16(thermal1) && t3d_aligned16(thermal2) && t3d_aligned16(dpred1) &&
               t3d_aligned16(dpred2) && t3d_aligned16(dconf1) && t3d_aligned16(dconf2);
    const bool ms = multi && thermal_on;
    int n_partials = L.tiles_x * L.tiles_y;
    int rc;
    const float* partials2 = nullptr;
    int tiles2 = 0;
    // gt at another size, downsampled: the marching kernel resamples it as it stages the rows (loss_march_rs_kernel)
    // when a strip's source segment is one it is faster at (gt_w ~ W); wider segments, upsampled gt, a gt-sized
    // confidence, multi-scale: tile kernel
    int rs_span = 0;
    const bool march_rs = vec && thermal_on && !conf_min_only && !ms && gt_h != 0 && conf_h == 0 &&
                          gt_h >= H && gt_w >= W && gt_w % 4 == 0 && t3d_aligned16(gt1) && t3d_aligned16(gt2) &&
                          t3d_loss_march_rs_fits(rs_span = t3d_loss_march_rs_span(W, gt_w));
    if (vec && thermal_on && !conf_min_only && (!resampled || march_rs) && (!ms || (H >= 4 && W >= 4))) {
        // fast path: TMA-fed warp-marching kernel (t3d_loss_march.cu); multi-scale: the half-resolution terms run
        // first as their own pass (t3d_loss_scale2.cu) and hand their gradient to the marching kernel
        MarchArgs ma;
        for (int v = 0; v < 2; ++v) {
            ma.pred[v] = la.pred[v]; ma.gt[v] = la.gt[v]; ma.conf[v] = la.conf[v]; ma.thermal[v] = la.thermal[v];
            ma.dpred[v] = la.dpred[v]; ma.dconf[v] = la.dconf[v]; ma.dzp[v] = nullptr;
        }
        // multi-scale with one staged thermal plane: both scales in one pass over the rows (loss_march_ms_kernel)
        const bool fused_ms = ms && (tch == 1 || replicated);
        if (ms && !fused_ms) {
            Scale2Args sa;
            float* dzp = reinterpret_cast<float*>(ws + L.s2_dzp);
            for (int v = 0; v < 2; ++v) {
                sa.pred[v] = la.pred[v]; sa.gt[v] = la.gt[v]; sa.thermal[v] = la.thermal[v]; sa.stats[v] = stats_v[v];
                sa.dzp[v] = dzp + (size_t)v * B * (H >> 1) * (W >> 1);
                if (bwd) ma.dzp[v] = sa.dzp[v];
            }
            sa.partials = reinterpret_cast<float*>(ws + L.s2_partials);
            sa.B = B; sa.H = H; sa.W = W; sa.tch = tch; sa.replicated = replicated; sa.stiles = stiles;
            sa.tiles_x = L.s2_tiles_x; sa.tiles_y = L.s2_tiles_y;
            sa.kE = la.kE[1]; sa.kS = la.kS[1]; sa.kD = la.kD[1];
            if (int rc2 = t3d_launch_loss_scale2(sa, bwd, st)) return rc2;
            partials2 = sa.partials; tiles2 = sa.tiles_x * sa.tiles_y;
        }
        ma.stats[0] = stats_v[0]; ma.stats[1] = stats_v[1]; ma.partials = loss_partials; ma.queue = counter + 1;
        ma.B = B; ma.H = H; ma.W = W; ma.tch = tch; ma.stiles = la.stiles; ma.replicated = replicated;
        // bands of 32 rows (a band re-reads the row above and the row below it: taller = less overfetch), the last ~1/8
        // of the image in 8-row bands queued behind all the large ones (shorter tail of the persistent grid); other band
        // heights and tails: DESIGN §4 experiment 12 and §5
        constexpr int kMarchRows = 32, kMarchTailDiv = 8;
        // (one-pass multi-scale: a band brings 4 halo rows instead of 2 and must start on an even row: 16-row tail bands)
        const int rows_l = kMarchRows, rows_s = fused_ms ? 16 : 8;
        const int small_rows = ((H / kMarchTailDiv + rows_s - 1) / rows_s) * rows_s;
        ma.rows_l = rows_l; ma.rows_s = rows_s;
        ma.nbands_l = (small_rows > 0) ? max(0, H - small_rows) / rows_l : (H + rows_l - 1) / rows_l;
        if (small_rows == 0) { ma.nbands_s = 0; /* the last large band may be ragged: handle it as one small band */
            if (ma.nbands_l * rows_l > H) { ma.nbands_l -= 1; ma.rows_s = rows_l; ma.nbands_s = 1; } }
        else ma.nbands_s = (H - ma.nbands_l * rows_l + rows_s - 1) / rows_s;
        ma.nstrips = (W + 127) / 128;
        ma.alpha = alpha; ma.kb = la.kb; ma.kc = la.kc; ma.kE = la.kE[0]; ma.kS = la.kS[0]; ma.kD = la.kD[0];
        ma.kE2 = la.kE[1]; ma.kS2 = la.kS[1]; ma.kD2 = la.kD[1];
        ma.gt_h = gt_h; ma.gt_w = gt_w;
        n_partials = (ma.nbands_l + ma.nbands_s) * ma.nstrips;
        rc = march_rs ? t3d_launch_loss_march_rs(ma, rs_span, bwd, st)
           : fused_ms ? t3d_launch_loss_march_ms(ma, bwd, st) : t3d_launch_loss_march(ma, bwd, st);
    } else if (bwd) {
        if (ms) rc = vec ? launch_loss<true, true, true>(la, st) : launch_loss<true, false, true>(la, st);
        else    rc = vec ? launch_loss<false, true, true>(la, st) : launch_loss<false, false, true>(la, st);
    } else {
        if (ms) rc = vec ? launch_loss<true, true, false>(la, st) : launch_loss<true, false, false>(la, st);
        else    rc = vec ? launch_loss<false, true, false>(la, st) : launch_loss<false, false, false>(la, st);
    }
    if (rc) return rc;
    if (g_main_done_event) {            // t3d_loss_set_main_done_event: lets a caller overlap the second stage with other work
        T3D_CUDA(cudaEventRecord(g_main_done_event, st));
        g_main_done_event = nullptr;
    }

    FinalizeArgs fa;
    fa.partials = loss_partials; fa.out_sample = out_sample; fa.out_batch = out_batch; fa.out_f64 = out_f64;
    fa.partials2 = partials2; fa.tiles2 = tiles2;
    fa.counter = counter; fa.B = B; fa.H = H; fa.W = W; fa.tiles = n_partials;
    fa.multi = ms ? 1 : 0; fa.thermal_on = thermal_on ? 1 : 0; fa.ew = ew; fa.sw = sw; fa.dw = dw;
    T3D_LAUNCH("loss_finalize_kernel", st, loss_finalize_kernel<<<B, 128, 0, st>>>(fa));
    return T3D_OK;
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int t3d_loss_set_main_done_event(void* cuda_event) {
    g_main_done_event = reinterpret_cast<cudaEvent_t>(cuda_event);
    return T3D_OK;
}

size_t t3d_loss_workspace_bytes(int B, int H, int W, int flags) {
    if (B < 1 || H < 1 || W < 1) return 0;
    return ws_layout(B, H, W, (flags & T3D_LOSS_MULTI_SCALE) ? 1 : 0).total;
}

int t3d_thermal_grad_stats(const float* thermal1, const float* thermal2, int thermal_channels,
                           int B, int H, int W, int multi_scale, float* out_stats,
                           void* workspace, size_t workspace_bytes, void* stream) {
    if (int rc = check_dims(B, H, W)) return rc;
    T3D_REQUIRE(thermal1 && thermal2 && out_stats && workspace, "NULL pointer");
    T3D_REQUIRE(thermal_channels == 1 || thermal_channels == 3, "thermal_channels must be 1 or 3");
    const WsLayout L = ws_layout(B, H, W);
    if (workspace_bytes < L.total) { t3d_set_error("workspace too small"); return T3D_ERR_WORKSPACE; }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + L.stats_partials);
    int stiles = 0;
    if (int rc = run_stats(thermal1, thermal2, thermal_channels, B, H, W, multi_scale, partials, L, st, 0, &stiles)) return rc;
    T3D_LAUNCH("thermal_stats_finalize_kernel", st, thermal_stats_finalize_kernel<<<B * 2, 32, 0, st>>>(partials, stiles, B, H, W, multi_scale, out_stats));
    return T3D_OK;
}

int t3d_loss_fwd_bwd(const float* pred1, const float* pred2, const float* gt1, const float* gt2,
                     const float* conf1, const float* conf2,
                     const float* thermal1, const float* thermal2, int thermal_channels,
                     const float* thermal_stats1, const float* thermal_stats2, int stats_tiles,
                     float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                     int B, int H, int W, int multi_scale,
                     float alpha, float edge_weight, float smoothness_weight, float detail_weight,
                     float grad_scale, float* out_sample, float* out_batch, double* out_sample_f64,
                     void* workspace, size_t workspace_bytes, void* stream) {
    return loss_impl(true, pred1, pred2, gt1, gt2, conf1, conf2, thermal1, thermal2, thermal_channels,
                     thermal_stats1, thermal_stats2, stats_tiles, dpred1, dpred2, dconf1, dconf2, B, H, W, multi_scale, alpha, edge_weight,
                     smoothness_weight, detail_weight, grad_scale, out_sample, out_batch, out_sample_f64,
                     workspace, workspace_bytes, stream);
}

int t3d_loss_fwd_bwd_resampled_stats(const float* pred1, const float* pred2, const float* gt1, const float* gt2,
                                     int gt_h, int gt_w, const float* conf1, const float* conf2, int conf_h, int conf_w,
                                     const float* thermal1, const float* thermal2, int thermal_channels,
                                     const float* thermal_stats1, const float* thermal_stats2, int stats_tiles,
                                     float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                                     int B, int H, int W, int flags,
                                     float alpha, float edge_weight, float smoothness_weight, float detail_weight,
                                     float grad_scale, float* out_sample, float* out_batch, double* out_sample_f64,
                                     void* workspace, size_t workspace_bytes, void* stream) {
    T3D_REQUIRE(gt_h >= 1 && gt_w >= 1, "bad gt size");
    T3D_REQUIRE((conf1 == nullptr && conf2 == nullptr) || (conf_h >= 1 && conf_w >= 1), "bad conf size");
    T3D_REQUIRE(!(dconf1 || dconf2) || (conf_h == H && conf_w == W), "a confidence that takes a gradient has the prediction's size");
    const bool bwd = dpred1 != nullptr && dpred2 != nullptr;
    return loss_impl(bwd, pred1, pred2, gt1, gt2, conf1, conf2, thermal1, thermal2, thermal_channels,
                     thermal_stats1, thermal_stats2, stats_tiles, dpred1, dpred2, dconf1, dconf2, B, H, W, flags, alpha,
                     edge_weight, smoothness_weight, detail_weight, grad_scale, out_sample, out_batch, out_sample_f64,
                     workspace, workspace_bytes, stream, gt_h, gt_w, conf1 ? conf_h : 0, conf1 ? conf_w : 0);
}

int t3d_loss_fwd_bwd_resampled(const float* pred1, const float* pred2, const float* gt1, const float* gt2, int gt_h, int gt_w,
                               const float* conf1, const float* conf2, int conf_h, int conf_w,
                               const float* thermal1, const float* thermal2, int thermal_channels,
                               float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                               int B, int H, int W, int flags,
                               float alpha, float edge_weight, float smoothness_weight, float detail_weight,
                               float grad_scale, float* out_sample, float* out_batch, double* out_sample_f64,
                               void* workspace, size_t workspace_bytes, void* stream) {
    return t3d_loss_fwd_bwd_resampled_stats(pred1, pred2, gt1, gt2, gt_h, gt_w, conf1, conf2, conf_h, conf_w,
                                            thermal1, thermal2, thermal_channels, nullptr, nullptr, 0,
                                            dpred1, dpred2, dconf1, dconf2, B, H, W, flags, alpha, edge_weight,
                                            smoothness_weight, detail_weight, grad_scale, out_sample, out_batch,
                                            out_sample_f64, workspace, workspace_bytes, stream);
}

int t3d_loss_fwd(const float* pred1, const float* pred2, const float* gt1, const float* gt2,
                 const float* conf1, const float* conf2,
                 const float* thermal1, const float* thermal2, int thermal_channels,
                 const float* thermal_stats1, const float* thermal_stats2, int stats_tiles,
                 int B, int H, int W, int multi_scale,
                 float alpha, float edge_weight, float smoothness_weight, float detail_weight,
                 float* out_sample, float* out_batch, double* out_sample_f64,
                 void* workspace, size_t workspace_bytes, void* stream) {
    return loss_impl(false, pred1, pred2, gt1, gt2, conf1, conf2, thermal1, thermal2, thermal_channels,
                     thermal_stats1, thermal_stats2, stats_tiles, nullptr, nullptr, nullptr, nullptr, B, H, W, multi_scale, alpha, edge_weight,
                     smoothness_weight, detail_weight, 1.0f, out_sample, out_batch, out_sample_f64,
                     workspace, workspace_bytes, stream);
}

static int scale_common(int mode, float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                        const float* out_sample, const float* out_batch, const float* grad_output,
                        int B, int H, int W, void* stream) {
    if (int rc = check_dims(B, H, W)) return rc;
    ScaleArgs sa;
    sa.dpred[0] = dpred1; sa.dpred[1] = dpred2; sa.dconf[0] = dconf1; sa.dconf[1] = dconf2;
    sa.out_sample = out_sample; sa.out_batch = out_batch; sa.grad_output = grad_output;
    sa.B = B; sa.plane = (size_t)H * W;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int grid = t3d_sm_count() * 8;
    if (mode == 0) T3D_LAUNCH("scale_grads_kernel", st, scale_grads_kernel<0><<<grid, 256, 0, st>>>(sa));
    else T3D_LAUNCH("scale_grads_kernel", st, scale_grads_kernel<1><<<grid, 256, 0, st>>>(sa));
    return T3D_OK;
}

int t3d_loss_rescale_invalid(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                             const float* out_sample, const float* out_batch,
                             int B, int H, int W, void* stream) {
    T3D_REQUIRE(out_sample && out_batch, "NULL pointer");
    return scale_common(0, dpred1, dpred2, dconf1, dconf2, out_sample, out_batch, nullptr, B, H, W, stream);
}

int t3d_scale_grads(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                    const float* grad_output, int B, int H, int W, void* stream) {
    T3D_REQUIRE(grad_output, "NULL pointer");
    return scale_common(1, dpred1, dpred2, dconf1, dconf2, nullptr, nullptr, grad_output, B, H, W, stream);
}

int t3d_loss_v1_fwd_bwd(const float* pred1, const float* pred2, const float* gt1, const float* gt2,
                        const float* conf1, const float* conf2,
                        const float* thermal1, const float* thermal2, int thermal_channels,
                        float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                        int B, int H, int W,
                        float alpha, float edge_weight, float smoothness_weight, float grad_scale,
                        float* out_sample, float* out_batch, double* out_sample_f64,
                        void* workspace, size_t workspace_bytes, void* stream) {
    if (int rc = check_dims(B, H, W)) return rc;
    T3D_REQUIRE(pred1 && pred2 && gt1 && gt2 && out_sample && out_batch && workspace, "NULL pointer");
    const bool thermal_on = thermal1 != nullptr && thermal2 != nullptr;
    if (thermal_on) T3D_REQUIRE(thermal_channels == 1 || thermal_channels == 3, "thermal_channels must be 1 or 3");
    const bool bwd = dpred1 != nullptr && dpred2 != nullptr;
    const size_t plane = (size_t)H * W;
    const int blocks = (int)((plane + 255) / 256);
    const size_t need = 256 + t3d_align_up((size_t)B * 2 * blocks * kNTerms * sizeof(float), 256);
    if (workspace_bytes < need) { t3d_set_error("workspace too small: %zu < %zu", workspace_bytes, need); return T3D_ERR_WORKSPACE; }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    unsigned int* counter = reinterpret_cast<unsigned int*>(workspace);
    float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + 256);
    T3D_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned int), st));
    V1Args a;
    a.pred[0] = pred1; a.pred[1] = pred2; a.gt[0] = gt1; a.gt[1] = gt2; a.conf[0] = conf1; a.conf[1] = conf2;
    a.thermal[0] = thermal1; a.thermal[1] = thermal2; a.dpred[0] = dpred1; a.dpred[1] = dpred2;
    a.dconf[0] = dconf1; a.dconf[1] = dconf2; a.partials = partials;
    a.B = B; a.H = H; a.W = W; a.tch = thermal_on ? thermal_channels : 0; a.blocks = blocks;
    const double N = (double)plane, nx = (double)H * (W - 1), ny = (double)(H - 1) * W;
    const double wsum = (double)edge_weight + (double)smoothness_weight;
    a.alpha = alpha; a.kb = (float)(grad_scale / (3.0 * N)); a.kc = (float)(grad_scale / N);
    a.kx = (float)(grad_scale * wsum / nx); a.ky = (float)(grad_scale * wsum / ny);   // W == 1 or H == 1: inf -> NaN like mean(empty)
    a.sx = (float)(N / nx); a.sy = (float)(N / ny);
    dim3 grid((unsigned)blocks, (unsigned)(B * 2));
    if (bwd) T3D_LAUNCH("loss_v1_kernel", st, loss_v1_kernel<true><<<grid, 256, 0, st>>>(a));
    else T3D_LAUNCH("loss_v1_kernel", st, loss_v1_kernel<false><<<grid, 256, 0, st>>>(a));
    FinalizeArgs fa;
    fa.partials = partials; fa.out_sample = out_sample; fa.out_batch = out_batch; fa.out_f64 = out_sample_f64;
    fa.partials2 = nullptr; fa.tiles2 = 0;
    fa.counter = counter; fa.B = B; fa.H = H; fa.W = W; fa.tiles = blocks;
    fa.multi = 0; fa.thermal_on = thermal_on ? 1 : 0; fa.ew = edge_weight; fa.sw = smoothness_weight; fa.dw = 0.f;
    T3D_LAUNCH("loss_finalize_kernel", st, loss_finalize_kernel<<<B, 128, 0, st>>>(fa));
    return T3D_OK;
}

size_t t3d_loss_v1_workspace_bytes(int B, int H, int W) {
    if (B < 1 || H < 1 || W < 1) return 0;
    const size_t blocks = ((size_t)H * W + 255) / 256;
    return 256 + t3d_align_up((size_t)B * 2 * blocks * kNTerms * sizeof(float), 256);
}

}  // extern "C"
