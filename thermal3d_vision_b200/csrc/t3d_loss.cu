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

// ------------------------------------------------------------------ fused loss tile kernel
constexpr int kTH = 16, kTW = 128, kThreads = 256;
constexpr int kPW = kTW + 8;          // raw plane row stride: col j -> c = j - j0 + 4
constexpr int kQPT = kTH * kTW / 4 / kThreads;  // quads per thread (2)
constexpr int kP2H = kTH / 2 + 2, kP2W = kTW / 2 + 4;  // pooled planes: (I,J) -> R = I-I0+1, C = J-J0+1

struct LossArgs {
    LossOperands op;
    const float* thermal[2];
    const float* stats[2];        // per view: [B][stiles][4]
    float* partials;              // [B*2][tiles][kNTerms]
    int B, H, W, tch, tiles_x, tiles_y, stiles;
    float kE[2], kS[2], kD[2];    // grad_scale * lambda_s * weight / n_s
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

// The confidence-weighted L1 term of one pixel (utils/loss.py:81-98) and its closed-form gradient: the tile kernel's
// per-pixel expressions, which loss_basic_kernel evaluates so that both write the same gradient bits.  p, g: the
// pixel's xyz; craw: its raw confidence; the term is added to `sum`.  Returns d/dpred xyz and d/dconf (BWD).
struct BasicGrad { float gx, gy, gz, dc; };
template <bool BWD>
__device__ __forceinline__ BasicGrad basic_px(float px, float py, float pz, float gx, float gy, float gz, float craw,
                                              float conf_max, float alpha, float kb, float kc, float& sum) {
    BasicGrad r = {0.f, 0.f, 0.f, 0.f};
    const float dx = px - gx, dy = py - gy, dz = pz - gz;
    const float l = ((fabsf(dx) + fabsf(dy)) + fabsf(dz)) / 3.0f;                 // utils/loss.py:82
    const float cc = (craw < kConfMin) ? kConfMin : ((craw > conf_max) ? conf_max : craw);   // :91, NaN passes
    sum += cc * l - alpha * logf(cc);                                              // :95
    if (BWD) {
        const float kc3 = cc * kb;
        r.gx = sgnf(dx) * kc3;
        r.gy = sgnf(dy) * kc3;
        r.gz = sgnf(dz) * kc3;
        const bool inside = (craw >= kConfMin) && (craw <= conf_max);              // clamp grad mask (inclusive)
        r.dc = inside ? (l - alpha / cc) * kc : 0.f;
    }
    return r;
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

    const float* __restrict__ pred = a.op.pred[view] + (size_t)b * plane * 3;
    const bool gt_rs = a.gt_h != 0, conf_rs = a.conf_h != 0;        // block-uniform: bilinear taps instead of direct reads
    const float* __restrict__ gt = a.op.gt[view] + (size_t)b * (gt_rs ? (size_t)a.gt_h * a.gt_w : plane) * 3;
    const float* __restrict__ conf = a.op.conf[view] ? a.op.conf[view] + (size_t)b * (conf_rs ? (size_t)a.conf_h * a.conf_w : plane) : nullptr;
    const float gsy = gt_rs ? (float)a.gt_h / (float)H : 1.f, gsx = gt_rs ? (float)a.gt_w / (float)W : 1.f;
    const float csy = conf_rs ? (float)a.conf_h / (float)H : 1.f, csx = conf_rs ? (float)a.conf_w / (float)W : 1.f;
    const float* __restrict__ th = thermal_on ? a.thermal[view] + (size_t)b * a.tch * plane : nullptr;
    float* __restrict__ dpred = BWD ? a.op.dpred[view] + (size_t)b * plane * 3 : nullptr;
    float* __restrict__ dconf = (BWD && a.op.dconf[view]) ? a.op.dconf[view] + (size_t)b * plane : nullptr;

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
                // (basic_px, written out: through the helper, ptxas allocates the registers of the two unaligned
                // backward instances differently)
                const float dx = p[3 * e] - g[3 * e], dy = p[3 * e + 1] - g[3 * e + 1], dz = p[3 * e + 2] - g[3 * e + 2];
                const float l = ((fabsf(dx) + fabsf(dy)) + fabsf(dz)) / 3.0f;             // utils/loss.py:82
                const float craw = c[e];
                const float cc = (craw < kConfMin) ? kConfMin : ((craw > a.op.conf_max) ? a.op.conf_max : craw);   // :91, NaN passes
                const bool ok = e < nvalid;
                if (ok) sum_basic += cc * l - a.op.alpha * logf(cc);                          // :95
                zq[e] = p[3 * e + 2];
                gzq[e] = g[3 * e + 2];
                if (BWD) {
                    const float kc3 = cc * a.op.kb;
                    gq[k][3 * e] = sgnf(dx) * kc3;
                    gq[k][3 * e + 1] = sgnf(dy) * kc3;
                    gq[k][3 * e + 2] = sgnf(dz) * kc3;
                    const bool inside = (craw >= kConfMin) && (craw <= a.op.conf_max);       // clamp grad mask (inclusive)
                    dc[e] = inside ? (l - a.op.alpha / cc) * a.op.kc : 0.f;
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

// ------------------------------------------------------------------ basic term only (no thermal images)
// loss_basic_kernel: the confidence-weighted L1 term alone -- train_thermal_dustr.py:305-318 (the loss without
// --use_thermal_aware_loss), the validation loss (:465-492), confidence_weighted_regression_loss.  No stencil: a pure
// per-pixel stream with one sum per sample.  Persistent grid; a warp pulls work items from the BandQueue
// (t3d_loss_internal.cuh) as loss_march_kernel does.  Each lane owns 4 pixels of a row: three 128-bit loads each of pred and gt (AoS),
// one of the confidence, 128-bit streaming stores of d/dpred and d/dconf; one row per lane in flight, the latency is
// covered by 20 (backward) / 32 (forward) resident warps per SM.  One partial per item (fixed butterfly), so a sample's
// sums depend neither on its position in the batch nor on the batch size.
// RS: the gt is downsampled (gt_h >= H, gt_w >= W), read through the bilinear taps of t3d_bilinear.cuh -- the
// arithmetic of interp_bilinear_kernel, so the result is bit-identical to resampling first.
struct BasicArgs {
    LossOperands op;
    float* partials;              // [B*2][bq.per_image_view()][kNTerms]: basic, 0 ...
    BandQueue bq;
    int B, H, W;
    int gt_h, gt_w;               // RS: size of the gt arrays
};
// 4-warp CTAs: the backward instance needs 87 registers (5 CTAs = 20 warps per SM without spilling), forward 64 (32);
// with the gt taps (RS) 166 / 128: 3 / 4 CTAs
constexpr int kBWarps = 4;
template <bool BWD, bool RS> constexpr int basic_blocks_per_sm() { return RS ? (BWD ? 3 : 4) : (BWD ? 5 : 8); }

template <bool BWD, bool RS>
__global__ void __launch_bounds__(kBWarps * 32, basic_blocks_per_sm<BWD, RS>()) loss_basic_kernel(const BasicArgs a) {
    const int lane = threadIdx.x & 31;
    const int H = a.H, W = a.W;
    const size_t plane = (size_t)H * W;
    const float conf_max = a.op.conf_max, alpha = a.op.alpha, kb = a.op.kb, kc = a.op.kc;
    const float gsy = RS ? bscale(a.gt_h, H) : 1.f, gsx = RS ? bscale(a.gt_w, W) : 1.f;

    BandItem it;
    while (next_band_item(a.bq, a.B, H, lane, it)) {
        const int b = it.b, view = it.view, ra = it.ra, rb = it.rb;
        const int x0 = it.strip * 128 + 4 * lane;

        float sum = 0.f;
        if (x0 < W) {                                  // W % 4 == 0: a lane's 4 pixels are all inside or all outside
            const float* __restrict__ pred = a.op.pred[view] + (size_t)b * plane * 3;
            const float* __restrict__ gt = a.op.gt[view] + (size_t)b * (RS ? (size_t)a.gt_h * a.gt_w : plane) * 3;
            BTap gtx[4];
            if (RS) {
#pragma unroll
                for (int e = 0; e < 4; ++e) gtx[e] = btap(x0 + e, a.gt_w, gsx);
            }
            const float* __restrict__ conf = a.op.conf[view] ? a.op.conf[view] + (size_t)b * plane : nullptr;
            float* __restrict__ dpred = BWD ? a.op.dpred[view] + (size_t)b * plane * 3 : nullptr;
            float* __restrict__ dconf = (BWD && a.op.dconf[view]) ? a.op.dconf[view] + (size_t)b * plane : nullptr;
            auto load = [&](int y, float p[12], float g[12], float c[4]) {
                const size_t pix = (size_t)y * W + x0;
                const float4 p0 = ldg_stream_f4(pred + pix * 3), p1 = ldg_stream_f4(pred + pix * 3 + 4),
                             p2 = ldg_stream_f4(pred + pix * 3 + 8);
                p[0] = p0.x; p[1] = p0.y; p[2] = p0.z; p[3] = p0.w; p[4] = p1.x; p[5] = p1.y;
                p[6] = p1.z; p[7] = p1.w; p[8] = p2.x; p[9] = p2.y; p[10] = p2.z; p[11] = p2.w;
                if (!RS) {
                    const float4 g0 = ldg_stream_f4(gt + pix * 3), g1 = ldg_stream_f4(gt + pix * 3 + 4),
                                 g2 = ldg_stream_f4(gt + pix * 3 + 8);
                    g[0] = g0.x; g[1] = g0.y; g[2] = g0.z; g[3] = g0.w; g[4] = g1.x; g[5] = g1.y;
                    g[6] = g1.z; g[7] = g1.w; g[8] = g2.x; g[9] = g2.y; g[10] = g2.z; g[11] = g2.w;
                } else {                               // bilinear taps (every tap is read, zero weights included)
                    const BTap gty = btap(y, a.gt_h, gsy);
#pragma unroll
                    for (int e = 0; e < 4; ++e)
#pragma unroll
                        for (int ch = 0; ch < 3; ++ch) g[3 * e + ch] = bsample(gt, a.gt_w, 3, ch, gty, gtx[e]);
                }
                if (!conf) { c[0] = c[1] = c[2] = c[3] = 1.f; }
                else {
                    const float4 cc = ldg_stream_f4(conf + pix);
                    c[0] = cc.x; c[1] = cc.y; c[2] = cc.z; c[3] = cc.w;
                }
            };
            auto eval = [&](int y, const float p[12], const float g[12], const float c[4]) {
                float gq[12], dc[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const BasicGrad bg = basic_px<BWD>(p[3 * e], p[3 * e + 1], p[3 * e + 2], g[3 * e], g[3 * e + 1],
                                                       g[3 * e + 2], c[e], conf_max, alpha, kb, kc, sum);
                    gq[3 * e] = bg.gx; gq[3 * e + 1] = bg.gy; gq[3 * e + 2] = bg.gz; dc[e] = bg.dc;
                }
                if (BWD) {
                    const size_t pix = (size_t)y * W + x0;
                    float* o = dpred + pix * 3;
                    stg_stream_f4(o, make_float4(gq[0], gq[1], gq[2], gq[3]));
                    stg_stream_f4(o + 4, make_float4(gq[4], gq[5], gq[6], gq[7]));
                    stg_stream_f4(o + 8, make_float4(gq[8], gq[9], gq[10], gq[11]));
                    if (dconf) stg_stream_f4(dconf + pix, make_float4(dc[0], dc[1], dc[2], dc[3]));
                }
            };
            for (int y = ra; y < rb; ++y) {
                float p[12], g[12], c[4];
                load(y, p, g, c);
                eval(y, p, g, c);
            }
        }
        sum = warp_sum(sum);
        if (lane == 0) {
            float4* o = reinterpret_cast<float4*>(a.partials + (size_t)it.pidx * kNTerms);
            o[0] = make_float4(sum, 0.f, 0.f, 0.f);
            o[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
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
    int loss_partials_n;               // partial vectors per image-view the loss_partials hold
};

WsLayout ws_layout(int B, int H, int W, int multi) {
    WsLayout L;
    L.stiles_x = (W + kSTW - 1) / kSTW; L.stiles_y = (H + kSTH - 1) / kSTH;
    L.tiles_x = (W + kTW - 1) / kTW;    L.tiles_y = (H + kTH - 1) / kTH;
    size_t off = 0;
    L.counter = off;        off += 256;
    L.sm_bands = (H + kStatsMarchRows - 1) / kStatsMarchRows; L.sm_strips = (W + 127) / 128;
    const size_t stats_tiles = (size_t)max(L.stiles_x * L.stiles_y, L.sm_bands * L.sm_strips);
    L.stats_partials = off; off += t3d_align_up((size_t)B * 2 * stats_tiles * 4 * sizeof(float), 256);
    // sized for the tile kernel (16-row tiles) and the persistent kernels (>= 8-row bands; loss_impl checks the plan)
    L.loss_partials_n = L.tiles_x * ((H + 7) / 8);
    L.loss_partials = off;  off += t3d_align_up((size_t)B * 2 * L.loss_partials_n * kNTerms * sizeof(float), 256);
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
    constexpr size_t smem = loss_smem_bytes<MULTI>();
    if (int rc = t3d_set_max_dynamic_smem<loss_tile_kernel<MULTI, VEC, BWD>>((int)smem)) return rc;
    const int grid = la.B * 2 * la.tiles_x * la.tiles_y;
    T3D_LAUNCH("loss_tile_kernel", st, loss_tile_kernel<MULTI, VEC, BWD><<<grid, kThreads, smem, st>>>(la));
    return T3D_OK;
}

// The persistent kernels' work items (BandQueue): nbands_l bands of rows_l rows from the top, then the last
// ~1/tail_div of the image in bands of rows_s rows (queued behind all the large ones: a shorter tail of the persistent
// grid).  An image too short for a tail has its ragged last large band handled as one small band of rows_l rows.
BandQueue plan_bands(int H, int W, int rows_l, int rows_s, int tail_div, unsigned int* queue) {
    BandQueue bq;
    bq.queue = queue;
    const int small_rows = ((H / tail_div + rows_s - 1) / rows_s) * rows_s;
    bq.rows_l = rows_l; bq.rows_s = rows_s;
    bq.nbands_l = (small_rows > 0) ? max(0, H - small_rows) / rows_l : (H + rows_l - 1) / rows_l;
    if (small_rows == 0) { bq.nbands_s = 0;
        if (bq.nbands_l * rows_l > H) { bq.nbands_l -= 1; bq.rows_s = rows_l; bq.nbands_s = 1; } }
    else bq.nbands_s = (H - bq.nbands_l * rows_l + rows_s - 1) / rows_s;
    bq.nstrips = (W + 127) / 128;
    return bq;
}

// loss_basic_kernel: 32-row bands, the last ~1/8 of the image in 8-row bands
constexpr int kBasicRows = 32, kBasicTailRows = 8, kBasicTailDiv = 8;
// loss_march_kernel: bands of 32 rows (a band re-reads the row above and the row below it: taller = less overfetch),
// the last ~1/8 of the image in 8-row bands; other band heights and tails: DESIGN §4 experiment 12 and §5.
// loss_march_ms_kernel: a band brings 4 halo rows instead of 2 and must start on an even row: 16-row tail bands.
constexpr int kMarchRows = 32, kMarchTailRows = 8, kMarchMsTailRows = 16, kMarchTailDiv = 8;

template <bool BWD, bool RS>
int launch_basic(const BasicArgs& ba, cudaStream_t st) {
    const int items = ba.B * 2 * ba.bq.per_image_view();
    const int grid = min(t3d_sm_count() * basic_blocks_per_sm<BWD, RS>(), (items + kBWarps - 1) / kBWarps);
    T3D_LAUNCH("loss_basic_kernel", st, loss_basic_kernel<BWD, RS><<<grid, kBWarps * 32, 0, st>>>(ba));
    return T3D_OK;
}

// The kernels that compute the loss; choose_loss_path picks one per call.
enum class LossPath {
    kBasic,         // loss_basic_kernel: no thermal images
    kBasicTaps,     // loss_basic_kernel<RS>: the same with a downsampled GT read through bilinear taps
    kMarch,         // loss_march_kernel: thermal-aware, single scale
    kMarchTaps,     // loss_march_rs_kernel: the same with a downsampled GT resampled as its rows are staged
    kMarchMs,       // loss_march_ms_kernel: multi-scale, both scales in one pass
    kScale2March,   // loss_scale2_kernel, then loss_march_kernel adding its gradient: multi-scale in two passes
    kTile,          // loss_tile_kernel: every other call
};
struct LossPathChoice { LossPath path; int span; };   // span: a strip's widest GT source segment (the *Taps paths)

// gt_h == 0 / conf_h == 0: the GT / confidence is at the prediction's size.  vec: W % 4 == 0 and every array the
// kernels stream is 16-byte aligned (a GT read through taps excepted).  gt_vec: gt_w % 4 == 0 and a 16-byte aligned GT.
// one_plane: a thermal row stages one plane (one channel, or three bit-identical replicas).  ms: multi-scale with
// thermal images.
LossPathChoice choose_loss_path(int H, int W, int gt_h, int gt_w, int conf_h, bool vec, bool gt_vec, bool thermal_on,
                                bool one_plane, bool ms, bool conf_min_only) {
    const LossPathChoice tile = {LossPath::kTile, 0};
    // The persistent kernels stream 4 pixels per lane with 128-bit loads or bulk copies, and read the confidence at
    // the prediction's size only: unaligned arrays, W % 4 != 0 and a GT-sized confidence take the tile kernel.
    if (!vec || conf_h != 0) return tile;
    // A downsampled GT is read through bilinear taps by the persistent kernels only while a strip's source segment is
    // at most 144 px (gt_w ~ W, t3d_loss_march_rs_fits).  Measured on a B200 at 1000 W against the tile kernel's fused
    // taps: 384x512 <- 512x512 at batch 64, 364 us against 696 us thermal-aware (loss_march_rs_kernel) and 321.5 us
    // against 341.1 us without thermal images (loss_basic_kernel, tools/plain_loss_time.py); 224x224 <- 512x512 at
    // batch 8, 92 us against 77 us and 88.1 us against 41.0 us.  Wider segments and an upsampled GT keep the tile
    // kernel (DESIGN §4).
    int span = 0;
    if (gt_h != 0) {
        if (gt_h < H || gt_w < W) return tile;
        span = t3d_loss_march_rs_span(W, gt_w);
        if (!t3d_loss_march_rs_fits(span)) return tile;
    }
    if (!thermal_on) return {gt_h != 0 ? LossPath::kBasicTaps : LossPath::kBasic, span};
    // the marching kernels clamp the confidence to [kConfMin, kConfMax]: the lower clamp alone takes the tile kernel
    if (conf_min_only) return tile;
    // the marching kernel bulk-copies the GT source rows; the one-pass multi-scale kernel has no registers left for
    // the taps (DESIGN §8)
    if (gt_h != 0) return (gt_vec && !ms) ? LossPathChoice{LossPath::kMarchTaps, span} : tile;
    if (!ms) return {LossPath::kMarch, 0};
    if (H < 4 || W < 4) return tile;     // the marching multi-scale paths need at least 2 x 2 pooled cells
    // One staged thermal plane: both scales in one pass over the rows.  Three distinct planes would leave no shared
    // memory for that kernel's deeper ring: the half-resolution terms run first as their own pass (DESIGN §4).
    return {one_plane ? LossPath::kMarchMs : LossPath::kScale2March, 0};
}

int loss_impl(bool bwd, const float* pred1, const float* pred2, const float* gt1, const float* gt2,
              const float* conf1, const float* conf2, const float* thermal1, const float* thermal2,
              int tch, const float* ustats1, const float* ustats2, int ustats_tiles, float* dpred1, float* dpred2, float* dconf1, float* dconf2,
              int B, int H, int W, int flags, float alpha, float ew, float sw, float dw, float gscale,
              float* out_sample, float* out_batch, double* out_f64, cudaEvent_t main_done,
              void* workspace, size_t ws_bytes, void* stream, int gt_h, int gt_w, int conf_h, int conf_w) {
    // ---- validate and normalise
    if (int rc = check_dims(B, H, W)) return rc;
    T3D_REQUIRE((flags & ~(T3D_LOSS_MULTI_SCALE | T3D_LOSS_CONF_MIN_ONLY | T3D_LOSS_STATS_TWO_SCALES)) == 0, "unknown loss flags 0x%x", flags);
    if (gt_h == H && gt_w == W) gt_h = gt_w = 0;                    // same size: direct reads
    if (conf_h == H && conf_w == W) conf_h = conf_w = 0;
    T3D_REQUIRE((gt_h == 0) == (gt_w == 0) && gt_h >= 0 && (conf_h == 0) == (conf_w == 0) && conf_h >= 0, "bad gt / conf size");
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
    const bool ms = multi && thermal_on;
    const bool vec = (W % 4 == 0) && t3d_aligned16(pred1) && t3d_aligned16(pred2) && (gt_h != 0 || (t3d_aligned16(gt1) &&
                     t3d_aligned16(gt2))) && (conf_h != 0 || (t3d_aligned16(conf1) && t3d_aligned16(conf2))) &&
                     t3d_aligned16(thermal1) && t3d_aligned16(thermal2) && t3d_aligned16(dpred1) &&
                     t3d_aligned16(dpred2) && t3d_aligned16(dconf1) && t3d_aligned16(dconf2);
    const bool gt_vec = gt_w % 4 == 0 && t3d_aligned16(gt1) && t3d_aligned16(gt2);

    // ---- choose the kernel; the persistent ones get their work items
    const LossPathChoice choice = choose_loss_path(H, W, gt_h, gt_w, conf_h, vec, gt_vec, thermal_on, tch == 1 || replicated,
                                                   ms, conf_min_only);
    const LossPath path = choice.path;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char* ws = reinterpret_cast<char*>(workspace);
    float* stats_partials = reinterpret_cast<float*>(ws + L.stats_partials);
    float* loss_partials = reinterpret_cast<float*>(ws + L.loss_partials);
    unsigned int* counter = reinterpret_cast<unsigned int*>(ws + L.counter);
    BandQueue bq = {};
    int n_partials = L.tiles_x * L.tiles_y;                          // loss_tile_kernel: one per 16 x 128 tile
    if (path == LossPath::kBasic || path == LossPath::kBasicTaps) {
        bq = plan_bands(H, W, kBasicRows, kBasicTailRows, kBasicTailDiv, counter + 1);
        n_partials = bq.per_image_view();
    } else if (path != LossPath::kTile) {
        bq = plan_bands(H, W, kMarchRows, path == LossPath::kMarchMs ? kMarchMsTailRows : kMarchTailRows, kMarchTailDiv, counter + 1);
        n_partials = bq.per_image_view();
    }
    T3D_REQUIRE(n_partials <= L.loss_partials_n, "%d partial vectors per image-view do not fit the %d of the workspace",
                n_partials, L.loss_partials_n);

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

    LossOperands op;
    op.pred[0] = pred1; op.pred[1] = pred2; op.gt[0] = gt1; op.gt[1] = gt2; op.conf[0] = conf1; op.conf[1] = conf2;
    op.dpred[0] = dpred1; op.dpred[1] = dpred2; op.dconf[0] = dconf1; op.dconf[1] = dconf2;
    op.alpha = alpha;
    const double N = (double)H * W, n2 = (double)(H / 2) * (W / 2);
    op.kb = (float)((double)gscale / (3.0 * N));
    op.kc = (float)((double)gscale / N);
    op.conf_max = conf_min_only ? __int_as_float_host(0x7f800000u) : kConfMax;
    const double l2 = (n2 > 0) ? (double)kScale2Weight / n2 : 0.0;
    const float kE[2] = {(float)((double)gscale * ew / N), (float)((double)gscale * ew * l2)};
    const float kS[2] = {(float)((double)gscale * sw / N), (float)((double)gscale * sw * l2)};
    const float kD[2] = {(float)((double)gscale * dw / N), (float)((double)gscale * dw * l2)};

    // ---- fill the chosen kernel's arguments and launch it
    int rc = T3D_OK;
    const float* partials2 = nullptr;
    int tiles2 = 0;
    switch (path) {
    case LossPath::kBasic:
    case LossPath::kBasicTaps: {
        BasicArgs ba;
        ba.op = op; ba.partials = loss_partials; ba.bq = bq;
        ba.B = B; ba.H = H; ba.W = W; ba.gt_h = gt_h; ba.gt_w = gt_w;
        if (path == LossPath::kBasicTaps) rc = bwd ? launch_basic<true, true>(ba, st) : launch_basic<false, true>(ba, st);
        else rc = bwd ? launch_basic<true, false>(ba, st) : launch_basic<false, false>(ba, st);
        break;
    }
    case LossPath::kMarch:
    case LossPath::kMarchTaps:
    case LossPath::kMarchMs:
    case LossPath::kScale2March: {
        // TMA-fed warp-marching kernels (t3d_loss_march.cu)
        MarchArgs ma;
        ma.op = op;
        for (int v = 0; v < 2; ++v) { ma.thermal[v] = v ? thermal2 : thermal1; ma.stats[v] = stats_v[v]; ma.dzp[v] = nullptr; }
        ma.partials = loss_partials; ma.bq = bq;
        ma.B = B; ma.H = H; ma.W = W; ma.tch = tch; ma.stiles = stiles; ma.replicated = replicated;
        ma.kE = kE[0]; ma.kS = kS[0]; ma.kD = kD[0]; ma.kE2 = kE[1]; ma.kS2 = kS[1]; ma.kD2 = kD[1];
        ma.gt_h = gt_h; ma.gt_w = gt_w;
        if (path == LossPath::kScale2March) {   // the half-resolution pass hands its gradient to the marching kernel
            Scale2Args sa;
            float* dzp = reinterpret_cast<float*>(ws + L.s2_dzp);
            for (int v = 0; v < 2; ++v) {
                sa.pred[v] = op.pred[v]; sa.gt[v] = op.gt[v]; sa.thermal[v] = ma.thermal[v]; sa.stats[v] = stats_v[v];
                sa.dzp[v] = dzp + (size_t)v * B * (H >> 1) * (W >> 1);
                if (bwd) ma.dzp[v] = sa.dzp[v];
            }
            sa.partials = reinterpret_cast<float*>(ws + L.s2_partials);
            sa.B = B; sa.H = H; sa.W = W; sa.tch = tch; sa.replicated = replicated; sa.stiles = stiles;
            sa.tiles_x = L.s2_tiles_x; sa.tiles_y = L.s2_tiles_y;
            sa.kE = kE[1]; sa.kS = kS[1]; sa.kD = kD[1];
            if (int rc2 = t3d_launch_loss_scale2(sa, bwd, st)) return rc2;
            partials2 = sa.partials; tiles2 = sa.tiles_x * sa.tiles_y;
        }
        rc = path == LossPath::kMarchTaps ? t3d_launch_loss_march_rs(ma, choice.span, bwd, st)
           : path == LossPath::kMarchMs ? t3d_launch_loss_march_ms(ma, bwd, st) : t3d_launch_loss_march(ma, bwd, st);
        break;
    }
    case LossPath::kTile: {
        LossArgs la;
        la.op = op;
        la.thermal[0] = thermal_on ? thermal1 : nullptr; la.thermal[1] = thermal_on ? thermal2 : nullptr;
        la.stats[0] = stats_v[0]; la.stats[1] = stats_v[1]; la.partials = loss_partials;
        la.B = B; la.H = H; la.W = W; la.tch = thermal_on ? tch : 0;
        la.tiles_x = L.tiles_x; la.tiles_y = L.tiles_y; la.stiles = stiles;
        for (int s = 0; s < 2; ++s) { la.kE[s] = kE[s]; la.kS[s] = kS[s]; la.kD[s] = kD[s]; }
        la.gt_h = gt_h; la.gt_w = gt_w; la.conf_h = conf_h; la.conf_w = conf_w;
        if (bwd) {
            if (ms) rc = vec ? launch_loss<true, true, true>(la, st) : launch_loss<true, false, true>(la, st);
            else    rc = vec ? launch_loss<false, true, true>(la, st) : launch_loss<false, false, true>(la, st);
        } else {
            if (ms) rc = vec ? launch_loss<true, true, false>(la, st) : launch_loss<true, false, false>(la, st);
            else    rc = vec ? launch_loss<false, true, false>(la, st) : launch_loss<false, false, false>(la, st);
        }
        break;
    }
    }
    if (rc) return rc;
    if (main_done) T3D_CUDA(cudaEventRecord(main_done, st));   // lets a caller overlap the second stage with other work

    // ---- second stage
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

size_t t3d_loss_workspace_bytes(int B, int H, int W, int flags) {
    if (B < 1 || H < 1 || W < 1) return 0;
    return ws_layout(B, H, W, (flags & T3D_LOSS_MULTI_SCALE) ? 1 : 0).total;
}

int t3d_loss_fwd_bwd(const float* pred1, const float* pred2, const float* gt1, const float* gt2, int gt_h, int gt_w,
                     const float* conf1, const float* conf2, int conf_h, int conf_w,
                     const float* thermal1, const float* thermal2, int thermal_channels,
                     const float* thermal_stats1, const float* thermal_stats2, int stats_tiles,
                     float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                     int B, int H, int W, int flags,
                     float alpha, float edge_weight, float smoothness_weight, float detail_weight,
                     float grad_scale, float* out_sample, float* out_batch, double* out_sample_f64,
                     void* main_done_event, void* workspace, size_t workspace_bytes, void* stream) {
    T3D_REQUIRE((dpred1 == nullptr) == (dpred2 == nullptr), "dpred1 / dpred2: both or neither may be NULL");
    const bool bwd = dpred1 != nullptr;
    if (!bwd) { dconf1 = dconf2 = nullptr; grad_scale = 1.0f; }          // forward only: no gradient writes
    if (!conf1 && !conf2) { conf_h = H; conf_w = W; }                   // ones
    T3D_REQUIRE(gt_h >= 1 && gt_w >= 1, "bad gt size");
    T3D_REQUIRE(conf_h >= 1 && conf_w >= 1, "bad conf size");
    T3D_REQUIRE(!(dconf1 || dconf2) || (conf_h == H && conf_w == W), "a confidence that takes a gradient has the prediction's size");
    return loss_impl(bwd, pred1, pred2, gt1, gt2, conf1, conf2, thermal1, thermal2, thermal_channels,
                     thermal_stats1, thermal_stats2, stats_tiles, dpred1, dpred2, dconf1, dconf2, B, H, W, flags, alpha,
                     edge_weight, smoothness_weight, detail_weight, grad_scale, out_sample, out_batch, out_sample_f64,
                     reinterpret_cast<cudaEvent_t>(main_done_event), workspace, workspace_bytes, stream,
                     gt_h, gt_w, conf_h, conf_w);
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
