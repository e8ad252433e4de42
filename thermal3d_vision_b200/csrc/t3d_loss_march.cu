// t3d_loss_march.cu -- fast path of the fused thermal-aware loss (single scale,
// 16-byte aligned, W % 4 == 0): warp-marching stencil fed by the TMA engine.
//
// Same math as loss_tile_kernel in t3d_loss.cu (utils/loss.py:75-98,100-305 and
// its closed-form backward, SURVEY.md Appendix A); different machine mapping:
//
//  * a work item is (image-view, 128-pixel strip, band of R rows); warps pull items
//    from a global queue (persistent grid, one CTA per SM, no inter-warp sync);
//  * the warp's lane 0 streams the strip's rows global -> shared with
//    cp.async.bulk (1-D TMA: pred / gt AoS segments, confidence, thermal planes)
//    into a warp-private NS-stage ring; completion is an mbarrier transaction
//    count, so loads in flight cost no registers and the LSU sees no 48-byte
//    strided AoS pattern;
//  * each lane owns 4 consecutive pixels and marches down the rows: vertical
//    neighbours live in registers (the row below is read once and becomes the
//    current row), horizontal neighbours come from warp shuffles, the one pixel
//    left/right of the strip from the 4-pixel halo the bulk copy brought along;
//  * every forward-difference term q is evaluated exactly once per pixel
//    (q_y of the row above is carried, q_x of the left neighbour is shuffled),
//    gradients are gathered (no atomics) and written once with 128-bit stores.
#include "t3d_loss_internal.cuh"
#include <type_traits>

namespace {

constexpr float kEps = 1e-5f;
constexpr float kHuber = 0.1f;
constexpr float kConfMin = 1e-5f, kConfMax = 10.0f;

constexpr int kStripPx = 128;            // 32 lanes x 4 pixels
constexpr int kSegPx = kStripPx + 8;     // + 4-pixel halo each side (keeps 16-byte alignment of AoS rows)

// SEG > 0 (loss_march_rs_kernel): the gt is not staged at the prediction's size; instead the two source rows of the
// row's bilinear y-tap, SEG pixels each (the strip's x-taps, 16-byte aligned segment), from which the lanes resample
template <int TCH, bool S2 = false, int SEG = 0> struct Stage {
    static constexpr int kPred = 0;
    static constexpr int kGt = kSegPx * 3;
    static constexpr int kConf = (SEG ? 1 : 2) * kSegPx * 3;
    static constexpr int kTh = kConf + kStripPx;
    static constexpr int kDz = kTh + TCH * kSegPx;         // multi-scale: the strip's 64 pooled-cell gradients of this row pair
    static constexpr int kSrc = kDz + (S2 ? kStripPx / 2 : 0);
    static constexpr int kFloats = kSrc + 2 * SEG * 3;     // 1352 floats (TCH = 3, single scale, SEG = 0)
};

// ------------------------------------------------------------------ PTX helpers (sm_100a)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine, SASS UBLKCP); completes `bytes` on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------ math
struct Sums { float E, S, D; };

// NaN-propagating min / max (SASS FMNMX.NAN): torch.clamp lets NaN through, fminf/fmaxf would not
__device__ __forceinline__ float min_nan(float a, float b) { float d; asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }
__device__ __forceinline__ float max_nan(float a, float b) { float d; asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }

// sgn(x) * |t-signed value|: (x > 0) ? t : (x < 0 ? -t : 0) with one compare (sgn(0) = 0 like ATen)
__device__ __forceinline__ float times_sgn(float t, float x) {
    const float r = __uint_as_float(__float_as_uint(t) ^ (__float_as_uint(x) & 0x80000000u));
    return (x != 0.f) ? r : 0.f;
}

// one forward-difference term (SURVEY.md Appendix A).  The zero-padded last column / row is expressed
// by the caller handing in zb == za, gb == ga (all contributions vanish, sgn(0) = 0).
__device__ __forceinline__ float q_term(float za, float zb, float ga, float gb, float w, float omw,
                                        float kE_omw, float kS2w, float kD, Sums& acc) {
    const float s = zb - za;
    const float a = fabsf(s);
    const float b = fabsf(gb - ga);
    const float e = a - b;
    const float d = fabsf(e);
    const float c = fminf(d, kHuber);                                     // huber(d) = c^2/2 + delta (d - c)
    acc.E = fmaf(a, omw, acc.E);
    acc.S = fmaf(a * a, w, acc.S);
    acc.D += fmaf(0.5f * c, c, kHuber * (d - c));
    const float dh = fminf(fmaxf(e, -kHuber), kHuber);                    // rho'(d) sgn(e)
    const float t = fmaf(kD, dh, fmaf(kS2w, a, kE_omw));
    return times_sgn(t, s);
}

__device__ __forceinline__ float edge_w(float tx, float ty, float inv_mx, float inv_my, float m) {
    // exp(-8 clamp(tx/mean,0,m)) * exp(-8 clamp(ty/mean,0,m))  (utils/loss.py:240-256); tx, ty >= 0
    const float cx = min_nan(tx * inv_mx, m);
    const float cy = min_nan(ty * inv_my, m);
    return __expf(-8.0f * (cx + cy));
}

// REP: the image's 3 planes are bit-identical replicas (what enhance_thermal_contrast always returns,
// utils/preprocessing.py:22-28): only plane 0 is staged and gray = gray3(v, v, v) -- the same bits as
// reading the three planes, a third of the thermal traffic.
template <int TCH, bool REP>
__device__ __forceinline__ void gray_quad(const float* __restrict__ th, int idx, float g[4]) {
    const float4 c0 = *reinterpret_cast<const float4*>(th + idx);
    if (REP) {
        g[0] = gray3(c0.x, c0.x, c0.x); g[1] = gray3(c0.y, c0.y, c0.y);
        g[2] = gray3(c0.z, c0.z, c0.z); g[3] = gray3(c0.w, c0.w, c0.w);
    } else if (TCH == 3) {
        const float4 c1 = *reinterpret_cast<const float4*>(th + kSegPx + idx);
        const float4 c2 = *reinterpret_cast<const float4*>(th + 2 * kSegPx + idx);
        g[0] = gray3(c0.x, c1.x, c2.x); g[1] = gray3(c0.y, c1.y, c2.y);
        g[2] = gray3(c0.z, c1.z, c2.z); g[3] = gray3(c0.w, c1.w, c2.w);
    } else {
        g[0] = c0.x; g[1] = c0.y; g[2] = c0.z; g[3] = c0.w;
    }
}
template <int TCH, bool REP>
__device__ __forceinline__ float gray_px(const float* __restrict__ th, int idx) {
    if (REP) { const float v = th[idx]; return gray3(v, v, v); }
    return (TCH == 3) ? gray3(th[idx], th[kSegPx + idx], th[2 * kSegPx + idx]) : th[idx];
}

struct RowRegs { float P[12], G[12], g[4]; };    // pred xyz, gt xyz (AoS order), gray of one lane's 4 pixels

template <int TCH, bool REP>
__device__ __forceinline__ void load_row(const float* __restrict__ st, int idx, RowRegs& r) {
    const float4* p = reinterpret_cast<const float4*>(st + Stage<TCH>::kPred + idx * 3);
    const float4* q = reinterpret_cast<const float4*>(st + Stage<TCH>::kGt + idx * 3);
    const float4 a = p[0], b = p[1], c = p[2], d = q[0], e = q[1], f = q[2];
    r.P[0] = a.x; r.P[1] = a.y; r.P[2] = a.z; r.P[3] = a.w; r.P[4] = b.x; r.P[5] = b.y; r.P[6] = b.z; r.P[7] = b.w;
    r.P[8] = c.x; r.P[9] = c.y; r.P[10] = c.z; r.P[11] = c.w;
    r.G[0] = d.x; r.G[1] = d.y; r.G[2] = d.z; r.G[3] = d.w; r.G[4] = e.x; r.G[5] = e.y; r.G[6] = e.z; r.G[7] = e.w;
    r.G[8] = f.x; r.G[9] = f.y; r.G[10] = f.z; r.G[11] = f.w;
    gray_quad<TCH, REP>(st + Stage<TCH>::kTh, idx, r.g);       // (offsets up to kTh do not depend on S2)
}

// Resampled gt (SEG > 0): the source rows staged at `src` (row i0, then row i1 at src + 3 SEG) start at source column
// s0; output column x of the row whose y-tap is ty.
struct RsCtx { int s0, gw; float sx; };
template <int SEG>
__device__ __forceinline__ float gt_rs(const float* __restrict__ src, int x, int ch, const RsCtx& rs, const BTap& ty) {
    const BTap tx = btap(x, rs.gw, rs.sx);
    const float* p0 = src + (tx.i0 - rs.s0) * 3 + ch;
    const float* p1 = src + (tx.i1 - rs.s0) * 3 + ch;
    return blerp(p0[0], p1[0], p0[SEG * 3], p1[SEG * 3], ty, tx);
}
// load_row with the gt resampled: columns x0 .. x0+3 (clamped to the image: lanes past its right edge compute garbage
// that is never used, but stay inside the staged segment)
template <int TCH, bool REP, int SEG>
__device__ __forceinline__ void load_row_rs(const float* __restrict__ st, int idx, int x0, int xmax, const RsCtx& rs,
                                            const BTap& ty, RowRegs& r) {
    using St = Stage<TCH, false, SEG>;
    const float4* p = reinterpret_cast<const float4*>(st + St::kPred + idx * 3);
    const float4 a = p[0], b = p[1], c = p[2];
    r.P[0] = a.x; r.P[1] = a.y; r.P[2] = a.z; r.P[3] = a.w; r.P[4] = b.x; r.P[5] = b.y; r.P[6] = b.z; r.P[7] = b.w;
    r.P[8] = c.x; r.P[9] = c.y; r.P[10] = c.z; r.P[11] = c.w;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int x = min(x0 + e, xmax);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) r.G[3 * e + ch] = gt_rs<SEG>(st + St::kSrc, x, ch, rs, ty);
    }
    gray_quad<TCH, REP>(st + St::kTh, idx, r.g);
}

// ------------------------------------------------------------------ kernel
// S2: multi-scale -- the scale-2 pass (t3d_loss_scale2.cu) left 0.25 * d(loss)/d(pooled z) per 2x2 cell in a.dzp
// SEG > 0: the gt is [B, gt_h, gt_w, 3] and is bilinearly resampled to H x W as its rows are loaded from the ring
// (loss_march_rs_kernel); everything downstream of the gt values is the same code
template <int TCH, bool REP, bool BWD, bool S2, int SEG, int NS, int WARPS>
__device__ __forceinline__ void march_body(const MarchArgs& a) {
    static_assert(!REP || TCH == 1, "replicated planes: one plane is staged");
    static_assert(!(S2 && SEG), "multi-scale with a resampled gt runs on the tile kernel");
    using St = Stage<TCH, S2, SEG>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    float* ring = reinterpret_cast<float*>(smem_raw) + (size_t)wrp * NS * St::kFloats;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)WARPS * NS * St::kFloats * sizeof(float)) + wrp * NS;

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();

    const int H = a.H, W = a.W;
    const size_t plane = (size_t)H * W;
    const int nbands = a.nbands_l + a.nbands_s;
    const int n_large = a.B * 2 * a.nbands_l * a.nstrips;
    const int ntasks = a.B * 2 * nbands * a.nstrips;
    const float kE = a.kE, kS2 = 2.0f * a.kS, kD = a.kD, kb = a.kb, kc = a.kc, alpha = a.alpha;
    const float alpha_ln2 = alpha * 0.69314718055994531f;
    uint32_t pos = 0;                                  // rows streamed so far by this warp (ring position)
    const int gh = SEG ? a.gt_h : H, gw = SEG ? a.gt_w : W;
    const float sy = SEG ? bscale(gh, H) : 1.f, sx = SEG ? bscale(gw, W) : 1.f;

    for (;;) {
        int task = 0;
        if (lane == 0) task = (int)atomicAdd(a.queue, 1u);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= ntasks) break;
        const bool large = task < n_large;
        const int t1 = large ? task : task - n_large;
        const int nb = large ? a.nbands_l : a.nbands_s;
        const int s = t1 % a.nstrips;
        const int t2 = t1 / a.nstrips;
        const int k = t2 % nb;
        const int img = t2 / nb;
        const int b = img >> 1, view = img & 1;
        const int ra = large ? k * a.rows_l : a.nbands_l * a.rows_l + k * a.rows_s;
        const int rb = large ? ra + a.rows_l : min(ra + a.rows_s, H);          // the large bands end at nbands_l * rows_l <= H
        const int pidx = (img * nbands + (large ? k : a.nbands_l + k)) * a.nstrips + s;     // partials: per image-view, band-major
        const int i_lo = max(ra - 1, 0), i_hi = min(rb, H - 1);
        const int n_rows = i_hi - i_lo + 1;
        const int col0 = s * kStripPx;
        const int c0 = max(col0 - 4, 0), c1 = min(col0 + kStripPx + 4, W);
        const int npx = c1 - c0, off = col0 - c0;
        const int own_n = min(kStripPx, W - col0);
        const int j = col0 + 4 * lane;
        const bool active = 4 * lane < own_n;
        const bool last_lane = active && (4 * lane + 4 >= own_n);
        const bool right_in_image = (j + 4 < W);
        const int idx = 4 * lane + off;                // smem pixel index of this lane's quad

        const float* __restrict__ pred = a.pred[view] + (size_t)b * plane * 3;
        const float* __restrict__ gt = a.gt[view] + (size_t)b * (size_t)gh * gw * 3;
        const float* __restrict__ conf = a.conf[view] ? a.conf[view] + (size_t)b * plane : nullptr;
        const float* __restrict__ th = a.thermal[view] + (size_t)b * (REP ? 3 : TCH) * plane;
        // resampled gt: the strip's source segment [s0, s0 + seg_px) covers the x-taps of columns c0 .. c1-1
        RsCtx rs = {0, gw, sx};
        uint32_t seg_bytes = 0;
        if (SEG) {
            rs.s0 = btap(c0, gw, sx).i0 & ~3;
            seg_bytes = (uint32_t)(((btap(c1 - 1, gw, sx).i1 + 4) & ~3) - rs.s0) * 12u;
        }
        // running output pointers of this lane's quad (row i_lo; advanced by one row per iteration)
        float* dp_ptr = BWD ? a.dpred[view] + ((size_t)b * plane + (size_t)i_lo * W + j) * 3 : nullptr;
        float* dc_ptr = (BWD && a.dconf[view]) ? a.dconf[view] + (size_t)b * plane + (size_t)i_lo * W + j : nullptr;
        // multi-scale: this lane's two pooled cells per row pair (W % 4 == 0: columns j .. j+3 are always inside 2 * (W / 2))
        const int w2 = W >> 1, rows2 = 2 * (H >> 1);
        const float* dz2_ptr = (S2 && BWD) ? a.dzp[view] + (size_t)b * (H >> 1) * w2 + (j >> 1) : nullptr;
        // W % 8 == 0: a pooled row segment is 16-byte aligned and a multiple of 16 bytes -> it travels with the
        // row's other segments through the bulk-copy ring; else each lane loads its two cells itself
        const bool dz_staged = S2 && BWD && ((W & 7) == 0);
        const float* dz2_strip = dz_staged ? a.dzp[view] + (size_t)b * (H >> 1) * w2 + (col0 >> 1) : nullptr;

        // 1 / (mean + eps) of |Dx gray|, |Dy gray| of this image: fixed-order sum of the stats partials
        float inv_mx, inv_my;
        {
            float sx = 0.f, sy = 0.f;
            const float* sp = a.stats[view] + (size_t)b * a.stiles * 4;
            for (int t = lane; t < a.stiles; t += 32) { sx += sp[t * 4]; sy += sp[t * 4 + 1]; }
            sx = warp_sum(sx); sy = warp_sum(sy);
            const float invN = 1.0f / (float)plane;
            inv_mx = 1.0f / (sx * invN + kEps);
            inv_my = 1.0f / (sy * invN + kEps);
        }
        // NaN / Inf thermal pixels make the reference loss NaN (clamp(NaN) = NaN): poison the task's sums
        const bool thermal_bad = !(inv_mx > 0.f && inv_mx <= 1.0e5f && inv_my > 0.f && inv_my <= 1.0e5f);
        const float m = (view == 0) ? 0.4f : 0.5f;       // utils/loss.py:253-256
        const uint32_t row_bytes = SEG ? (uint32_t)npx * (12u + 4u * TCH) + 2u * seg_bytes + (conf ? (uint32_t)own_n * 4u : 0u)
                                       : (uint32_t)npx * (24u + 4u * TCH) + (conf ? (uint32_t)own_n * 4u : 0u);

        auto issue_row = [&](int ri) {                    // lane 0 only
            const uint32_t p = pos + (uint32_t)ri;
            float* st = ring + (size_t)(p % NS) * St::kFloats;
            uint64_t* bar = &bars[p % NS];
            const size_t rowpix = (size_t)(i_lo + ri) * W;
            const bool with_dz = dz_staged && (i_lo + ri) < rows2;
            mbar_arrive_expect_tx(bar, row_bytes + (with_dz ? (uint32_t)own_n * 2u : 0u));
            if (with_dz) bulk_g2s(st + St::kDz, dz2_strip + (size_t)((i_lo + ri) >> 1) * w2, (uint32_t)own_n * 2u, bar);
            bulk_g2s(st + St::kPred, pred + (rowpix + c0) * 3, (uint32_t)npx * 12u, bar);
            if (SEG) {
                const BTap ty = btap(i_lo + ri, gh, sy);
                bulk_g2s(st + St::kSrc, gt + ((size_t)ty.i0 * gw + rs.s0) * 3, seg_bytes, bar);
                bulk_g2s(st + St::kSrc + SEG * 3, gt + ((size_t)ty.i1 * gw + rs.s0) * 3, seg_bytes, bar);
            } else {
                bulk_g2s(st + St::kGt, gt + (rowpix + c0) * 3, (uint32_t)npx * 12u, bar);
            }
            if (conf) bulk_g2s(st + St::kConf, conf + rowpix + col0, (uint32_t)own_n * 4u, bar);
#pragma unroll
            for (int c = 0; c < TCH; ++c)
                bulk_g2s(st + St::kTh + c * kSegPx, th + (size_t)c * plane + rowpix + c0, (uint32_t)npx * 4u, bar);
        };
        auto stage_of = [&](int ri) { return ring + (size_t)((pos + (uint32_t)ri) % NS) * St::kFloats; };
        auto wait_row = [&](int ri) {
            const uint32_t p = pos + (uint32_t)ri;
            mbar_wait(&bars[p % NS], (p / NS) & 1u);
        };
        auto load = [&](const float* stg, int ri, RowRegs& r) {
            if constexpr (SEG > 0) load_row_rs<TCH, REP, SEG>(stg, idx, j, W - 1, rs, btap(i_lo + ri, gh, sy), r);
            else load_row<TCH, REP>(stg, idx, r);
        };
        auto gt_z = [&](const float* stg, int ri, int px) {          // gt z of smem pixel px of row i_lo + ri
            if constexpr (SEG > 0) return gt_rs<SEG>(stg + St::kSrc, c0 + px, 2, rs, btap(i_lo + ri, gh, sy));
            else return stg[St::kGt + px * 3 + 2];
        };

        if (lane == 0) {
            const int pre = min(NS, n_rows);
            for (int ri = 0; ri < pre; ++ri) issue_row(ri);
        }

        float qy_prev[4] = {0.f, 0.f, 0.f, 0.f};
        float sum_b = 0.f;
        Sums tot = {0.f, 0.f, 0.f};

        // one row: `cur` holds row r, `nxt` receives row r+1 (read once from the ring, current next time)
        auto step = [&](RowRegs& cur, RowRegs& nxt, int ri) {
            const int r = i_lo + ri;
            const bool own = r >= ra;
            const bool has_below = r + 1 < H;
            const float* st = stage_of(ri);
            const float* stn = st;
            if (has_below) {
                wait_row(ri + 1);
                stn = stage_of(ri + 1);
                load(stn, ri + 1, nxt);
            } else {                                      // zero-padded last image row: dy == 0
#pragma unroll
                for (int e = 0; e < 4; ++e) { nxt.P[3 * e + 2] = cur.P[3 * e + 2]; nxt.G[3 * e + 2] = cur.G[3 * e + 2]; nxt.g[e] = cur.g[e]; }
            }

            // ---- horizontal neighbours of the current row (zero-padded last column: dx == 0)
            float zr = __shfl_down_sync(0xffffffffu, cur.P[2], 1);
            float gzr = __shfl_down_sync(0xffffffffu, cur.G[2], 1);
            float gr = __shfl_down_sync(0xffffffffu, cur.g[0], 1);
            if (last_lane) {
                if (right_in_image) {                     // the strip's right halo pixel
                    zr = st[St::kPred + (idx + 4) * 3 + 2];
                    gzr = gt_z(st, ri, idx + 4);
                    gr = gray_px<TCH, REP>(st + St::kTh, idx + 4);
                } else { zr = cur.P[11]; gzr = cur.G[11]; gr = cur.g[3]; }
            }
            const float zx[5] = {cur.P[2], cur.P[5], cur.P[8], cur.P[11], zr};
            const float gzx[5] = {cur.G[2], cur.G[5], cur.G[8], cur.G[11], gzr};
            const float gx[5] = {cur.g[0], cur.g[1], cur.g[2], cur.g[3], gr};

            // ---- edge weights, q terms (each exactly once)
            Sums acc = {0.f, 0.f, 0.f};
            float qx[4], qy[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float w = edge_w(fabsf(gx[e + 1] - gx[e]), fabsf(nxt.g[e] - gx[e]), inv_mx, inv_my, m);
                const float omw = 1.0f - w;
                const float kE_omw = kE * omw, kS2w = kS2 * w;
                qx[e] = q_term(zx[e], zx[e + 1], gzx[e], gzx[e + 1], w, omw, kE_omw, kS2w, kD, acc);
                qy[e] = q_term(zx[e], nxt.P[3 * e + 2], gzx[e], nxt.G[3 * e + 2], w, omw, kE_omw, kS2w, kD, acc);
            }
            // q_x of the pixel left of this quad
            float qxl = __shfl_up_sync(0xffffffffu, qx[3], 1);
            if (lane == 0) {
                qxl = 0.f;
                if (col0 > 0) {                           // pixel col0-1 is in the halo (idx - 1)
                    const float zl = st[St::kPred + (idx - 1) * 3 + 2];
                    const float gzl = gt_z(st, ri, idx - 1);
                    const float gl = gray_px<TCH, REP>(st + St::kTh, idx - 1);
                    const float gln = has_below ? gray_px<TCH, REP>(stn + St::kTh, idx - 1) : gl;
                    const float wl = edge_w(fabsf(gx[0] - gl), fabsf(gln - gl), inv_mx, inv_my, m);
                    const float omw = 1.0f - wl;
                    Sums dummy = {0.f, 0.f, 0.f};
                    qxl = q_term(zl, zx[0], gzl, gzx[0], wl, omw, kE * omw, kS2 * wl, kD, dummy);
                }
            }

            if (own) {
                tot.E += acc.E; tot.S += acc.S; tot.D += acc.D;
                // ---- basic term: utils/loss.py:81-98
                float c[4] = {1.f, 1.f, 1.f, 1.f};
                if (conf) {
                    const float4 cc = *reinterpret_cast<const float4*>(st + St::kConf + 4 * lane);
                    c[0] = cc.x; c[1] = cc.y; c[2] = cc.z; c[3] = cc.w;
                }
                const float dzs[4] = {-qx[0] + qxl - qy[0] + qy_prev[0], -qx[1] + qx[0] - qy[1] + qy_prev[1],
                                      -qx[2] + qx[1] - qy[2] + qy_prev[2], -qx[3] + qx[2] - qy[3] + qy_prev[3]};
                float gq[12], dc[4];
                float2 d2 = make_float2(0.f, 0.f);
                if (S2 && BWD && active && r < rows2)
                    d2 = dz_staged ? *reinterpret_cast<const float2*>(st + St::kDz + 2 * lane)
                                   : __ldg(reinterpret_cast<const float2*>(dz2_ptr + (size_t)(r >> 1) * w2));
                const float dz2[4] = {d2.x, d2.x, d2.y, d2.y};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float dx = cur.P[3 * e] - cur.G[3 * e], dy = cur.P[3 * e + 1] - cur.G[3 * e + 1],
                                dz = cur.P[3 * e + 2] - cur.G[3 * e + 2];
                    const float l = ((fabsf(dx) + fabsf(dy)) + fabsf(dz)) * (1.0f / 3.0f);
                    const float craw = c[e];
                    const float cc = min_nan(max_nan(craw, kConfMin), kConfMax);
                    sum_b += fmaf(cc, l, -alpha_ln2 * __log2f(cc));
                    if (BWD) {
                        const float k3 = cc * kb;
                        gq[3 * e] = times_sgn(k3, dx);
                        gq[3 * e + 1] = times_sgn(k3, dy);
                        gq[3 * e + 2] = times_sgn(k3, dz) + dzs[e] + (S2 ? dz2[e] : 0.f);
                        const bool inside = (craw >= kConfMin) && (craw <= kConfMax);
                        dc[e] = inside ? (l - __fdividef(alpha, cc)) * kc : 0.f;
                    }
                }
                if (BWD && active) {
                    if (dc_ptr) stg_stream_f4(dc_ptr, make_float4(dc[0], dc[1], dc[2], dc[3]));
                    stg_stream_f4(dp_ptr, make_float4(gq[0], gq[1], gq[2], gq[3]));
                    stg_stream_f4(dp_ptr + 4, make_float4(gq[4], gq[5], gq[6], gq[7]));
                    stg_stream_f4(dp_ptr + 8, make_float4(gq[8], gq[9], gq[10], gq[11]));
                }
            }
            if (BWD) { dp_ptr += (size_t)W * 3; if (dc_ptr) dc_ptr += W; }
#pragma unroll
            for (int e = 0; e < 4; ++e) qy_prev[e] = qy[e];

            __syncwarp();                                 // every lane is done reading stage(ri)
            if (lane == 0 && ri + NS < n_rows) issue_row(ri + NS);
        };

        RowRegs A, Bq;
        wait_row(0);
        load(stage_of(0), 0, A);
        const int n_cur = rb - i_lo;                      // rows that are "current" at some iteration
        for (int ri = 0; ri < n_cur; ri += 2) {           // ping-pong the two register sets: no row copies
            step(A, Bq, ri);
            if (ri + 1 < n_cur) step(Bq, A, ri + 1);
        }
        pos += (uint32_t)n_rows;

        // ---- per-task partial sums (fixed butterfly: deterministic); inactive lanes hold garbage
        if (!active) { sum_b = 0.f; tot.E = 0.f; tot.S = 0.f; tot.D = 0.f; }
        sum_b = warp_sum(sum_b);
        tot.E = warp_sum(tot.E); tot.S = warp_sum(tot.S); tot.D = warp_sum(tot.D);
        if (lane == 0) {
            if (thermal_bad) tot.E = __int_as_float(0x7fc00000);
            float4* o = reinterpret_cast<float4*>(a.partials + (size_t)pidx * 8);
            o[0] = make_float4(sum_b, tot.E, tot.S, tot.D);
            o[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

template <int TCH, bool REP, bool BWD, bool S2, int NS, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1) loss_march_kernel(const MarchArgs a) {
    march_body<TCH, REP, BWD, S2, 0, NS, WARPS>(a);
}
template <int TCH, bool REP, bool BWD, int SEG, int NS, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1) loss_march_rs_kernel(const MarchArgs a) {
    march_body<TCH, REP, BWD, false, SEG, NS, WARPS>(a);
}

// ====================================================================== multi-scale in ONE pass
// loss_march_ms_kernel: the full-resolution march above AND the half-resolution (scale 2) terms of
// utils/loss.py:133-174,288-292 over the same staged rows, so that pred / gt / thermal are read from DRAM once
// (the split path -- t3d_loss_scale2.cu, then the marching kernel -- reads them twice and round-trips the pooled
// gradient through memory).  The scale-2 gradient of pooled cell (I, J) needs the pooled rows I-1, I, I+1, i.e. the
// full-resolution rows up to 2I+3 while row 2I is being written: the ring is two stages deeper and the warp pools
// rows r+2, r+3 when it starts the row pair (r, r+1); a band brings two more halo rows (r-2 and rb+1).
// The confidence row no longer travels through the ring (it is not needed ahead of time): each lane fetches its
// four values one row ahead into registers, which leaves shared memory for the deeper ring.
// Thermal: one staged plane (TCH == 1, or three bit-identical replicas).
struct StageF {
    static constexpr int kPred = 0;
    static constexpr int kGt = kSegPx * 3;
    static constexpr int kTh = 2 * kSegPx * 3;
    static constexpr int kFloats = kTh + kSegPx;           // 952 floats = 3808 bytes
};

struct Cell3 { float z, gz, g; };
struct Row2 { float z[2], gz[2], g[2]; Cell3 h; };     // one lane's two pooled cells; h: the strip's left halo cell in lane 0,
                                                        // its right halo cell in the last lane (a lane never needs both: a strip
                                                        // of 4 pixels is the image's last)

// Z of 4 consecutive AoS pixels (3 x 128-bit shared loads)
__device__ __forceinline__ void z_quad(const float* __restrict__ base, int idx, float z[4]) {
    const float4* v = reinterpret_cast<const float4*>(base + idx * 3);
    const float4 x0 = v[0], x1 = v[1], x2 = v[2];
    z[0] = x0.z; z[1] = x1.y; z[2] = x2.x; z[3] = x2.w;
}
__device__ __forceinline__ float pool4(float a0, float a1, float b0, float b1) { return 0.25f * (((a0 + a1) + b0) + b1); }

template <bool REP>
__device__ __forceinline__ Cell3 pool_cell(const float* __restrict__ s0, const float* __restrict__ s1, int px) {
    Cell3 c;
    c.z = pool4(s0[StageF::kPred + px * 3 + 2], s0[StageF::kPred + px * 3 + 5], s1[StageF::kPred + px * 3 + 2], s1[StageF::kPred + px * 3 + 5]);
    c.gz = pool4(s0[StageF::kGt + px * 3 + 2], s0[StageF::kGt + px * 3 + 5], s1[StageF::kGt + px * 3 + 2], s1[StageF::kGt + px * 3 + 5]);
    c.g = pool4(gray_px<1, REP>(s0 + StageF::kTh, px), gray_px<1, REP>(s0 + StageF::kTh, px + 1),
                gray_px<1, REP>(s1 + StageF::kTh, px), gray_px<1, REP>(s1 + StageF::kTh, px + 1));
    return c;
}

template <bool REP, bool BWD, int NS, int WARPS>
__global__ void __maxnreg__((WARPS >= 12) ? 168 : 255) loss_march_ms_kernel(const MarchArgs a) {
    using St = StageF;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    float* ring = reinterpret_cast<float*>(smem_raw) + (size_t)wrp * NS * St::kFloats;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)WARPS * NS * St::kFloats * sizeof(float)) + wrp * NS;

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();

    const int H = a.H, W = a.W, h2 = H >> 1, w2 = W >> 1;
    const size_t plane = (size_t)H * W;
    const int nbands = a.nbands_l + a.nbands_s;
    const int n_large = a.B * 2 * a.nbands_l * a.nstrips;
    const int ntasks = a.B * 2 * nbands * a.nstrips;
    const float kE = a.kE, kS2 = 2.0f * a.kS, kD = a.kD, kb = a.kb, kc = a.kc, alpha = a.alpha;
    const float kE_2 = a.kE2, kS2_2 = 2.0f * a.kS2, kD_2 = a.kD2;
    const float alpha_ln2 = alpha * 0.69314718055994531f;
    uint32_t pos = 0;

    for (;;) {
        int task = 0;
        if (lane == 0) task = (int)atomicAdd(a.queue, 1u);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= ntasks) break;
        const bool large = task < n_large;
        const int t1 = large ? task : task - n_large;
        const int nb = large ? a.nbands_l : a.nbands_s;
        const int s = t1 % a.nstrips;
        const int t2 = t1 / a.nstrips;
        const int k = t2 % nb;
        const int img = t2 / nb;
        const int b = img >> 1, view = img & 1;
        const int ra = large ? k * a.rows_l : a.nbands_l * a.rows_l + k * a.rows_s;            // even (rows_l, rows_s are)
        const int rb = large ? ra + a.rows_l : min(ra + a.rows_s, H);
        const int pidx = (img * nbands + (large ? k : a.nbands_l + k)) * a.nstrips + s;
        const int i_lo = max(ra - 2, 0), i_hi = min(rb + 1, H - 1);                            // i_lo even
        const int n_rows = i_hi - i_lo + 1;
        const int ri_first = (ra > 0) ? 1 : 0;             // ring index of the first row that is "current" for the full-resolution march
        const int I_a = ra >> 1;                            // pooled rows [I_a, min(rb / 2, h2)) are this band's own
        const int col0 = s * kStripPx;
        const int c0 = max(col0 - 4, 0), c1 = min(col0 + kStripPx + 4, W);
        const int npx = c1 - c0, off = col0 - c0;
        const int own_n = min(kStripPx, W - col0);
        const int j = col0 + 4 * lane;
        const bool active = 4 * lane < own_n;
        const bool last_lane = active && (4 * lane + 4 >= own_n);
        const bool right_in_image = (j + 4 < W);
        const int idx = 4 * lane + off;

        const float* __restrict__ pred = a.pred[view] + (size_t)b * plane * 3;
        const float* __restrict__ gt = a.gt[view] + (size_t)b * plane * 3;
        const float* __restrict__ th = a.thermal[view] + (size_t)b * (REP ? 3 : 1) * plane;
        const int r_first = i_lo + ri_first;
        const float* c_ptr = a.conf[view] ? a.conf[view] + (size_t)b * plane + (size_t)r_first * W + j : nullptr;
        float* dp_ptr = BWD ? a.dpred[view] + ((size_t)b * plane + (size_t)r_first * W + j) * 3 : nullptr;
        float* dc_ptr = (BWD && a.dconf[view]) ? a.dconf[view] + (size_t)b * plane + (size_t)r_first * W + j : nullptr;

        // 1 / (mean + eps) of the thermal gradients at both scales: fixed-order sums of the stats partials
        float inv_mx, inv_my, inv_mx2, inv_my2;
        {
            float sx = 0.f, sy = 0.f;
            double sx2 = 0.0, sy2 = 0.0;
            const float4* sp = reinterpret_cast<const float4*>(a.stats[view] + (size_t)b * a.stiles * 4);
            for (int t = lane; t < a.stiles; t += 32) { const float4 v = sp[t]; sx += v.x; sy += v.y; sx2 += (double)v.z; sy2 += (double)v.w; }
            sx = warp_sum(sx); sy = warp_sum(sy); sx2 = warp_sum(sx2); sy2 = warp_sum(sy2);
            const float invN = 1.0f / (float)plane;
            inv_mx = 1.0f / (sx * invN + kEps);
            inv_my = 1.0f / (sy * invN + kEps);
            const double n2 = (double)h2 * w2;
            inv_mx2 = 1.0f / ((float)(sx2 / n2) + kEps);
            inv_my2 = 1.0f / ((float)(sy2 / n2) + kEps);
        }
        const bool thermal_bad = !(inv_mx > 0.f && inv_mx <= 1.0e5f && inv_my > 0.f && inv_my <= 1.0e5f);
        const bool thermal_bad2 = !(inv_mx2 > 0.f && inv_mx2 <= 1.0e5f && inv_my2 > 0.f && inv_my2 <= 1.0e5f);
        const float m = (view == 0) ? 0.4f : 0.5f;
        const uint32_t row_bytes = (uint32_t)npx * 28u;

        auto issue_row = [&](int ri) {                    // lane 0 only
            const uint32_t p = pos + (uint32_t)ri;
            float* st = ring + (size_t)(p % NS) * St::kFloats;
            uint64_t* bar = &bars[p % NS];
            const size_t rowpix = (size_t)(i_lo + ri) * W;
            mbar_arrive_expect_tx(bar, row_bytes);
            bulk_g2s(st + St::kPred, pred + (rowpix + c0) * 3, (uint32_t)npx * 12u, bar);
            bulk_g2s(st + St::kGt, gt + (rowpix + c0) * 3, (uint32_t)npx * 12u, bar);
            bulk_g2s(st + St::kTh, th + rowpix + c0, (uint32_t)npx * 4u, bar);
        };
        auto stage_of = [&](int ri) { return ring + (size_t)((pos + (uint32_t)ri) % NS) * St::kFloats; };
        auto wait_row = [&](int ri) {
            const uint32_t p = pos + (uint32_t)ri;
            mbar_wait(&bars[p % NS], (p / NS) & 1u);
        };
        const bool left_halo = (lane == 0) && (col0 > 0), right_halo = last_lane && right_in_image;
        const bool halo_lane = left_halo || right_halo;
        const int halo_px = left_halo ? idx - 2 : idx + 4;
        // pooled row from two staged rows: this lane's two cells, and the strip's halo cells in lane 0 / the last lane
        auto pool_row = [&](int ri, Row2& o) {
            const float* s0 = stage_of(ri);
            const float* s1 = stage_of(ri + 1);
            float u[4], v[4];
            z_quad(s0 + St::kPred, idx, u); z_quad(s1 + St::kPred, idx, v);
            o.z[0] = pool4(u[0], u[1], v[0], v[1]); o.z[1] = pool4(u[2], u[3], v[2], v[3]);
            z_quad(s0 + St::kGt, idx, u); z_quad(s1 + St::kGt, idx, v);
            o.gz[0] = pool4(u[0], u[1], v[0], v[1]); o.gz[1] = pool4(u[2], u[3], v[2], v[3]);
            gray_quad<1, REP>(s0 + St::kTh, idx, u); gray_quad<1, REP>(s1 + St::kTh, idx, v);
            o.g[0] = pool4(u[0], u[1], v[0], v[1]); o.g[1] = pool4(u[2], u[3], v[2], v[3]);
            if (halo_lane) o.h = pool_cell<REP>(s0, s1, halo_px);
        };

        if (lane == 0) {
            const int pre = min(NS, n_rows);
            for (int ri = 0; ri < pre; ++ri) issue_row(ri);
        }

        float qy_prev[4] = {0.f, 0.f, 0.f, 0.f};
        float qy2_prev[2] = {0.f, 0.f};
        float sum_b = 0.f;
        Sums tot = {0.f, 0.f, 0.f}, tot2 = {0.f, 0.f, 0.f};
        float4 c_cur = make_float4(1.f, 1.f, 1.f, 1.f), c_nxt = c_cur;
        if (c_ptr && active && r_first >= ra) c_cur = ldg_stream_f4(c_ptr);

        // one full-resolution row (same as loss_march_kernel's step); d2 = this lane's two pooled-cell gradients
        // HOLD (the even row of a pair): its pooled cell's gradient is not known yet -- d(pred) stays in `held` and is
        // written by the caller once the next pooled row has arrived (two rows of lookahead instead of three)
        float held[12];
        // Register diet (12 warps x 168 registers): only the gray values of the current row are carried from step to
        // step; its pointmaps are read from its (still resident) stage when the step starts, and of the row below only
        // z, gt z and gray are read.
        float g_cur[4];
        auto step = [&](int ri, float2 d2, auto hold_tag) {
            constexpr bool HOLD = decltype(hold_tag)::value;
            const int r = i_lo + ri;
            const bool own = r >= ra;
            const bool has_below = r + 1 < H;
            if (c_ptr && active && r + 1 < rb) c_nxt = ldg_stream_f4(c_ptr + W);      // the next row's confidences, one row ahead
            const float* st = stage_of(ri);
            const float* stn = st;
            RowRegs cur;
            {
                const float4* p = reinterpret_cast<const float4*>(st + St::kPred + idx * 3);
                const float4* q = reinterpret_cast<const float4*>(st + St::kGt + idx * 3);
                const float4 a = p[0], b = p[1], c = p[2], d = q[0], e = q[1], f = q[2];
                cur.P[0] = a.x; cur.P[1] = a.y; cur.P[2] = a.z; cur.P[3] = a.w; cur.P[4] = b.x; cur.P[5] = b.y; cur.P[6] = b.z; cur.P[7] = b.w;
                cur.P[8] = c.x; cur.P[9] = c.y; cur.P[10] = c.z; cur.P[11] = c.w;
                cur.G[0] = d.x; cur.G[1] = d.y; cur.G[2] = d.z; cur.G[3] = d.w; cur.G[4] = e.x; cur.G[5] = e.y; cur.G[6] = e.z; cur.G[7] = e.w;
                cur.G[8] = f.x; cur.G[9] = f.y; cur.G[10] = f.z; cur.G[11] = f.w;
#pragma unroll
                for (int e2 = 0; e2 < 4; ++e2) cur.g[e2] = g_cur[e2];
            }
            float nz[4], ngz[4], ng[4];
            if (has_below) {
                wait_row(ri + 1);
                stn = stage_of(ri + 1);
#pragma unroll
                for (int e = 0; e < 4; ++e) { nz[e] = stn[St::kPred + (idx + e) * 3 + 2]; ngz[e] = stn[St::kGt + (idx + e) * 3 + 2]; }
                gray_quad<1, REP>(stn + St::kTh, idx, ng);
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) { nz[e] = cur.P[3 * e + 2]; ngz[e] = cur.G[3 * e + 2]; ng[e] = cur.g[e]; }
            }
            float zr = __shfl_down_sync(0xffffffffu, cur.P[2], 1);
            float gzr = __shfl_down_sync(0xffffffffu, cur.G[2], 1);
            float gr = __shfl_down_sync(0xffffffffu, cur.g[0], 1);
            if (last_lane) {
                if (right_in_image) {
                    zr = st[St::kPred + (idx + 4) * 3 + 2];
                    gzr = st[St::kGt + (idx + 4) * 3 + 2];
                    gr = gray_px<1, REP>(st + St::kTh, idx + 4);
                } else { zr = cur.P[11]; gzr = cur.G[11]; gr = cur.g[3]; }
            }
            const float zx[5] = {cur.P[2], cur.P[5], cur.P[8], cur.P[11], zr};
            const float gzx[5] = {cur.G[2], cur.G[5], cur.G[8], cur.G[11], gzr};
            const float gx[5] = {cur.g[0], cur.g[1], cur.g[2], cur.g[3], gr};
            Sums acc = {0.f, 0.f, 0.f};
            float qx[4], qy[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float w = edge_w(fabsf(gx[e + 1] - gx[e]), fabsf(ng[e] - gx[e]), inv_mx, inv_my, m);
                const float omw = 1.0f - w;
                const float kE_omw = kE * omw, kS2w = kS2 * w;
                qx[e] = q_term(zx[e], zx[e + 1], gzx[e], gzx[e + 1], w, omw, kE_omw, kS2w, kD, acc);
                qy[e] = q_term(zx[e], nz[e], gzx[e], ngz[e], w, omw, kE_omw, kS2w, kD, acc);
            }
            float qxl = __shfl_up_sync(0xffffffffu, qx[3], 1);
            if (lane == 0) {
                qxl = 0.f;
                if (col0 > 0) {
                    const float zl = st[St::kPred + (idx - 1) * 3 + 2];
                    const float gzl = st[St::kGt + (idx - 1) * 3 + 2];
                    const float gl = gray_px<1, REP>(st + St::kTh, idx - 1);
                    const float gln = has_below ? gray_px<1, REP>(stn + St::kTh, idx - 1) : gl;
                    const float wl = edge_w(fabsf(gx[0] - gl), fabsf(gln - gl), inv_mx, inv_my, m);
                    const float omw = 1.0f - wl;
                    Sums dummy = {0.f, 0.f, 0.f};
                    qxl = q_term(zl, zx[0], gzl, gzx[0], wl, omw, kE * omw, kS2 * wl, kD, dummy);
                }
            }
            if (own) {
                tot.E += acc.E; tot.S += acc.S; tot.D += acc.D;
                const float c[4] = {c_cur.x, c_cur.y, c_cur.z, c_cur.w};
                const float dzs[4] = {-qx[0] + qxl - qy[0] + qy_prev[0], -qx[1] + qx[0] - qy[1] + qy_prev[1],
                                      -qx[2] + qx[1] - qy[2] + qy_prev[2], -qx[3] + qx[2] - qy[3] + qy_prev[3]};
                const float dz2[4] = {d2.x, d2.x, d2.y, d2.y};
                float gq[12], dc[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float dx = cur.P[3 * e] - cur.G[3 * e], dy = cur.P[3 * e + 1] - cur.G[3 * e + 1],
                                dz = cur.P[3 * e + 2] - cur.G[3 * e + 2];
                    const float l = ((fabsf(dx) + fabsf(dy)) + fabsf(dz)) * (1.0f / 3.0f);
                    const float craw = c[e];
                    const float cc = min_nan(max_nan(craw, kConfMin), kConfMax);
                    sum_b += fmaf(cc, l, -alpha_ln2 * __log2f(cc));
                    if (BWD) {
                        const float k3 = cc * kb;
                        gq[3 * e] = times_sgn(k3, dx);
                        gq[3 * e + 1] = times_sgn(k3, dy);
                        gq[3 * e + 2] = times_sgn(k3, dz) + dzs[e] + dz2[e];
                        const bool inside = (craw >= kConfMin) && (craw <= kConfMax);
                        dc[e] = inside ? (l - __fdividef(alpha, cc)) * kc : 0.f;
                    }
                }
                if (BWD && active) {
                    if (dc_ptr) stg_stream_f4(dc_ptr, make_float4(dc[0], dc[1], dc[2], dc[3]));
                    if (!HOLD) {
                        stg_stream_f4(dp_ptr, make_float4(gq[0], gq[1], gq[2], gq[3]));
                        stg_stream_f4(dp_ptr + 4, make_float4(gq[4], gq[5], gq[6], gq[7]));
                        stg_stream_f4(dp_ptr + 8, make_float4(gq[8], gq[9], gq[10], gq[11]));
                    }
                }
                if (BWD && HOLD) {
#pragma unroll
                    for (int e = 0; e < 12; ++e) held[e] = gq[e];
                }
            }
            if (BWD) { dp_ptr += (size_t)W * 3; if (dc_ptr) dc_ptr += W; }
            if (c_ptr) { c_ptr += W; c_cur = c_nxt; }
#pragma unroll
            for (int e = 0; e < 4; ++e) { qy_prev[e] = qy[e]; g_cur[e] = ng[e]; }
            __syncwarp();
            if (lane == 0 && ri + NS < n_rows) issue_row(ri + NS);
        };

        Row2 C2, N2;
        C2.h = Cell3{0.f, 0.f, 0.f}; N2.h = C2.h;
        wait_row(0);
        if (n_rows > 1) wait_row(1);
        if ((i_lo >> 1) < h2) pool_row(0, C2);              // n_rows >= 2 whenever a pooled row starts at i_lo
        gray_quad<1, REP>(stage_of(ri_first) + St::kTh, idx, g_cur);
        const int n_cur = rb - i_lo;
        for (int ri = 0; ri < n_cur; ri += 2) {             // row pair (2I, 2I+1) = pooled row I
            const int I = (i_lo + ri) >> 1;
            const bool even_own = BWD && (ri >= ri_first) && (i_lo + ri >= ra);
            // ---- the even row: everything but the pooled cell's share of d(pred z)
            if (ri >= ri_first) step(ri, make_float2(0.f, 0.f), std::true_type{});
            else {                                          // row ra-2 only feeds the pooled row above the band
                __syncwarp();
                if (lane == 0 && NS < n_rows) issue_row(NS);
            }
            // ---- pooled row I (needs pooled row I+1 = rows 2I+2, 2I+3)
            float2 d2 = make_float2(0.f, 0.f);
            if (I < h2) {
                if (I + 1 < h2) { wait_row(ri + 2); wait_row(ri + 3); pool_row(ri + 2, N2); }
                else N2 = C2;                               // zero-padded last pooled row: dy == 0
                float zr = __shfl_down_sync(0xffffffffu, C2.z[0], 1);
                float gzr = __shfl_down_sync(0xffffffffu, C2.gz[0], 1);
                float gr = __shfl_down_sync(0xffffffffu, C2.g[0], 1);
                if (last_lane) {
                    if (right_in_image) { zr = C2.h.z; gzr = C2.h.gz; gr = C2.h.g; }
                    else { zr = C2.z[1]; gzr = C2.gz[1]; gr = C2.g[1]; }      // zero-padded last pooled column: dx == 0
                }
                const float zx[3] = {C2.z[0], C2.z[1], zr}, gzx[3] = {C2.gz[0], C2.gz[1], gzr}, gx[3] = {C2.g[0], C2.g[1], gr};
                Sums acc = {0.f, 0.f, 0.f};
                float qx[2], qy[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const float w = edge_w(fabsf(gx[e + 1] - gx[e]), fabsf(N2.g[e] - gx[e]), inv_mx2, inv_my2, m);
                    const float omw = 1.0f - w;
                    const float kE_omw = kE_2 * omw, kS2w = kS2_2 * w;
                    qx[e] = q_term(zx[e], zx[e + 1], gzx[e], gzx[e + 1], w, omw, kE_omw, kS2w, kD_2, acc);
                    qy[e] = q_term(zx[e], N2.z[e], gzx[e], N2.gz[e], w, omw, kE_omw, kS2w, kD_2, acc);
                }
                float qxl = __shfl_up_sync(0xffffffffu, qx[1], 1);
                if (lane == 0) {
                    qxl = 0.f;
                    if (col0 > 0) {
                        const float wl = edge_w(fabsf(gx[0] - C2.h.g), fabsf(N2.h.g - C2.h.g), inv_mx2, inv_my2, m);
                        const float omw = 1.0f - wl;
                        Sums dummy = {0.f, 0.f, 0.f};
                        qxl = q_term(C2.h.z, zx[0], C2.h.gz, gzx[0], wl, omw, kE_2 * omw, kS2_2 * wl, kD_2, dummy);
                    }
                }
                if (I >= I_a) { tot2.E += acc.E; tot2.S += acc.S; tot2.D += acc.D; }
                d2.x = 0.25f * (-qx[0] + qxl - qy[0] + qy2_prev[0]);
                d2.y = 0.25f * (-qx[1] + qx[0] - qy[1] + qy2_prev[1]);
                qy2_prev[0] = qy[0]; qy2_prev[1] = qy[1];
                C2 = N2;
            }
            // ---- the held even row leaves with its pooled cells' share (dp_ptr already points at the odd row)
            if (even_own && active) {
                float* o = dp_ptr - (size_t)W * 3;
                stg_stream_f4(o, make_float4(held[0], held[1], held[2] + d2.x, held[3]));
                stg_stream_f4(o + 4, make_float4(held[4], held[5] + d2.x, held[6], held[7]));
                stg_stream_f4(o + 8, make_float4(held[8] + d2.y, held[9], held[10], held[11] + d2.y));
            }
            if (ri + 1 < n_cur) step(ri + 1, d2, std::false_type{});
        }
        pos += (uint32_t)n_rows;

        if (!active) { sum_b = 0.f; tot.E = 0.f; tot.S = 0.f; tot.D = 0.f; tot2.E = 0.f; tot2.S = 0.f; tot2.D = 0.f; }
        sum_b = warp_sum(sum_b);
        tot.E = warp_sum(tot.E); tot.S = warp_sum(tot.S); tot.D = warp_sum(tot.D);
        tot2.E = warp_sum(tot2.E); tot2.S = warp_sum(tot2.S); tot2.D = warp_sum(tot2.D);
        if (lane == 0) {
            if (thermal_bad) tot.E = __int_as_float(0x7fc00000);
            if (thermal_bad2) tot2.E = __int_as_float(0x7fc00000);
            float4* o = reinterpret_cast<float4*>(a.partials + (size_t)pidx * 8);
            o[0] = make_float4(sum_b, tot.E, tot.S, tot.D);
            o[1] = make_float4(tot2.E, tot2.S, tot2.D, 0.f);
        }
    }
}

// 12 warps x 5 ring stages x 168 registers: registers are allocated to a CTA in units of 4 warps, so 10 or 11 warps with
// more registers each do not launch, and 8 warps run slower (DESIGN §4, loss_march_ms_kernel)
template <bool REP, bool BWD>
int launch_ms(const MarchArgs& a, cudaStream_t st) {
    constexpr int NS = 5, WARPS = 12;
    constexpr size_t smem = (size_t)WARPS * NS * StageF::kFloats * sizeof(float) + (size_t)WARPS * NS * 8;
    static_assert(smem <= 227 * 1024, "ring does not fit in shared memory");
    static bool attr_done[kT3dMaxDevices] = {};
    bool& attr_set = attr_done[t3d_device_slot()];
    if (!attr_set) {
        T3D_CUDA(cudaFuncSetAttribute(loss_march_ms_kernel<REP, BWD, NS, WARPS>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    T3D_LAUNCH("loss_march_ms_kernel", st,
               loss_march_ms_kernel<REP, BWD, NS, WARPS><<<t3d_sm_count(), WARPS * 32, smem, st>>>(a));
    return T3D_OK;
}

// One persistent CTA per SM with as many warps as the register file / shared memory hold: 12, or 10 with three staged
// thermal planes.  Fewer warps (DESIGN §4 experiment 2) or fewer CTAs (experiment 15) slow the step.
template <int TCH, bool REP, bool BWD, bool S2>
int launch(const MarchArgs& a, cudaStream_t st) {
    constexpr int NS = 4, WARPS = (TCH == 3) ? 10 : 12;
    constexpr size_t smem = (size_t)WARPS * NS * Stage<TCH, S2>::kFloats * sizeof(float) + (size_t)WARPS * NS * 8;
    static_assert(smem <= 227 * 1024, "ring does not fit in shared memory");
    static bool attr_done[kT3dMaxDevices] = {};
    bool& attr_set = attr_done[t3d_device_slot()];
    if (!attr_set) {
        T3D_CUDA(cudaFuncSetAttribute(loss_march_kernel<TCH, REP, BWD, S2, NS, WARPS>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    T3D_LAUNCH("loss_march_kernel", st,
               loss_march_kernel<TCH, REP, BWD, S2, NS, WARPS><<<t3d_sm_count(), WARPS * 32, smem, st>>>(a));
    return T3D_OK;
}

// Resampled gt: the marching kernel stages the gt source rows only while a strip's segment (t3d_loss_march_rs_span)
// is at most kSegMax pixels -- gt_w = W, e.g. 512x384 <- 512x512: 364 us against 696 us on the tile kernel (batch 64).
// Wider segments (gt_w up to 2.3 W, e.g. 224x224 <- 512x512) measured slower than the tile kernel with its fused taps
// (92 vs 77 us at batch 8: a third of the warps of a 320-pixel ring, a grid far from full) and stay there (DESIGN §4).
// 8 warps x 4 stages: the backward instances need ~230 registers (the taps), 8 warps of them fit an SM without spilling.
constexpr int kSegMax = 144;
template <int TCH, bool REP, bool BWD>
int launch_rs(const MarchArgs& a, cudaStream_t st) {
    constexpr int NS = 4, WARPS = 8;
    constexpr size_t smem = (size_t)WARPS * NS * Stage<TCH, false, kSegMax>::kFloats * sizeof(float) + (size_t)WARPS * NS * 8;
    static_assert(smem <= 227 * 1024, "ring does not fit in shared memory");
    static bool attr_done[kT3dMaxDevices] = {};
    bool& attr_set = attr_done[t3d_device_slot()];
    if (!attr_set) {
        T3D_CUDA(cudaFuncSetAttribute(loss_march_rs_kernel<TCH, REP, BWD, kSegMax, NS, WARPS>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    T3D_LAUNCH("loss_march_rs_kernel", st,
               loss_march_rs_kernel<TCH, REP, BWD, kSegMax, NS, WARPS><<<t3d_sm_count(), WARPS * 32, smem, st>>>(a));
    return T3D_OK;
}

}  // namespace

// the kernel's segment arithmetic (march_body), evaluated on the host with the same roundings (btap)
int t3d_loss_march_rs_span(int W, int gt_w) {
    const float sx = bscale(gt_w, W);
    int span = 0;
    for (int col0 = 0; col0 < W; col0 += kStripPx) {
        const int c0 = max(col0 - 4, 0), c1 = min(col0 + kStripPx + 4, W);
        const int s0 = btap(c0, gt_w, sx).i0 & ~3, s1 = (btap(c1 - 1, gt_w, sx).i1 + 4) & ~3;
        span = max(span, s1 - s0);
    }
    return span;
}

bool t3d_loss_march_rs_fits(int span) { return span <= kSegMax; }

int t3d_launch_loss_march_rs(const MarchArgs& a, int span, bool bwd, cudaStream_t st) {
    T3D_REQUIRE(t3d_loss_march_rs_fits(span), "gt segment of %d pixels does not fit the resampling kernel", span);
    if (a.tch == 3 && a.replicated) return bwd ? launch_rs<1, true, true>(a, st) : launch_rs<1, true, false>(a, st);
    if (a.tch == 3) return bwd ? launch_rs<3, false, true>(a, st) : launch_rs<3, false, false>(a, st);
    return bwd ? launch_rs<1, false, true>(a, st) : launch_rs<1, false, false>(a, st);
}

// multi-scale in one pass; requires what t3d_launch_loss_march does, plus: tch == 1 or replicated planes, H >= 4,
// rows_l and rows_s even
int t3d_launch_loss_march_ms(const MarchArgs& a, bool bwd, cudaStream_t st) {
    if (a.tch == 3 && a.replicated) return bwd ? launch_ms<true, true>(a, st) : launch_ms<true, false>(a, st);
    return bwd ? launch_ms<false, true>(a, st) : launch_ms<false, false>(a, st);
}

int t3d_launch_loss_march(const MarchArgs& a, bool bwd, cudaStream_t st) {
    const bool s2 = bwd && a.dzp[0] != nullptr && a.dzp[1] != nullptr;
    if (s2) {       // multi-scale backward: add the scale-2 gradient
        if (a.tch == 3 && a.replicated) return launch<1, true, true, true>(a, st);
        if (a.tch == 3) return launch<3, false, true, true>(a, st);
        return launch<1, false, true, true>(a, st);
    }
    if (a.tch == 3 && a.replicated) return bwd ? launch<1, true, true, false>(a, st) : launch<1, true, false, false>(a, st);
    if (a.tch == 3) return bwd ? launch<3, false, true, false>(a, st) : launch<3, false, false, false>(a, st);
    return bwd ? launch<1, false, true, false>(a, st) : launch<1, false, false, false>(a, st);
}
