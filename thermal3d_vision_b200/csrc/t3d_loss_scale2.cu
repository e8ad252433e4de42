// t3d_loss_scale2.cu -- the half-resolution (scale 2) terms of the multi-scale thermal-aware loss
// (utils/loss.py:133-174,288-292) as their own pass, so that the full-resolution terms and the basic term
// can stay on the TMA-fed marching kernel (t3d_loss_march.cu).
//
// Per (image, view): z, gt z and gray are 2x2 average-pooled (floor division of H, W; sum * 0.25), the edge,
// smoothness and detail terms are evaluated on the pooled planes exactly as at full resolution (zero-padded
// forward differences, weights from the pooled gray gradients normalised by their image mean) with the scale
// weight 0.7 / 2, and the gradient with respect to a pooled cell is spread 0.25 to each of its four pixels
// (SURVEY.md Appendix A).  Outputs: the three partial sums per tile, and dzp[b][I][J] = 0.25 * d(loss)/d(pooled z)
// which the marching kernel adds to d(loss)/d(pred z) of the four pixels of cell (I, J).
#include "t3d_loss_internal.cuh"

namespace {

constexpr int kT2H = 16, kT2W = 64, kS2Threads = 256;      // pooled cells per CTA
constexpr int kR2H = kT2H + 2, kR2W = kT2W + 4;            // rows: one halo cell each side; columns: two on the left (so that a
                                                           // region row starts on a 4-pixel boundary), one used + one spare right

struct Sums3 { float E, S, D; };

// one forward-difference term; `valid` false = zero-padded last column / row
__device__ __forceinline__ float q_term2(bool valid, float za, float zb, float ga, float gb, float w,
                                         float kE, float kS2, float kD, bool count, Sums3& acc) {
    if (!valid) return 0.f;
    const float s = zb - za, a = fabsf(s), b = fabsf(gb - ga), e = a - b, d = fabsf(e);
    const float c = fminf(d, kHuber);
    if (count) {
        acc.E = fmaf(a, 1.0f - w, acc.E);
        acc.S = fmaf(a * a, w, acc.S);
        acc.D += fmaf(0.5f * c, c, kHuber * (d - c));           // huber(d) = c^2 / 2 + delta (d - c)
    }
    const float dh = fminf(fmaxf(e, -kHuber), kHuber);          // rho'(d) sgn(e)
    return times_sgn(fmaf(kD, dh, fmaf(kS2 * w, a, kE * (1.0f - w))), s);
}

template <bool BWD>
__global__ void __launch_bounds__(kS2Threads) loss_scale2_kernel(const Scale2Args a) {
    __shared__ float pz[kR2H][kR2W], pgz[kR2H][kR2W], pg[kR2H][kR2W];
    __shared__ float sqx[kT2H + 1][kT2W + 1], sqy[kT2H + 1][kT2W + 1];   // q of cells I0-1.., J0-1..
    __shared__ float red[kS2Threads / 32][3];
    __shared__ float s_inv[2];
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int H = a.H, W = a.W, h2 = H >> 1, w2 = W >> 1;
    const int tiles = a.tiles_x * a.tiles_y;
    const int img = blockIdx.x / tiles, tile = blockIdx.x - img * tiles;
    const int tyi = tile / a.tiles_x, txi = tile - tyi * a.tiles_x;
    const int I0 = tyi * kT2H, J0 = txi * kT2W;
    const int b = img >> 1, view = img & 1;
    const size_t plane = (size_t)H * W;
    const float* __restrict__ pred = a.pred[view] + (size_t)b * plane * 3;
    const float* __restrict__ gt = a.gt[view] + (size_t)b * plane * 3;
    const float* __restrict__ th = a.thermal[view] + (size_t)b * a.tch * plane;
    const int tch = a.replicated ? 1 : a.tch;

    // 1 / (mean + eps) of the pooled thermal gradients of this image (fixed-order sum of the stats partials)
    if (wrp < 2) {                      // warp 0: Dx sums, warp 1: Dy sums; lane t owns partials t, t + 32, ...; fixed butterfly
        double s = 0.0;
        const float* sp = a.stats[view] + (size_t)b * a.stiles * 4 + 2 + wrp;
        for (int t = lane; t < a.stiles; t += 32) s += (double)sp[(size_t)t * 4];
        s = warp_sum(s);
        const double n2 = (double)h2 * w2;
        if (lane == 0) s_inv[wrp] = 1.0f / ((float)(s / n2) + kEps);
    }
    // ---- pooled planes of cells I0-1 .. I0+kT2H, J0-2 .. J0+kT2W+1 (cells outside the pooled image: 0).
    // One work item = two horizontally adjacent cells = 4 pixels x 2 rows: 128-bit loads (W % 4 == 0, aligned).
    for (int k = tid; k < kR2H * (kR2W / 2); k += kS2Threads) {
        const int R = k / (kR2W / 2), Cp = k - R * (kR2W / 2);
        const int I = I0 - 1 + R, J = J0 - 2 + 2 * Cp;          // J even; w2 even: the pair is inside or outside together
        float2 vz = make_float2(0.f, 0.f), vgz = vz, vg = vz;
        if (I >= 0 && J >= 0 && I < h2 && J < w2) {
            const size_t p0 = (size_t)(2 * I) * W + 2 * J, p1 = p0 + W;
            auto zrow = [&](const float* q, size_t p, float z[4]) {      // Z of 4 consecutive AoS pixels
                const float4* v = reinterpret_cast<const float4*>(q + p * 3);
                const float4 x0 = __ldg(v), x1 = __ldg(v + 1), x2 = __ldg(v + 2);
                z[0] = x0.z; z[1] = x1.y; z[2] = x2.x; z[3] = x2.w;
            };
            auto grow = [&](size_t p, float g[4]) {
                const float4 c0 = __ldg(reinterpret_cast<const float4*>(th + p));
                if (a.replicated) {
                    g[0] = gray3(c0.x, c0.x, c0.x); g[1] = gray3(c0.y, c0.y, c0.y); g[2] = gray3(c0.z, c0.z, c0.z); g[3] = gray3(c0.w, c0.w, c0.w);
                } else if (tch == 3) {
                    const float4 c1 = __ldg(reinterpret_cast<const float4*>(th + plane + p)), c2 = __ldg(reinterpret_cast<const float4*>(th + 2 * plane + p));
                    g[0] = gray3(c0.x, c1.x, c2.x); g[1] = gray3(c0.y, c1.y, c2.y); g[2] = gray3(c0.z, c1.z, c2.z); g[3] = gray3(c0.w, c1.w, c2.w);
                } else { g[0] = c0.x; g[1] = c0.y; g[2] = c0.z; g[3] = c0.w; }
            };
            float t0[4], t1[4];
            zrow(pred, p0, t0); zrow(pred, p1, t1);
            vz = make_float2(0.25f * (((t0[0] + t0[1]) + t1[0]) + t1[1]), 0.25f * (((t0[2] + t0[3]) + t1[2]) + t1[3]));
            zrow(gt, p0, t0); zrow(gt, p1, t1);
            vgz = make_float2(0.25f * (((t0[0] + t0[1]) + t1[0]) + t1[1]), 0.25f * (((t0[2] + t0[3]) + t1[2]) + t1[3]));
            grow(p0, t0); grow(p1, t1);
            vg = make_float2(0.25f * (((t0[0] + t0[1]) + t1[0]) + t1[1]), 0.25f * (((t0[2] + t0[3]) + t1[2]) + t1[3]));
        }
        pz[R][2 * Cp] = vz.x; pz[R][2 * Cp + 1] = vz.y;
        pgz[R][2 * Cp] = vgz.x; pgz[R][2 * Cp + 1] = vgz.y;
        pg[R][2 * Cp] = vg.x; pg[R][2 * Cp + 1] = vg.y;
    }
    __syncthreads();
    const float inv_mx = s_inv[0], inv_my = s_inv[1];
    const bool thermal_bad = !(inv_mx > 0.f && inv_mx <= 1.0e5f && inv_my > 0.f && inv_my <= 1.0e5f);   // NaN / Inf thermal
    const float m = (view == 0) ? 0.4f : 0.5f;                   // utils/loss.py:253-256
    // ---- q_x, q_y of cells I0-1 .. I0+kT2H-1, J0-1 .. J0+kT2W-1; sums only over this tile's own cells
    Sums3 acc = {0.f, 0.f, 0.f};
    for (int k = tid; k < (kT2H + 1) * (kT2W + 1); k += kS2Threads) {
        const int r = k / (kT2W + 1), c = k - r * (kT2W + 1);
        const int I = I0 - 1 + r, J = J0 - 1 + c;
        float qx = 0.f, qy = 0.f;
        if (I >= 0 && J >= 0 && I < h2 && J < w2) {
            const int R = r, C = c + 1;                          // plane index of cell (I, J): columns start at J0 - 2
            const bool vx = J < w2 - 1, vy = I < h2 - 1;
            const float g0 = pg[R][C];
            const float tx = vx ? fabsf(pg[R][C + 1] - g0) : 0.f, ty = vy ? fabsf(pg[R + 1][C] - g0) : 0.f;
            const float w = __expf(-kThermalFactor * (min_nan(tx * inv_mx, m) + min_nan(ty * inv_my, m)));
            const bool own = (r >= 1) && (c >= 1);
            qx = q_term2(vx, pz[R][C], pz[R][C + 1], pgz[R][C], pgz[R][C + 1], w, a.kE, 2.0f * a.kS, a.kD, own, acc);
            qy = q_term2(vy, pz[R][C], pz[R + 1][C], pgz[R][C], pgz[R + 1][C], w, a.kE, 2.0f * a.kS, a.kD, own, acc);
        }
        sqx[r][c] = qx; sqy[r][c] = qy;
    }
    __syncthreads();
    // ---- gradient of the pooled cells of this tile, spread 0.25 to each of the four pixels
    if (BWD) {
        float* __restrict__ dzp = a.dzp[view] + (size_t)b * h2 * w2;
        for (int k = tid; k < kT2H * kT2W; k += kS2Threads) {
            const int r = k / kT2W + 1, c = k % kT2W + 1;
            const int I = I0 - 1 + r, J = J0 - 1 + c;
            if (I < h2 && J < w2)
                dzp[(size_t)I * w2 + J] = 0.25f * (-sqx[r][c] + sqx[r][c - 1] - sqy[r][c] + sqy[r - 1][c]);
        }
    }
    // ---- per-tile partial sums (fixed butterfly + fixed order over the warps: deterministic)
    acc.E = warp_sum(acc.E); acc.S = warp_sum(acc.S); acc.D = warp_sum(acc.D);
    if (lane == 0) { red[wrp][0] = acc.E; red[wrp][1] = acc.S; red[wrp][2] = acc.D; }
    __syncthreads();
    if (tid < 3) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < kS2Threads / 32; ++w) v += red[w][tid];
        if (tid == 0 && thermal_bad) v = __int_as_float(0x7fc00000);
        a.partials[((size_t)img * tiles + tile) * 4 + tid] = v;
    }
    if (tid == 3) a.partials[((size_t)img * tiles + tile) * 4 + 3] = 0.f;
}

}  // namespace

void t3d_scale2_tiles(int H, int W, int* tiles_x, int* tiles_y) {
    const int h2 = H >> 1, w2 = W >> 1;
    *tiles_x = (w2 + kT2W - 1) / kT2W;
    *tiles_y = (h2 + kT2H - 1) / kT2H;
}

int t3d_launch_loss_scale2(const Scale2Args& a, bool bwd, cudaStream_t st) {
    const int grid = a.B * 2 * a.tiles_x * a.tiles_y;
    if (bwd) T3D_LAUNCH("loss_scale2_kernel", st, loss_scale2_kernel<true><<<grid, kS2Threads, 0, st>>>(a));
    else T3D_LAUNCH("loss_scale2_kernel", st, loss_scale2_kernel<false><<<grid, kS2Threads, 0, st>>>(a));
    return T3D_OK;
}
