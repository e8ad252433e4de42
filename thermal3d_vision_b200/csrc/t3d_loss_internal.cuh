// t3d_loss_internal.cuh -- what the loss kernels share: the loss constants and device helpers, the persistent kernels'
// work-item queue, and the interface between t3d_loss.cu (entry points, tile kernel, basic-term kernel, second-stage
// reduction), t3d_loss_march.cu (TMA-fed warp-marching fast path) and t3d_loss_scale2.cu.
#pragma once
#include "t3d_common.cuh"
#include "t3d_bilinear.cuh"

// ------------------------------------------------------------------ constants of the loss
constexpr float kEps = 1e-5f;          // utils/loss.py:240
constexpr float kThermalFactor = 8.0f; // utils/loss.py:252
constexpr float kHuber = 0.1f;         // utils/loss.py:267
constexpr float kConfMin = 1e-5f, kConfMax = 10.0f;  // utils/loss.py:91-92
constexpr float kScale2Weight = 0.35f; // 0.7 / scale, utils/loss.py:288
constexpr int kNTerms = 8;             // width of a partial vector: basic, E1, S1, D1, E2, S2, D2, (pad)

// NaN-propagating min / max (SASS FMNMX.NAN): torch.clamp lets NaN through, fminf/fmaxf would not
__device__ __forceinline__ float min_nan(float a, float b) { float d; asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }
__device__ __forceinline__ float max_nan(float a, float b) { float d; asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }

// sgn(x) * |t-signed value|: (x > 0) ? t : (x < 0 ? -t : 0) with one compare (sgn(0) = 0 like ATen)
__device__ __forceinline__ float times_sgn(float t, float x) {
    const float r = __uint_as_float(__float_as_uint(t) ^ (__float_as_uint(x) & 0x80000000u));
    return (x != 0.f) ? r : 0.f;
}

// ------------------------------------------------------------------ work items of the persistent kernels
// loss_basic_kernel, loss_march_kernel, loss_march_rs_kernel and loss_march_ms_kernel: a work item is one image-view,
// one 128-pixel strip and one band of rows.  nbands_l bands of rows_l rows from the top of the image, then nbands_s
// bands of rows_s rows down to the last row; ALL large items of the batch are queued before the small ones (the
// fine-grained items fill the tail of the persistent grid: a warp spends ~20-30 us on a large item).  Each item writes
// one partial vector; per image-view they are band-major.
struct BandQueue {
    unsigned int* queue;           // work-item counter, zero on entry
    int rows_l, nbands_l, rows_s, nbands_s, nstrips;
    int per_image_view() const { return (nbands_l + nbands_s) * nstrips; }   // work items = partial vectors
};

struct BandItem { int b, view, strip, ra, rb, pidx; };   // sample, view, strip, rows [ra, rb), partial vector

// The warp's next work item (lane 0 pulls the ticket); false once the queue is exhausted.
__device__ __forceinline__ bool next_band_item(const BandQueue& q, int B, int H, int lane, BandItem& it) {
    const int nbands = q.nbands_l + q.nbands_s;
    const int n_large = B * 2 * q.nbands_l * q.nstrips;
    const int ntasks = B * 2 * nbands * q.nstrips;
    int task = 0;
    if (lane == 0) task = (int)atomicAdd(q.queue, 1u);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= ntasks) return false;
    const bool large = task < n_large;
    const int t1 = large ? task : task - n_large;
    const int nb = large ? q.nbands_l : q.nbands_s;
    const int s = t1 % q.nstrips;
    const int t2 = t1 / q.nstrips;
    const int k = t2 % nb;
    const int img = t2 / nb;
    it.b = img >> 1; it.view = img & 1; it.strip = s;
    it.ra = large ? k * q.rows_l : q.nbands_l * q.rows_l + k * q.rows_s;
    it.rb = large ? it.ra + q.rows_l : min(it.ra + q.rows_s, H);     // the large bands end at nbands_l * rows_l <= H
    it.pidx = (img * nbands + (large ? k : q.nbands_l + k)) * q.nstrips + s;
    return true;
}

// ------------------------------------------------------------------ kernel arguments
// What every loss kernel reads: per view the [B, H, W, 3] prediction and gt, the confidence ([B, H, W] or NULL), the
// gradient outputs (backward only; dconf NULL: none), and the constants of the basic term.
struct LossOperands {
    const float* pred[2]; const float* gt[2]; const float* conf[2];
    float* dpred[2]; float* dconf[2];
    float conf_max;                // upper clamp of the confidence: 10 (utils/loss.py:91), +inf with T3D_LOSS_CONF_MIN_ONLY
    float alpha;
    float kb;                      // grad_scale / (3 H W)
    float kc;                      // grad_scale / (H W)
};

struct MarchArgs {
    LossOperands op;               // conf_max is not read: the marching kernels clamp to kConfMax
    const float* thermal[2];
    const float* stats[2];         // per view: [B][stiles][4]
    float* partials;               // [B*2][bq.per_image_view()][kNTerms]: basic, E, S, D, 0...
    BandQueue bq;
    int B, H, W, tch, stiles;
    int replicated;                // tch == 3 and the planes of every image are bit-identical: read plane 0 only
    float kE, kS, kD;
    float kE2, kS2, kD2;           // scale-2 constants of the one-pass multi-scale kernel
    const float* dzp[2];           // multi-scale: per view [B][H/2][W/2], added to d/d(pred z) of each cell's 4 pixels (or NULL)
    int gt_h, gt_w;                // t3d_launch_loss_march_rs: size of the gt arrays (bilinearly resampled to H x W)
};

// half-resolution (scale 2) terms of the multi-scale loss as their own pass (t3d_loss_scale2.cu)
struct Scale2Args {
    const float* pred[2]; const float* gt[2]; const float* thermal[2];
    const float* stats[2];         // per view: [B][stiles][4], scale-2 sums in [2], [3]
    float* dzp[2];                 // out, per view [B][H/2][W/2] (backward only)
    float* partials;               // out [B*2][tiles_x*tiles_y][4]: E2, S2, D2, 0
    int B, H, W, tch, replicated, stiles, tiles_x, tiles_y;
    float kE, kS, kD;              // grad_scale * 0.35 * weight / (H/2 * W/2)
};
void t3d_scale2_tiles(int H, int W, int* tiles_x, int* tiles_y);
int t3d_launch_loss_scale2(const Scale2Args& a, bool bwd, cudaStream_t st);

// requires: W % 4 == 0, all pointers 16-byte aligned, tch in {1, 3}, single scale
int t3d_launch_loss_march(const MarchArgs& a, bool bwd, cudaStream_t st);
// multi-scale, full and half resolution in one pass (tch == 1 or replicated planes; H >= 4; even band heights)
int t3d_launch_loss_march_ms(const MarchArgs& a, bool bwd, cudaStream_t st);
// single scale with the gt at gt_h x gt_w, bilinearly resampled while it is staged: what t3d_launch_loss_march
// requires, plus gt_h >= H, gt_w >= W, gt_w % 4 == 0, 16-byte aligned gt.  t3d_loss_march_rs_span: the widest gt
// source segment (pixels) a strip stages; t3d_loss_march_rs_fits: whether the kernel takes that width (the widths
// it measured faster than the tile kernel at).
int t3d_loss_march_rs_span(int W, int gt_w);
bool t3d_loss_march_rs_fits(int span);
int t3d_launch_loss_march_rs(const MarchArgs& a, int span, bool bwd, cudaStream_t st);
