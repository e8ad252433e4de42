// t3d_loss_internal.cuh -- interface between t3d_loss.cu (entry points, tile kernel,
// second-stage reduction) and t3d_loss_march.cu (TMA-fed warp-marching fast path).
#pragma once
#include "t3d_common.cuh"
#include "t3d_bilinear.cuh"

struct MarchArgs {
    const float* pred[2]; const float* gt[2]; const float* conf[2]; const float* thermal[2];
    float* dpred[2]; float* dconf[2];
    const float* stats[2];         // per view: [B][stiles][4]
    float* partials;               // [B*2][nbands*nstrips][8]: basic, E, S, D, 0...
    unsigned int* queue;           // work-item counter, zero on entry
    int B, H, W, tch, stiles;
    int replicated;                // tch == 3 and the planes of every image are bit-identical: read plane 0 only
    // work items: nbands_l bands of rows_l rows from the top of the image, then nbands_s bands of rows_s rows down to
    // the last row; ALL large items of the batch are queued before the small ones (the fine-grained items fill the
    // tail of the persistent grid: a warp spends ~20-30 us on a large item)
    int rows_l, nbands_l, rows_s, nbands_s, nstrips;
    float alpha, kb, kc, kE, kS, kD;
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
