/* t3d.h -- C ABI of libt3d_sm100.so, the B200 (sm_100a) implementation of the
 * Thermal3D-Vision per-pixel hot path.
 *
 * The reference has no FFI: its boundary is a set of Python module-level
 * functions (SURVEY.md section 8b).  Every entry point below names the
 * reference function (file:line under /root/reference) whose arithmetic it
 * replaces; the Python host side in thermal3d_vision_b200/ keeps the
 * reference's signatures and binds these symbols with ctypes.
 *
 * Conventions (all entry points):
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *    its name ends in _host;
 *  - the caller allocates every buffer (inputs, outputs, workspace); the
 *    library never allocates, frees or retains pointers;
 *  - all work is enqueued on `stream` (a cudaStream_t passed as void*); no
 *    implicit synchronisation, no host callbacks;
 *  - returns 0 (T3D_OK) on success, a negative t3d_status otherwise;
 *    t3d_last_error() gives a thread-local message;
 *  - tensors are dense, row-major, float32 unless stated.  Pointmaps are AoS
 *    [B,H,W,3]; thermal images planar [B,C,H,W]; confidences / depths [B,H,W].
 *    The 128-bit vector path is used when W % 4 == 0 and every pointer is
 *    16-byte aligned; otherwise the same kernels run their scalar-load
 *    variant (never a CPU fallback).
 */
#ifndef T3D_H_
#define T3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    T3D_OK = 0,
    T3D_ERR_BAD_ARG = -1,     /* bad shape / null pointer / unsupported option */
    T3D_ERR_WORKSPACE = -2,   /* workspace too small */
    T3D_ERR_CUDA = -3,        /* a CUDA runtime call or kernel launch failed */
    T3D_ERR_DEVICE = -4       /* not an sm_100 device */
} t3d_status;

#define T3D_ABI_VERSION 3

/* ------------------------------------------------------------------ library */
int t3d_version(void);
const char* t3d_last_error(void);
/* SM count and compute capability of the current device. */
int t3d_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Number of kernels this library has launched from the calling process
 * (monotonic; bench.py reports the delta over the timed region). */
uint64_t t3d_launch_count(void);
/* Per-kernel device timing for roofline reports: between begin and end, every
 * launch of a kernel whose name contains `kernel_name_substr` (several
 * alternatives may be given separated by '|') is bracketed by
 * CUDA events on its launching stream (at most max_launches of them).
 * t3d_profile_end synchronises on the last event and returns the summed kernel
 * time and the number of launches timed. */
int t3d_profile_begin(const char* kernel_name_substr, int max_launches);
int t3d_profile_end(double* total_ms, int* launches);
/* After t3d_profile_begin: bracket only every every_nth-th matching launch (the two event records per
 * launch cost a few microseconds of stream time; a sample keeps the timed region close to an untimed run). */
int t3d_profile_stride(int every_nth);
/* Developer instrumentation: call BEFORE t3d_profile_end.  Start / stop times
 * (ms, relative to the first timed launch's start event) and names of the
 * launches timed since t3d_profile_begin; `names` holds cap strings of
 * name_stride bytes.  Stops further timing; t3d_profile_end then frees. */
int t3d_profile_timeline(char* names, int name_stride, double* start_ms, double* stop_ms, int cap, int* launches);

/* -------------------------------------------------------------------- loss */
/* Replaces utils/loss.py:75-98 (confidence_weighted_regression_loss) and
 * utils/loss.py:100-305 (enhanced_thermal_aware_loss) forward AND backward,
 * batched over B independent samples (the reference is called once per sample,
 * train_thermal_dustr.py:182-293; B = 1 reproduces that call).
 *
 * Layout of `out_sample` [B][8] float32:
 *   0 total  1 basic  2 edge  3 smoothness  4 detail   (unweighted components,
 *   utils/loss.py:298-303)   5 valid (1.0 iff total is finite and > 0,
 *   train_thermal_dustr.py:320)   6,7 reserved.
 * Layout of `out_batch` [8] float32:
 *   0 mean total over valid samples (train_thermal_dustr.py:359)  1..4 mean
 *   components over valid samples  5 n_valid  6 B  7 reserved.
 * `out_sample_f64` (nullable) [B][8] double: the same per-sample numbers before
 * rounding to float32.
 */
#define T3D_LOSS_OUT_STRIDE 8

/* `flags` of the loss entry points: */
#define T3D_LOSS_MULTI_SCALE 0x1   /* utils/loss.py:104,133: also evaluate the 2x2 average-pooled scale (weight 0.35) */
#define T3D_LOSS_CONF_MIN_ONLY 0x2 /* clamp the confidence from below only (>= 1e-5, no upper clamp at 10): the
                                    * "original loss calculation" of train_thermal_dustr.py:278-279,305-318, which
                                    * never goes through utils/loss.py's clamp(conf, 1e-5, 10) */
#define T3D_LOSS_STATS_TWO_SCALES 0x4 /* the caller's thermal_stats hold the half-resolution sums too ([..][2], [3];
                                    * t3d_preprocess_train_u16 with stats_scales 2): with T3D_LOSS_MULTI_SCALE they are
                                    * used instead of a statistics pass (without this flag, multi-scale ignores
                                    * thermal_stats) */
size_t t3d_loss_workspace_bytes(int B, int H, int W, int flags);

/* thermal_channels is 1 or 3 (gray = 0.299 c0 + 0.587 c1 + 0.114 c2 in fp32, utils/loss.py:119-124); 3 may be
 * OR-ed with T3D_THERMAL_REPLICATED: the caller guarantees that the three planes of every image are bit-identical
 * (what enhance_thermal_contrast always returns, utils/preprocessing.py:22-28; t3d_preprocess_train_u16 with
 * out_channels 3 produces exactly that), so the kernel reads plane 0 only and evaluates gray3(v, v, v) -- the same
 * bits, a third of the thermal traffic. */
#define T3D_THERMAL_REPLICATED 0x100

/* Fused forward + backward.  Launches: thermal statistics -> main kernel (loss partials + all gradients in one
 * pass) -> deterministic second-stage reduction.
 *  - gt1/gt2 [B,gt_h,gt_w,3]: gt_h x gt_w == H x W is a pseudo-GT at the prediction's size.  At ANOTHER
 *    resolution -- the normal case in training: 512x512 pseudo-GT (scripts/pseudo_gt.py:620) against 224x224
 *    predictions -- the reference resamples it to the prediction's size first (train_thermal_dustr.py:234-271:
 *    F.interpolate(mode='bilinear', align_corners=False) on [1,3,H,W] / [1,1,H,W] views); here the four bilinear
 *    taps are evaluated inside the loss kernel's loads (same ATen arithmetic), so the resampled pointmaps are never
 *    written or re-read.
 *  - conf1/conf2 [B,conf_h,conf_w]: conf_h x conf_w = H x W for a predicted confidence, which may take a gradient,
 *    = gt_h x gt_w for a pseudo-GT confidence, which never does.  Both NULL -> ones (utils/loss.py:85-88), and
 *    conf_h / conf_w are ignored.
 *  - thermal1/thermal2 may both be NULL (-> basic loss only, utils/loss.py:116).
 *  - thermal_stats1/2 (nullable) [B][stats_tiles][4]: partial sums of |Dx gray|, |Dy gray| of each thermal image
 *    as t3d_preprocess_train_u16 emits them; when given (and single scale, or T3D_LOSS_STATS_TWO_SCALES) the
 *    statistics pass over the thermal images is skipped.
 *  - dpred1/dpred2 both NULL -> forward only (no gradient writes; dconf1/dconf2 and grad_scale are ignored);
 *    exactly one NULL is rejected.  dconf1/dconf2 may be NULL (confidence without grad).
 *  - Gradients are those of  grad_scale * loss_b  for every sample b (pass 1/B for a batch mean);
 *    t3d_loss_rescale_invalid turns them into the gradients of the mean over VALID samples without a host sync.
 *  - main_done_event (a cudaEvent_t, nullable) is recorded on `stream` right behind the main kernel, i.e. BEFORE
 *    the small second-stage reduction: the moment the machine is free again.  A caller that overlaps consecutive
 *    steps lets the next batch's preprocessing wait for it instead of for the end of the call.  It is recorded only
 *    when the call gets that far.
 * Main kernel: the TMA-fed marching kernel where thermal is on, single scale or multi-scale with H, W >= 4, no
 * T3D_LOSS_CONF_MIN_ONLY, W % 4 == 0 and 16-byte aligned arrays, and the gt either at the prediction's size or
 * downsampled (gt_h >= H, gt_w >= W, gt_w % 4 == 0, single scale, no confidence or one at the prediction's size)
 * with a 128-pixel strip's gt source segment of at most 144 pixels (gt_w = W, e.g. 512x384 <- 512x512): that
 * kernel resamples the gt rows as it stages them (loss_march_rs_kernel), bit-identical to t3d_interp_bilinear_f32
 * followed by this call at the prediction's size.  Everything else (wider segments such as 224x224 <- 512x512,
 * where the tile kernel measured faster; upsampled gt, a gt-sized confidence, unaligned data) runs on the general
 * tile kernel.  With no thermal images (both NULL: the basic term alone, e.g. with T3D_LOSS_CONF_MIN_ONLY the plain
 * confidence-weighted loss), W % 4 == 0, 16-byte aligned arrays, the confidence absent or at the prediction's size and
 * the gt at the prediction's size or downsampled with a strip's source segment of at most 144 pixels (gt_w = W, e.g.
 * 512x384 <- 512x512), the main kernel is loss_basic_kernel, a persistent per-pixel stream whose gradients are
 * bit-identical to the tile kernel's (with a downsampled gt: to t3d_interp_bilinear_f32 followed by the same-size
 * call).  Wider segments (224x224 <- 512x512, measured faster on the tile kernel), an upsampled gt and a gt-sized
 * confidence keep the tile kernel's fused bilinear taps. */
int t3d_loss_fwd_bwd(const float* pred1, const float* pred2,
                     const float* gt1, const float* gt2, int gt_h, int gt_w,
                     const float* conf1, const float* conf2, int conf_h, int conf_w,
                     const float* thermal1, const float* thermal2, int thermal_channels,
                     const float* thermal_stats1, const float* thermal_stats2, int stats_tiles,
                     float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                     int B, int H, int W, int flags,
                     float alpha, float edge_weight, float smoothness_weight, float detail_weight,
                     float grad_scale,
                     float* out_sample, float* out_batch, double* out_sample_f64,
                     void* main_done_event,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Per-sample validity fix-up (train_thermal_dustr.py:320,359): multiplies the
 * gradients of sample b by  valid_b * B / n_valid  (read from out_sample /
 * out_batch on the device).  Every block exits immediately when all samples
 * are valid, so the common case costs one near-empty launch and no traffic. */
int t3d_loss_rescale_invalid(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                             const float* out_sample, const float* out_batch,
                             int B, int H, int W, void* stream);

/* Generic upstream gradient: grads *= *grad_output (a device scalar); no-op on
 * the device when *grad_output == 1.0f.  Used by autograd backward. */
int t3d_scale_grads(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                    const float* grad_output, int B, int H, int W, void* stream);

/* v1 loss, utils/loss.py:4-72 (thermal_aware_loss; imported but never called by the
 * reference's training loop -- kept for API completeness): basic + unpadded
 * |dz| * exp(-10 |d gray|) means; the reference evaluates that expression twice, as
 * "edge" and as "smoothness".  out_sample slot 2 == slot 3, slot 4 = 0.  dpred1/dpred2
 * NULL -> forward only. */
size_t t3d_loss_v1_workspace_bytes(int B, int H, int W);
int t3d_loss_v1_fwd_bwd(const float* pred1, const float* pred2, const float* gt1, const float* gt2,
                        const float* conf1, const float* conf2,
                        const float* thermal1, const float* thermal2, int thermal_channels,
                        float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                        int B, int H, int W,
                        float alpha, float edge_weight, float smoothness_weight, float grad_scale,
                        float* out_sample, float* out_batch, double* out_sample_f64,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ----------------------------------------------------------- preprocessing */
/* cv2.resize(src, (dst_w, dst_h)) INTER_LINEAR, OpenCV C++ path (IPP off), bit-exact
 * (SURVEY.md Appendix B).  mode 0: uint16 -> uint16, round-half-even + saturate
 * (train path, data/dataset_loader.py:242); mode 1: uint16 -> (/65535.0f) ->
 * float32 (inference path, thermal_dustr_inference.py:42-52 and
 * utils/evaluate_depth_metrics.py:179-189); mode 2: float32 -> float32.
 * src [B,src_h,src_w], dst [B,dst_h,dst_w]. */
int t3d_resize_bilinear(const void* src, void* dst, int mode, int B, int src_h, int src_w,
                        int dst_h, int dst_w, void* stream);

/* cv2.resize(..., interpolation=INTER_NEAREST) of float32 maps
 * (utils/evaluate_depth_metrics.py:320-323). */
int t3d_resize_nearest_f32(const float* src, float* dst, int B, int src_h, int src_w,
                           int dst_h, int dst_w, void* stream);

/* F.interpolate(mode='bilinear', align_corners=False) of channels-LAST float32 data
 * [B,src_h,src_w,C] -> [B,dst_h,dst_w,C] (C = 3: AoS pointmaps, C = 1: confidences), the
 * resampling train_thermal_dustr.py:234-271,465-481 applies to the pseudo-GT when its
 * size differs from the prediction's. */
int t3d_interp_bilinear_f32(const float* src, float* dst, int B, int channels_last, int src_h, int src_w,
                            int dst_h, int dst_w, void* stream);

size_t t3d_preprocess_workspace_bytes(int B, int dst_h, int dst_w);

/* Train path, batched: raw uint16 frames [B,src_h,src_w] -> cv2.resize (uint16)
 * -> float raw counts -> enhance_thermal_contrast (data/dataset_loader.py:237-249
 * + :110,118 + utils/preprocessing.py:6-30): exact 65 536-bin histogram
 * (shared-memory privatised), p2/p98 as np.percentile returns them (float64),
 * clip((x - p2) / (p98 - p2), 0, 1) in float64, one rounding to float32,
 * replicated into out_channels (1 or 3) identical planes.
 * out [B,out_channels,dst_h,dst_w] float32; hist [B,65536] uint32 (== np.bincount
 * of the resized frame); percentiles [B,2] float64.
 * grad_stats (nullable) [B][t3d_preprocess_stats_tiles()][4] float32: partial sums of
 * |Dx gray|, |Dy gray| of the OUTPUT image (utils/loss.py:184-201), produced while the
 * output is written; hand them to t3d_loss_fwd_bwd to skip its statistics pass.
 * stats_scales (1 or 2): with 2, grad_stats[..][2], [3] also receive the sums of |Dx|, |Dy| of the 2x2
 * average-pooled gray image (the multi-scale loss, utils/loss.py:133-174) where t3d_preprocess_stats_scales(dst_h,
 * dst_w) returns 2; elsewhere those slots stay 0 and the loss computes its own statistics.  Pass such statistics to
 * t3d_loss_fwd_bwd with T3D_LOSS_STATS_TWO_SCALES.
 * shared != 0 is a scheduling hint: the caller runs other kernels concurrently (another stream), so the issue-bound
 * resize kernel leaves registers on every SM for them.  Results do not depend on it.
 * phase (T3D_PHASE_*, see t3d_depth_metrics; phases other than T3D_PHASE_ALL need hist == NULL): T3D_PHASE_SAMPLE
 * launches only the window-sampling kernel (its outputs stay in `workspace`), T3D_PHASE_REST everything after it. */
int t3d_preprocess_train_u16(const uint16_t* raw, int B, int src_h, int src_w, int dst_h, int dst_w,
                             float* out, int out_channels, unsigned int* hist, double* percentiles,
                             float* grad_stats, int stats_scales, int shared,
                             void* workspace, size_t workspace_bytes, int phase, void* stream);
/* Number of statistic partials per frame written to grad_stats (0: not available for this shape). */
int t3d_preprocess_stats_tiles(int dst_h, int dst_w);
/* 2 where t3d_preprocess_train_u16 with stats_scales 2 writes the half-resolution statistics, else 1 (0: no
 * statistics for this shape). */
int t3d_preprocess_stats_scales(int dst_h, int dst_w);

/* Diagnostics of the last t3d_preprocess_train_u16 call with hist == NULL on `workspace`: the number of frames
 * whose percentile ranks fell outside the sampled value windows and were found by the exact per-frame select
 * instead (same result, slower).  Synchronises `stream`; *count_host is host memory. */
int t3d_preprocess_fallback_count(const void* workspace, int B, int dst_h, int dst_w, unsigned int* count_host,
                                  void* stream);

/* enhance_thermal_contrast on float data (utils/preprocessing.py:6-30): x is
 * [B,channels,n].  channels == 3: if np.allclose(c0,c1) and np.allclose(c0,c2)
 * the plane is c0, else the fp32 gray 0.299 c0 + 0.587 c1 + 0.114 c2 (:13-19;
 * close_flags[B] int32 receives the decision); any other channel count: the
 * whole array is one plane of channels*n values.  Percentiles are exact (sampled
 * brackets + candidate select on the monotone float keys, full radix select as
 * the fallback); out [B,out_channels,plane] float32; percentiles [B,2] float64.
 * workspace: t3d_contrast_normalize_workspace_bytes(B) bytes, 16-byte aligned. */
size_t t3d_contrast_normalize_workspace_bytes(int B);
int t3d_contrast_normalize_f32(const float* x, int B, int channels, int n, float* out, int out_channels,
                               double* percentiles, int* close_flags, void* workspace, size_t workspace_bytes,
                               void* stream);

/* close_flags[b] = np.allclose(c0, c1) and np.allclose(c0, c2) for x [B,3,n]
 * (rtol 1e-5, atol 1e-8, float32; utils/preprocessing.py:15,40). */
int t3d_channels_close(const float* x, int B, int n, int* close_flags, void* stream);

/* enhance_thermal_fixed_range arithmetic (utils/preprocessing.py:47-62), float32
 * throughout: (optional x*65535) -> clip [21800, 25000] -> (x - 21800) / 3200 over
 * n elements.  close_flag (nullable, device int): when *close_flag != 0 every
 * output plane of `plane` elements is computed from the first plane (the
 * reference collapses np.allclose channels to channel 0 and re-replicates, :39-41,67-71). */
int t3d_fixed_range_normalize(const float* x, float* y, size_t n, size_t plane, const int* close_flag,
                              int normalized, void* stream);

/* Batched enhance_thermal_fixed_range of raw uint16 frames [B,src_h,src_w], resize included, in one pass:
 * out [B,out_channels,dst_h,dst_w] float32, out_channels (1 or 3) identical planes.
 *   T3D_PATH_TRAIN:     cv2.resize to uint16 (data/dataset_loader.py:242), raw counts, then the window with
 *                       normalized=False: clip [21800, 25000] -> (x - 21800) / 3200, float32.
 *   T3D_PATH_INFERENCE: /65535.0f, float cv2.resize (thermal_dustr_inference.py:42-52), then the window with
 *                       normalized=True (x * 65535.0f first), float32.
 * Each path uses the `normalized` flag that matches the values it holds; both are bit-exact against the reference.
 * grad_stats / stats_scales: as t3d_preprocess_train_u16 writes them (same layout, same shapes), gray(v, v, v) of the
 * output for 3 planes; grad_stats must be NULL where t3d_preprocess_stats_tiles(dst_h, dst_w) == 0 or `out` is not
 * 16-byte aligned.  No workspace. */
#define T3D_PATH_TRAIN 0
#define T3D_PATH_INFERENCE 1
int t3d_preprocess_fixed_range_u16(const uint16_t* raw, int B, int src_h, int src_w, int dst_h, int dst_w, int path,
                                   float* out, int out_channels, float* grad_stats, int stats_scales, void* stream);

/* ------------------------------------------------- pointmap -> depth, metrics */
size_t t3d_depth_metrics_workspace_bytes(int B, int H, int W);

/* compute_depth_metrics (utils/metrics.py:4-69; the 3-metric variant of
 * utils/evaluate_depth_metrics.py:20-80 is a subset), batched over B images.
 * pred element (b,i) is read at pred[(b*H*W + i)*pred_stride + pred_offset]:
 * stride 3 / offset 2 evaluates the Z channel of an AoS pointmap in place
 * (pointmap -> depth, utils/metrics.py:121); stride 1 / offset 0 is a depth map.
 * gt [B,gt_h,gt_w] is nearest-resampled to (H,W) when the sizes differ
 * (utils/evaluate_depth_metrics.py:320-323).  mask (nullable) [B,H,W] uint8;
 * NULL -> gt > 0 & finite (:27).
 * out [B][8] float32: abs_rel, sq_rel, rmse, rmse_log, acc_1, acc_2, acc_3,
 * n_valid (n_valid == 0 -> NaN,NaN,NaN,NaN,0,0,0 as :34-43); out_f64 (nullable)
 * the same in double (acc_k are float64 in numpy); out_medians (nullable)
 * [B][2] = median(gt), median(pred).
 * Phases (T3D_PHASE_ALL: the whole call; also taken by t3d_preprocess_train_u16): T3D_PHASE_SAMPLE launches only
 * the sampling kernel (the value windows / brackets the streaming passes classify against), as a thin CTA shape
 * that fits beside other kernels; T3D_PHASE_REST everything after it.  A caller that knows step i+1's inputs while
 * step i is still running samples them ahead of time, off the step's critical path; results are identical to
 * T3D_PHASE_ALL.
 * `state` (t3d_depth_metrics_state_bytes(B) bytes, 16-byte aligned, nullable): where the sampling pass leaves its
 * outputs (brackets, zeroed counters) -- per step, so that the big scratch in `workspace` can be shared by steps in
 * flight; NULL = inside `workspace`.  Both phases of a step take the same workspace / state, and T3D_PHASE_REST
 * REQUIRES that T3D_PHASE_SAMPLE ran on them since their last use (it also resets the counters / window histograms
 * the streaming passes accumulate into).  The sampled windows are hints: if the data changed after it was sampled the
 * results are still exact (a rank outside its window takes the exact-select fallback), only slower. */
#define T3D_PHASE_ALL 0
#define T3D_PHASE_SAMPLE 1
#define T3D_PHASE_REST 2
size_t t3d_depth_metrics_state_bytes(int B);
int t3d_depth_metrics(const float* pred, int pred_stride, int pred_offset,
                      const float* gt, int gt_h, int gt_w, const unsigned char* mask,
                      int B, int H, int W, int median_scaling,
                      float* out, double* out_f64, float* out_medians,
                      void* workspace, size_t workspace_bytes, void* state, int phase, void* stream);

/* Dataset accumulator of utils/metrics.py:128-136 (evaluate_thermal_depth): state[0..6] += the finite
 * per-image metrics of metrics_f64 [B][8] (t3d_depth_metrics' out_f64), state[7] += B (non-finite values are
 * skipped but the image still counts).  `state` is 8 doubles on the device; all-reducing it (SUM) over ranks
 * gives the data-parallel accumulator.  Deterministic (fixed summation order). */
int t3d_metrics_accumulate(const double* metrics_f64, int B, double* state, void* stream);

/* depth = pointmap[..., 2] materialised (thermal_dustr_inference.py:133-134). */
int t3d_pointmap_to_depth(const float* pointmap, float* depth, size_t n_pixels, void* stream);

/* estimate_camera_intrinsics, estimation branch (scripts/pseudo_gt.py:151-184):
 * fx = median((u - W/2) / (X/Z)), fy = median((v - H/2) / (Y/Z)) over Z > 0.
 * depth (nullable) [B,H,W] supplies Z, else the pointmap's Z.  out_K [B][9] float64. */
int t3d_estimate_focal(const float* pointmap, const float* depth, int B, int H, int W,
                       double* out_K, void* stream);

/* EXTENSION (the reference never applies K): u = fx X/Z + cx, v = fy Y/Z + cy; uv [n][2]. */
int t3d_project_points(const float* pointmap, float fx, float fy, float cx, float cy,
                       float* uv, size_t n_pixels, void* stream);

/* ------------------------------------------------------ Sobel thermal enhancer */
/* ThermalDUSt3R.preprocess_thermal (thermal_dustr_model.py:110-142).  x [B,C,H,W] with
 * C in {1,3}; a 1-channel input is replicated to 3 (:116-117), so out is always
 * [B,3,H,W].  params = device float[2] {edge_weight, temp_scale} (:104-107);
 * local_norm = use_local_normalization (:108). */
size_t t3d_sobel_workspace_bytes(int B, int C, int H, int W);
int t3d_sobel_enhance_fwd(const float* x, const float* params, int B, int C, int H, int W, int local_norm,
                          float* out, void* workspace, size_t workspace_bytes, void* stream);
/* d(sum dout*out)/d edge_weight and /d temp_scale -> dparams float[2] (what autograd gives the
 * two nn.Parameters).  dout [B,3,H,W]. */
int t3d_sobel_enhance_bwd_params(const float* x, const float* params, const float* dout, int B, int C, int H, int W,
                                 int local_norm, float* dparams, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------- experimental fire-scene pipeline */
/* Image operators of thermal_dustr_inference_for_experiment.py:62-377 (SURVEY.md 8f row 4).  The reference builds
 * them from OpenCV / NumPy / SciPy calls; these restate the libraries' algorithms: byte / integer results are
 * bit-identical (CLAHE, Canny, histogram), float results agree to rounding (Sobel, bilateral). */
/* np.percentile(x[b], (pct_lo, pct_hi)), float64 results [B][2] (:95); workspace: t3d_contrast_normalize_workspace_bytes(B). */
int t3d_percentiles_f32(const float* x, int B, int n, double pct_lo, double pct_hi, double* percentiles,
                        void* workspace, size_t workspace_bytes, void* stream);
/* cv2.createCLAHE(clipLimit, (tiles_x, tiles_y)).apply(src) on uint8 images [B,H,W] (:108-109, :220-221). */
size_t t3d_clahe_workspace_bytes(int B, int tiles_x, int tiles_y);
int t3d_clahe_u8(const unsigned char* src, unsigned char* dst, int B, int H, int W, double clip_limit, int tiles_x, int tiles_y,
                 void* workspace, size_t workspace_bytes, void* stream);
/* cv2.Canny(src, low, high) on one uint8 image (aperture 3, L1 gradient; :135, :225).  Synchronises `stream`. */
size_t t3d_canny_workspace_bytes(int H, int W);
int t3d_canny_u8(const unsigned char* src, unsigned char* dst, int H, int W, double low_thresh, double high_thresh,
                 void* workspace, size_t workspace_bytes, void* stream);
/* cv2.Sobel(src, CV_32F, 1, 0, ksize=3) -> dx and cv2.Sobel(src, CV_32F, 0, 1, ksize=3) -> dy (:228-229). */
int t3d_sobel3_f32(const float* src, float* dx, float* dy, int H, int W, void* stream);
/* np.histogram(x, bins=100, range=(0, 1))[0] -> hist100 (uint32[100]) (:188). */
int t3d_histogram100(const float* x, size_t n, unsigned int* hist100, void* stream);
/* cv2.bilateralFilter(src, d, sigma_color, sigma_space), float32, channels LAST [H,W,channels], channels 1 or 3
 * (:273, :375); scratch2: 2 floats. */
int t3d_bilateral_f32(const float* src, float* dst, int H, int W, int channels, int d, double sigma_color, double sigma_space,
                      float* scratch2, void* stream);
/* depth_refinement_with_outlier_removal step 1 (:335-356): stats2 <- {nanmean, nanstd}; out <- depth with the 3-sigma
 * outliers replaced by the median of their 5x5 inlier neighbours (the mean when there is none); mask (nullable). */
int t3d_depth_outlier_median(const float* depth, float* out, int H, int W, float* stats2, unsigned char* mask, void* stream);
/* Per-pixel stages of preprocess_fire_scene_thermal (:62-152) and advanced_fire_scene_processing (:154-282); the host
 * side (thermal3d_vision_b200/fire.py) strings them together with the operators above. */
int t3d_fire_gray(const float* img_chw, int channels, int H, int W, float* gray, void* stream);
int t3d_fire_norm_u8(const float* gray, int H, int W, const double* percentiles2, unsigned char* base_u8, unsigned char* norm_u8, void* stream);
int t3d_fire_compose(const float* gray, int H, int W, const double* percentiles2, const unsigned char* clahe_u8,
                     const unsigned char* canny_u8, const float* noise, float* out_chw, void* stream);
int t3d_fire_adv_u8(const float* gray, int H, int W, unsigned char* inverted_u8, unsigned char* gray_u8, void* stream);
int t3d_fire_adv_compose(const float* gray, int H, int W, double fire_threshold, const unsigned char* clahe_u8,
                         const unsigned char* canny_u8, const float* noise, float* out_hwc, float* scratch, void* stream);
int t3d_hwc_to_chw_clip01(const float* hwc, int H, int W, float* chw, void* stream);

/* ------------------------------------------------------ step result packing */
/* The packed step vector: T3D_RESULT_SIZE doubles.
 *   [0] sum over VALID samples of the per-sample loss, [1..4] sums of basic/edge/smoothness/detail,
 *   [5] n_valid, [6] B (train_thermal_dustr.py:320,359);
 *   [7..13] sums of the FINITE per-image metrics abs_rel..acc_3, [14] n_images (utils/metrics.py:128-136); [15] 0;
 *   [16..23] parameter gradients riding along (data-parallel training sums parameter gradients over the ranks --
 *   DDP's gradient all-reduce; on this path the only parameters are ThermalDUSt3R's two scalars edge_weight and
 *   temp_scale, thermal_dustr_model.py:104-107: slots 16, 17), else 0.
 * This is the one vector a data-parallel job sums over its ranks per step. */
#define T3D_RESULT_SIZE 24
/* t3d_loss_rescale_invalid + the packing of that vector as ONE launch (the tail of a training step,
 * train_thermal_dustr.py:320,359-360): out_vec as above (metrics_f64 may be NULL); when some samples are invalid their
 * gradients are zeroed and the others rescaled by B / n_valid (dconf may be NULL).
 * defer_rescale != 0 (data parallel, the batch spans several ranks): only the zeroing happens here; after the
 * vector has been summed over the ranks, t3d_rescale_global multiplies this rank's gradients by
 * out_vec_global[6] / out_vec_global[5] = (samples / valid samples) of the GLOBAL batch (a no-op kernel when equal). */
int t3d_step_epilogue(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                      const float* loss_per_sample, const float* loss_batch, const double* metrics_f64,
                      int B, int H, int W, int n_images, int defer_rescale,
                      const float* param_grads, int n_param_grads, double* out_vec, void* stream);
int t3d_rescale_global(float* dpred1, float* dpred2, float* dconf1, float* dconf2, const float* loss_per_sample,
                       const double* out_vec_global, int B, int H, int W, void* stream);
/* Data-parallel variant over peer memory (one process per GPU, one NVLink / NVSwitch node; replaces the per-step
 * NCCL all-reduce of the packed vector -- SURVEY.md 8e): every rank owns a mailbox of t3d_mailbox_bytes() zero-initialised bytes
 * that its peers can address (CUDA IPC / symmetric memory); peer_mailboxes = HOST array of the `world` device
 * addresses under which THIS process sees them, in rank order.  t3d_step_epilogue_peers does what
 * t3d_step_epilogue does and also stores the rank's vector into every rank's mailbox (step = 0, 1, 2, ...);
 * t3d_mailbox_reduce waits (on the device) for the world's vectors of `step` and adds them in rank order into
 * out_vec.  Per rank, reduce(step) must be enqueued before epilogue(step + 1) -- that is what makes the two
 * alternating slots safe to reuse.
 * Validity across ranks (train_thermal_dustr.py:320,357-360 over the GLOBAL batch): the gradients carry the a-priori
 * scale 1 / (B * world); t3d_step_epilogue_peers zeroes the gradients of this rank's invalid samples, and
 * t3d_mailbox_reduce -- given the gradient buffers of that step (dpred1 != NULL) -- multiplies this rank's gradients
 * by (B * world) / n_valid_global when any sample of any rank was invalid (all blocks return at once otherwise).
 * The gradients of a data-parallel step are therefore final once its reduction has run. */
#define T3D_MAX_PEERS 16
size_t t3d_mailbox_bytes(void);
int t3d_step_epilogue_peers(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                            const float* loss_per_sample, const float* loss_batch, const double* metrics_f64,
                            int B, int H, int W, int n_images,
                            const float* param_grads, int n_param_grads, double* out_vec_local,
                            const unsigned long long* peer_mailboxes, int world, int rank,
                            unsigned long long step, void* stream);
int t3d_mailbox_reduce(const void* my_mailbox, int world, unsigned long long step, double* out_vec,
                       float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                       const float* loss_per_sample, int B, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* T3D_H_ */
