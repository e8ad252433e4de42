// t3d_metrics.cu -- pointmap -> depth and the depth-metric reductions (sm_100a).
//
// Replaces /root/reference/utils/metrics.py:4-69 (compute_depth_metrics, 7
// metrics), utils/evaluate_depth_metrics.py:20-80 (3-metric variant, a subset),
// the z-extraction `pointmap[..., 2]` (utils/metrics.py:121,
// thermal_dustr_inference.py:133-134, scripts/pseudo_gt.py:115-116), the GT
// nearest resample (utils/evaluate_depth_metrics.py:320-323) and the median
// focal estimate of scripts/pseudo_gt.py:151-184.
//
// Per image: mask = gt > 0 & finite (or the caller's mask); exact float32
// medians of gt[mask] and pred[mask] by radix select; pred *= med_gt/med_pred;
// then every per-pixel term in float32 exactly as numpy evaluates it
// (IEEE div/mul, no FMA), summed in fp64 in a fixed order (deterministic).
#include "t3d_metrics_internal.cuh"

namespace {

using namespace t3d_metrics;

constexpr int kChunkThreads = 256;

// Batched exact medians in two passes over the data (np.median, utils/metrics.py:47):
//   S  sample 4096 valid pixels per image, sort them in shared memory, and bracket the median of each
//      stream (0 = gt, 1 = pred) by two sample order statistics 7 sigma either side;
//   X  the extraction pass (the only full read of the AoS pointmap) counts the elements below the bracket
//      and collects the few percent that fall inside it;
//   M  one CTA per image selects the exact middle order statistics among the candidates (radix select in
//      shared memory).  If a bracket misses (probability ~1e-6, or degenerate data) that image falls back
//      to a full 3-pass radix select over the planar copies -- slower, same exact result.
constexpr int kSample = 4096;
constexpr int kCandCap = 32768;     // candidates per (image, stream)
constexpr int kCtaCand = 2048;      // candidates per CTA per stream staged in shared memory

struct MetricsWs {
    float* vz; float* vg;
    int* counters;          // [B][8]: n_valid, pred_nan, gt_nan, fallback, lt_g, lt_p, ncand_g, ncand_p
    unsigned int* bracket;  // [B][2 streams][2]: lo key, hi key (inclusive); lo > hi = no bracket
    unsigned int* cand;     // [B][2][kCandCap] keys
    float* scale;           // [B]
    double* partials;       // [B][chunks][kNPart]
    size_t total;
};

MetricsWs metrics_ws(void* base, int B, int n, int chunks) {
    MetricsWs w;
    size_t off = 0;
    char* p = reinterpret_cast<char*>(base);
    auto take = [&](size_t bytes) { char* r = p ? p + off : nullptr; off += t3d_align_up(bytes, 256); return r; };
    w.counters = reinterpret_cast<int*>(take((size_t)B * 8 * sizeof(int)));
    w.bracket = reinterpret_cast<unsigned int*>(take((size_t)B * 4 * sizeof(unsigned int)));
    w.vz = reinterpret_cast<float*>(take((size_t)B * n * 4));
    w.vg = reinterpret_cast<float*>(take((size_t)B * n * 4));
    w.cand = reinterpret_cast<unsigned int*>(take((size_t)B * 2 * kCandCap * sizeof(unsigned int)));
    w.scale = reinterpret_cast<float*>(take((size_t)B * 2 * sizeof(float)));
    w.partials = reinterpret_cast<double*>(take((size_t)B * chunks * kNPart * sizeof(double)));
    w.total = off;
    return w;
}

int chunks_for(int n) {
    // 16 CTAs per 512x384 image: 1.15 waves instead of 1.73 with 8 192 (DESIGN §4 experiment 7); must stay below
    // 24 576, which overflows the per-CTA candidate stage (kCtaCand)
    constexpr int kChunkPx = 12288;
    return max(1, min(96, (n + kChunkPx - 1) / kChunkPx));
}

struct PixelSrc {            // how to read (gt, pred, valid) of pixel i of image b
    const float* pred; const float* gt; const unsigned char* mask;
    int pred_stride, gt_h, gt_w, H, W, resample;
    double fx, fy;
};

__device__ __forceinline__ void read_pixel(const PixelSrc& s, const float* __restrict__ g, const float* __restrict__ p,
                                           const unsigned char* __restrict__ m, int i, float& gv, float& pv, bool& ok) {
    if (s.resample) {   // cv2 INTER_NEAREST
        const int y = i / s.W, x = i - y * s.W;
        const int sx = nearest_src(x, s.fx, s.gt_w), sy = nearest_src(y, s.fy, s.gt_h);
        gv = __ldg(g + (size_t)sy * s.gt_w + sx);
    } else {
        gv = __ldg(g + i);
    }
    pv = __ldg(p + (size_t)i * s.pred_stride);
    ok = m ? (m[i] != 0) : (gv > 0.f && isfinite(gv));     // utils/metrics.py:27
}

// ------------------------------------------------------------------ S: sample + bracket
// grid (2, B): blockIdx.x = stream (0 = gt, 1 = pred).  THREADS = 1024: one CTA fills an SM and is done after one
// exposed memory latency (the chain is waiting for it); THREADS = 256: the thin form for sampling AHEAD of time
// (T3D_PHASE_SAMPLE), few enough registers to run beside any other kernel, four latencies.  Same samples, same brackets.
template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 1024 ? 1 : 4) metrics_sample_kernel(const PixelSrc s, int pred_offset,
                                                                 unsigned int* __restrict__ bracket,
                                                                 int* __restrict__ counters) {
    __shared__ unsigned int key[kSample];
    __shared__ t3d_select::Smem sm, sm2;
    __shared__ int cnt;
    const int a = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, n = s.H * s.W;
    const float* g = s.gt + (size_t)b * s.gt_h * s.gt_w;
    const float* p = s.pred + (size_t)b * n * s.pred_stride + pred_offset;
    const unsigned char* m = s.mask ? s.mask + (size_t)b * n : nullptr;
    if (tid == 0) cnt = 0;
    if (a == 0 && tid < 8) counters[8 * b + tid] = 0;        // this image's counters for the extraction pass
    __syncthreads();
    int c = 0;
    // n >= kSample: 1024 evenly strided quads of 4 consecutive pixels (they share their cache lines: a
    // quarter of the scattered DRAM reads); smaller images: every pixel exactly once.
    // All of a thread's samples are loaded before the first one is used: ONE exposed DRAM latency.
    constexpr int kQ = 4, kRounds = kSample / (kQ * THREADS);        // kQ loads of gt and pred in flight per thread and round
#pragma unroll 1
    for (int round = 0; round < kRounds; ++round) {
        float gvs[kQ], pvs[kQ]; unsigned char mks[kQ];
#pragma unroll
        for (int q = 0; q < kQ; ++q) {
            const int k = (round * kQ + q) * THREADS + tid;
            const int i0 = (n >= kSample) ? 4 * (int)(((long long)(k >> 2) * (n >> 2)) / (kSample >> 2)) + (k & 3) : k;
            const int i = min(i0, n - 1);
            size_t gi = (size_t)i;
            if (s.resample) {   // as read_pixel
                const int y = i / s.W, x = i - y * s.W;
                const int sx = nearest_src(x, s.fx, s.gt_w), sy = nearest_src(y, s.fy, s.gt_h);
                gi = (size_t)sy * s.gt_w + sx;
            }
            gvs[q] = __ldg(g + gi);
            pvs[q] = __ldg(p + (size_t)i * s.pred_stride);
            mks[q] = m ? m[i] : (unsigned char)1;
        }
#pragma unroll
        for (int q = 0; q < kQ; ++q) {
            const int k = (round * kQ + q) * THREADS + tid;
            const int i0 = (n >= kSample) ? 4 * (int)(((long long)(k >> 2) * (n >> 2)) / (kSample >> 2)) + (k & 3) : k;
            const bool ok = (i0 < n) && (m ? (mks[q] != 0) : (gvs[q] > 0.f && isfinite(gvs[q])));     // utils/metrics.py:27
            const float v = (a == 0) ? gvs[q] : pvs[q];
            unsigned int kk = 0xffffffffu;                             // sentinel: not part of the sample
            if (ok && !isnan(v)) { kk = t3d_select::float_key(v); ++c; }
            key[k] = kk;
        }
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if ((tid & 31) == 0) atomicAdd(&cnt, c);
    __syncthreads();
    // two sample order statistics 7 sigma either side of the sample median rank, to 22 bits of the key (radix
    // select in smem: 11 + 11 bits; the pass over the top 11 bits is shared by the two ranks).  lo is rounded
    // down and hi up to the 22-bit prefix: the bracket only has to CONTAIN the median (the extraction pass counts
    // what lies below it and the select among the candidates is exact), not to be a sample statistic itself.
    const int mm = cnt;
    unsigned int lo = 1u, hi = 0u;                                 // no bracket -> fallback
    if (mm >= 64) {                                                // block-uniform
        const int d = (int)ceilf(3.5f * sqrtf((float)mm)) + 2;      // +-7 sigma: neighbouring samples are correlated
        const int mid = mm / 2, rl = mid - d, rh = mid + d;
        const bool need_lo = rl > 0, need_hi = rh < mm - 1;
        lo = 0u; hi = 0xfffffffeu;
        for (int i = tid; i < t3d_select::kBins; i += THREADS) { sm.hist[i] = 0u; sm2.hist[i] = 0u; }
        __syncthreads();
        for (int i = tid; i < kSample; i += THREADS) { const unsigned int kq = key[i]; if (kq != 0xffffffffu) atomicAdd(&sm.hist[kq >> 21], 1u); }
        __syncthreads();
        unsigned int b_lo = 0u, r_lo = 0u, b_hi = 0u, r_hi = 0u;
        if (need_lo) { t3d_select::pick_bin_t<THREADS>(sm, (unsigned)rl, 2048); b_lo = sm.sel_bin; r_lo = sm.sel_rank; __syncthreads(); }
        if (need_hi) { t3d_select::pick_bin_t<THREADS>(sm, (unsigned)rh, 2048); b_hi = sm.sel_bin; r_hi = sm.sel_rank; __syncthreads(); }
        for (int i = tid; i < t3d_select::kBins; i += THREADS) sm.hist[i] = 0u;
        __syncthreads();
        for (int i = tid; i < kSample; i += THREADS) {
            const unsigned int kq = key[i];
            if (kq == 0xffffffffu) continue;
            const unsigned int top = kq >> 21, nxt = (kq >> 10) & 2047u;
            if (need_lo && top == b_lo) atomicAdd(&sm.hist[nxt], 1u);
            if (need_hi && top == b_hi) atomicAdd(&sm2.hist[nxt], 1u);
        }
        __syncthreads();
        if (need_lo) { t3d_select::pick_bin_t<THREADS>(sm, r_lo, 2048); lo = (b_lo << 21) | (sm.sel_bin << 10); __syncthreads(); }
        if (need_hi) { t3d_select::pick_bin_t<THREADS>(sm2, r_hi, 2048); hi = (b_hi << 21) | (sm2.sel_bin << 10) | 0x3ffu; hi = min(hi, 0xfffffffeu); }
    }
    if (tid == 0) { bracket[4 * b + 2 * a] = lo; bracket[4 * b + 2 * a + 1] = hi; }
}

// The CTA's candidate stage is full (spatially coherent depth: a whole chunk inside the bracket): the thread's
// candidates of this iteration go to the stage while it lasts, the rest straight to the image's list.  Rare: kept
// out of line so that the hot loop pays one compare per thread and iteration for it.
template <int U>
__device__ __noinline__ void spill_candidates(unsigned int* __restrict__ stage, int slot, unsigned int flags, const unsigned int (&keys)[U],
                                              int* __restrict__ list_count, int* __restrict__ overflow_flag,
                                              unsigned int* __restrict__ list) {
#pragma unroll
    for (int u = 0; u < U; ++u)
        if (flags & (1u << u)) {
            if (slot < kCtaCand) stage[slot] = keys[u];
            else {
                const int g = atomicAdd(list_count, 1);
                if (g < kCandCap) list[g] = keys[u]; else atomicExch(overflow_flag, 1);
            }
            ++slot;
        }
}

// The candidates of stream a (0 = gt, 1 = pred) that a thread flagged in one iteration (bit u: keys[u]) go to the CTA
// stage from the slot the thread reserved for them on; past the stage's end they go to image b's list.
template <int U>
__device__ __forceinline__ void stage_candidates(unsigned int (&scand)[2][kCtaCand], int a, int slot, unsigned int flags,
                                                 const unsigned int (&keys)[U], int* __restrict__ counters,
                                                 unsigned int* __restrict__ cand, int b) {
    if (slot + U <= kCtaCand) {
#pragma unroll
        for (int u = 0; u < U; ++u) if (flags & (1u << u)) scand[a][slot++] = keys[u];
    } else spill_candidates<U>(scand[a], slot, flags, keys, &counters[8 * b + 6 + a], &counters[8 * b + 3], cand + ((size_t)b * 2 + a) * kCandCap);
}

// The end of an extraction CTA: the counts {n_valid, pred_nan, gt_nan (if GT_NAN), lt_g, lt_p} go to image b's counters
// with one global atomic per counter and CTA, then the staged candidates of each stream (scount[a] slots reserved)
// reserve their place in the image's list and are copied there.  The helpers here take the kernel's tid: a threadIdx.x
// read of their own would lose the range the kernel's launch bounds give it, and with it some of the kernel's code.
template <bool GT_NAN>
__device__ __forceinline__ void finish_extract_cta(int tid, int (&cnt)[5], int (&sred)[5], const int (&scount)[2], int (&sbase)[2],
                                                   const unsigned int (&scand)[2][kCtaCand], int* __restrict__ counters,
                                                   unsigned int* __restrict__ cand, int b) {
#pragma unroll
    for (int k = 0; k < 5; ++k) if (GT_NAN || k != 2) cnt[k] = __reduce_add_sync(0xffffffffu, cnt[k]);
    int* c = counters + 8 * b;
    if ((tid & 31) == 0) {                             // CTA-level first: one global atomic per counter per CTA
#pragma unroll
        for (int k = 0; k < 5; ++k) if ((GT_NAN || k != 2) && cnt[k]) atomicAdd(&sred[k], cnt[k]);
    }
    __syncthreads();
    if (tid < 5 && sred[tid]) atomicAdd(&c[tid < 3 ? tid : tid + 1], sred[tid]);
    if (tid < 2) {
        const int k = min(scount[tid], kCtaCand);        // what did not fit the stage went to the list directly (spill)
        const int base = k ? atomicAdd(&c[6 + tid], k) : 0;
        if (base + k > kCandCap) { atomicExch(&c[3], 1); sbase[tid] = -1; }      // list overflow (heavy ties) -> exact fallback
        else sbase[tid] = base;
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int base = sbase[a], k = min(scount[a], kCtaCand);
        if (base >= 0)
            for (int q = tid; q < k; q += kChunkThreads) cand[((size_t)b * 2 + a) * kCandCap + base + q] = scand[a][q];
    }
}

// The nearest-resample index tables of a fast-path CTA (H + W <= kResampleMaxDim): stab[x] = source column of column x,
// stab[W + y] = offset of the source row of row y.  Readable after the next __syncthreads.
__device__ __forceinline__ void fill_nearest_tables(int* stab, int tid, int H, int W, int gt_h, int gt_w) {
    const double fx = (double)gt_w / (double)W, fy = (double)gt_h / (double)H;
    for (int i = tid; i < W + H; i += kChunkThreads) {
        if (i < W) stab[i] = nearest_src(i, fx, gt_w);
        else stab[i] = nearest_src(i - W, fy, gt_h) * gt_w;
    }
}

// ------------------------------------------------------------------ X: extract (K5) + count + collect
// pred element (b, i) lives at pred[(b*n + i) * pred_stride + pred_offset]: stride 3 / offset 2 reads
// the Z channel of an AoS pointmap in place (depth is never materialised by the caller).
// Invalid pixels are stored as vg = NaN (a *selected* NaN GT makes every metric NaN anyway: gt_nan counter).
template <bool GENERAL>      // GENERAL: user mask and/or GT nearest-resample; else mask = gt > 0 & finite, same size
__global__ void __launch_bounds__(kChunkThreads, 6)
depth_extract_kernel(const PixelSrc s, int pred_offset, float* __restrict__ vz, float* __restrict__ vg,
                     int* __restrict__ counters, const unsigned int* __restrict__ bracket,
                     unsigned int* __restrict__ cand) {
    __shared__ unsigned int scand[2][kCtaCand];
    __shared__ int scount[2], sbase[2], sred[5];
    const int b = blockIdx.y, n = s.H * s.W, tid = threadIdx.x;
    const float* __restrict__ g = s.gt + (size_t)b * s.gt_h * s.gt_w;
    const float* __restrict__ p = s.pred + (size_t)b * n * s.pred_stride + pred_offset;
    const unsigned char* __restrict__ m = s.mask ? s.mask + (size_t)b * n : nullptr;
    float* __restrict__ oz = vz + (size_t)b * n;
    float* __restrict__ og = vg + (size_t)b * n;
    const unsigned int lo_g = bracket[4 * b], hi_g = bracket[4 * b + 1], lo_p = bracket[4 * b + 2], hi_p = bracket[4 * b + 3];
    const int pstride = s.pred_stride;
    if (tid < 2) scount[tid] = 0;
    if (tid < 5) sred[tid] = 0;
    __syncthreads();
    int nv = 0, pnan = 0, gnan = 0, lt_g = 0, lt_p = 0;
    const int per = (n + gridDim.x - 1) / gridDim.x;
    const int i_begin = blockIdx.x * per, i_end = min(i_begin + per, n);
    constexpr int U = 4;
    for (int i0 = i_begin + tid; i0 < i_end; i0 += U * kChunkThreads) {
        float gv[U], pv[U]; bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {                                      // all loads first (MLP)
            const int i = i0 + u * kChunkThreads;
            gv[u] = 0.f; pv[u] = 0.f; ok[u] = false;
            if (i < i_end) {
                if (GENERAL) read_pixel(s, g, p, m, i, gv[u], pv[u], ok[u]);
                else { gv[u] = __ldg(g + i); pv[u] = __ldg(p + i * pstride); }
            }
        }
        unsigned int kgs[U], kps[U];    // keys of this iteration; fg / fp: which are candidates
        unsigned int fg = 0, fp = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kChunkThreads;
            if (!GENERAL) ok[u] = (i < i_end) && gv[u] > 0.f && gv[u] <= 3.402823466e38f;   // gt > 0 & finite (:27)
            if (i < i_end) {
                oz[i] = pv[u];
                og[i] = ok[u] ? gv[u] : __int_as_float(0x7fc00000);
            }
            const bool gn = GENERAL && isnan(gv[u]), pn = isnan(pv[u]);
            const bool okg = ok[u] && !gn, okp = ok[u] && !pn;
            nv += ok[u]; pnan += ok[u] && pn; gnan += ok[u] && gn;
            kgs[u] = t3d_select::float_key(gv[u]); kps[u] = t3d_select::float_key(pv[u]);
            lt_g += okg && kgs[u] < lo_g; lt_p += okp && kps[u] < lo_p;
            fg |= (unsigned)(okg && kgs[u] >= lo_g && kgs[u] <= hi_g) << u;
            fp |= (unsigned)(okp && kps[u] >= lo_p && kps[u] <= hi_p) << u;
        }
        // one shared-memory atomic per thread with candidates (~1 in 4)
        if (fg) stage_candidates<U>(scand, 0, atomicAdd(&scount[0], __popc(fg)), fg, kgs, counters, cand, b);
        if (fp) stage_candidates<U>(scand, 1, atomicAdd(&scount[1], __popc(fp)), fp, kps, counters, cand, b);
    }
    int cnt[5] = {nv, pnan, gnan, lt_g, lt_p};
    finish_extract_cta<true>(tid, cnt, sred, scount, sbase, scand, counters, cand, b);
}

// Fast form of X for the common case: no caller mask, 16-byte aligned, n % 4 == 0, prediction either planar
// (PSTRIDE 1) or the Z channel of an AoS pointmap (PSTRIDE 3, offset 2), GT optionally nearest-resampled.  A thread
// takes 4 consecutive pixels: one 128-bit load of GT, one (planar) or three (AoS: all 48 bytes are fetched from DRAM
// anyway) of the prediction; the integer keys are compared as raw bits; every counter is a predicated add.
// Only the planar Z copy is written (the sum pass re-reads the caller's GT and re-derives the validity from it),
// with an L2 evict_last policy: the 4 bytes / pixel the second pass needs stay in the L2 between the two passes and
// are overwritten there by the next call -- they never travel to DRAM.  Counters / candidates as depth_extract_kernel.

template <int PSTRIDE, bool RESAMPLE>
__global__ void __launch_bounds__(kChunkThreads, 6)
depth_extract_fast_kernel(const float* __restrict__ pred, const float* __restrict__ gt, int n,
                          float* __restrict__ vz, int* __restrict__ counters,
                          const unsigned int* __restrict__ bracket, unsigned int* __restrict__ cand,
                          int H, int W, int gt_h, int gt_w) {
    __shared__ unsigned int scand[2][kCtaCand];
    __shared__ int scount[2], sbase[2], sred[5];
    __shared__ unsigned int scount2;                              // slot counters of both streams: gt low half, pred high half
    __shared__ int stab[RESAMPLE ? kResampleMaxDim : 1];          // cv2 INTER_NEAREST source column (W) / row offset (H)
    const int b = blockIdx.y, tid = threadIdx.x;
    if (RESAMPLE) fill_nearest_tables(stab, tid, H, W, gt_h, gt_w);
    const float* __restrict__ gimg = gt + (size_t)b * gt_h * gt_w;
    const float4* __restrict__ g4 = reinterpret_cast<const float4*>(gimg);
    const float4* __restrict__ p4 = reinterpret_cast<const float4*>(pred + (size_t)b * n * PSTRIDE);
    float* __restrict__ oz = vz + (size_t)b * n;
    const uint64_t keep = l2_policy_evict_last();
    const uint4 br = __ldg(reinterpret_cast<const uint4*>(bracket) + b);
    const unsigned int lo_g = br.x, w_g = br.y - br.x, lo_p = br.z, w_p = br.w - br.z;       // lo > hi (no bracket): w wraps,
    const bool has_g = br.y >= br.x, has_p = br.w >= br.z;                                    // masked by has_*
    if (tid < 2) scount[tid] = 0;
    if (tid == 2) scount2 = 0u;
    if (tid < 5) sred[tid] = 0;
    __syncthreads();
    int nv = 0, pnan = 0, lt_g = 0, lt_p = 0;
    const int nq = n >> 2, per = (nq + gridDim.x - 1) / gridDim.x;
    const int q_begin = blockIdx.x * per, q_end = min(q_begin + per, nq);
    const bool packed = per < 16384;                      // < 65 536 pixels per CTA: two 16-bit slot counters in one word
    for (int q = q_begin + tid; q < q_end; q += kChunkThreads) {
        float4 g;
        if (RESAMPLE) {                                   // W % 4 == 0: the quad lies in one row
            const int y = (4 * q) / W, x = 4 * q - y * W;
            const float* row = gimg + stab[W + y];
            // same width (only the height differs, e.g. 512x512 GT for 384x512 predictions): the column map is the
            // identity and the quad is one aligned 128-bit load of the source row (gt_w % 4 == 0 with W)
            if (gt_w == W) g = __ldg(reinterpret_cast<const float4*>(row + x));
            else g = make_float4(__ldg(row + stab[x]), __ldg(row + stab[x + 1]), __ldg(row + stab[x + 2]), __ldg(row + stab[x + 3]));
        } else {
            g = __ldg(g4 + q);
        }
        float4 z;
        if (PSTRIDE == 3) {
            const float4 a = __ldg(p4 + 3 * q), bq = __ldg(p4 + 3 * q + 1), c = __ldg(p4 + 3 * q + 2);
            z = make_float4(a.z, bq.y, c.x, c.w);
        } else {
            z = __ldg(p4 + q);
        }
        const float gv[4] = {g.x, g.y, g.z, g.w}, pv[4] = {z.x, z.y, z.z, z.w};
        unsigned int kgs[4], kps[4], fg = 0, fp = 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const unsigned int gb = __float_as_uint(gv[u]), pb = __float_as_uint(pv[u]);
            const bool ok = (gb - 1u) < 0x7f7fffffu;                     // gt > 0 & finite (utils/metrics.py:27)
            const bool pn = pv[u] != pv[u];
            const bool okp = ok && !pn;
            kgs[u] = gb | 0x80000000u;                                   // key of a positive float
            kps[u] = key_of_bits(pb);
            nv += ok; pnan += (ok && pn);
            lt_g += (ok && kgs[u] < lo_g); lt_p += (okp && kps[u] < lo_p);
            fg |= (unsigned)(ok && has_g && (kgs[u] - lo_g) <= w_g) << u;
            fp |= (unsigned)(okp && has_p && (kps[u] - lo_p) <= w_p) << u;
        }
        if (PSTRIDE == 3) stg_f4_l2hint(oz + 4 * (size_t)q, z, keep);      // planar: the caller's array IS the Z plane
        if (fg | fp) {                  // ONE shared-memory atomic per thread with candidates: both streams' slot counters in
            // one word (16 bits each when the CTA sees < 65 536 pixels, else two atomics) -- the compiler aggregates the
            // atomic over the warp with a shuffle scan, which costs as much as the rest of the iteration when done twice
            unsigned int old;
            if (packed) old = atomicAdd(&scount2, (unsigned)__popc(fg) | ((unsigned)__popc(fp) << 16));
            else {
                const unsigned int og = fg ? (unsigned)atomicAdd(&scount[0], __popc(fg)) : 0u;
                const unsigned int op = fp ? (unsigned)atomicAdd(&scount[1], __popc(fp)) : 0u;
                old = min(og, 0xffffu) | (min(op, 0xffffu) << 16);        // >= kCtaCand either way: spills
            }
            if (fg) stage_candidates<4>(scand, 0, (int)(old & 0xffffu), fg, kgs, counters, cand, b);
            if (fp) stage_candidates<4>(scand, 1, (int)(old >> 16), fp, kps, counters, cand, b);
        }
    }
    __syncthreads();
    if (packed && tid < 2) scount[tid] = (int)((scount2 >> (16 * tid)) & 0xffffu);
    int cnt[5] = {nv, pnan, 0, lt_g, lt_p};           // no NaN GT passes the validity test: gt_nan is not counted
    finish_extract_cta<false>(tid, cnt, sred, scount, sbase, scand, counters, cand, b);
}

// ------------------------------------------------------------------ M: exact medians -> scale
constexpr int kMedThreads = t3d_select::kThreads;

// grid (2, B): blockIdx.x = stream (0 = gt, 1 = pred); writes medians[b][stream]
__global__ void __launch_bounds__(kMedThreads, 1)
median_scale_kernel(const float* __restrict__ vz, const float* __restrict__ vg, const int* __restrict__ counters,
                    const unsigned int* __restrict__ cand, const unsigned int* __restrict__ bracket, int n,
                    int median_scaling, float* __restrict__ medians, const PixelSrc src, int pred_offset) {
    extern __shared__ unsigned int skeys[];                       // kCandCap keys
    __shared__ t3d_select::Smem sm;
    const int a = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
    const int* c = counters + 8 * b;
    const int nv = c[0];
    float med = 0.f;
    if (nv > 0 && median_scaling) {
        const unsigned int r0 = (unsigned)(nv - 1) / 2, r1 = (unsigned)nv / 2;
        if (c[a == 0 ? 2 : 1] > 0) med = __int_as_float(0x7fc00000);      // NaN in the stream -> median NaN
        else {
            const int lt = c[4 + a], nc = c[6 + a];
            const bool bracket_ok = (c[3] == 0) && ((int)r0 >= lt) && ((int)r1 < lt + nc) && nc <= kCandCap;
            float x0, x1;
            if (bracket_ok) {
                // candidates as offsets from the bracket's lower key (all lie in [lo, hi]): the select then runs
                // over the ~20 significant bits of the bracket width instead of 32 bits whose top 11 are shared
                const unsigned int* src = cand + ((size_t)b * 2 + a) * kCandCap;
                const unsigned int lo = bracket[4 * b + 2 * a], width = bracket[4 * b + 2 * a + 1] - lo;
                const int nbits = 32 - __clz(width | 1u);
                for (int q = tid; q < nc; q += kMedThreads) skeys[q] = src[q] - lo;
                __syncthreads();
                const unsigned int k0 = t3d_select::select_rank_offsets(sm, skeys, nc, r0 - lt, nbits);
                x0 = t3d_select::key_float(k0 + lo);
                x1 = x0;
                if (r1 != r0) {      // x_(r0+1): x0 again if it has duplicates past rank r0, else the next larger key
                    unsigned int le = 0, nxt = 0xffffffffu;
                    for (int q = tid; q < nc; q += kMedThreads) {
                        const unsigned int k = skeys[q];
                        le += k <= k0;
                        if (k > k0) nxt = min(nxt, k);
                    }
                    le = __reduce_add_sync(0xffffffffu, le); nxt = __reduce_min_sync(0xffffffffu, nxt);
                    if ((tid & 31) == 0) { sm.hist[tid >> 5] = le; sm.hist[64 + (tid >> 5)] = nxt; }
                    __syncthreads();
                    le = 0; nxt = 0xffffffffu;
                    for (int w = 0; w < kMedThreads / 32; ++w) { le += sm.hist[w]; nxt = min(nxt, sm.hist[64 + w]); }
                    __syncthreads();
                    x1 = (le > r1 - lt) ? x0 : t3d_select::key_float(nxt + lo);
                }
            } else {                                              // fallback: full radix select, same result
                if (vg) {                                         // general path: planar copies, NaN marks an unselected pixel
                    const float* v = (a == 0 ? vg : vz) + (size_t)b * n;
                    const float* gm = vg + (size_t)b * n;
                    auto get = [&](int i, float* o) { *o = v[i]; return !isnan(gm[i]); };
                    x0 = t3d_select::select_rank(sm, n, r0, get);
                    x1 = (r1 == r0) ? x0 : t3d_select::select_rank(sm, n, r1, get);
                } else {                                          // fast path: straight from the caller's arrays
                    const float* g = src.gt + (size_t)b * src.gt_h * src.gt_w;
                    const float* p = src.pred + (size_t)b * n * src.pred_stride + pred_offset;
                    auto get = [&](int i, float* o) {
                        float gv, pv; bool ok;
                        read_pixel(src, g, p, nullptr, i, gv, pv, ok);
                        *o = (a == 0) ? gv : pv;
                        return ok;
                    };
                    x0 = t3d_select::select_rank(sm, n, r0, get);
                    x1 = (r1 == r0) ? x0 : t3d_select::select_rank(sm, n, r1, get);
                }
            }
            med = (r1 == r0) ? x0 : __fmul_rn(__fadd_rn(x0, x1), 0.5f);   // np.median: fp32 mean of the middles
        }
    }
    if (tid == 0) medians[2 * b + a] = med;
}

// ------------------------------------------------------------------ M3: per-pixel terms (t3d_metrics_internal.cuh)
// The partial vector of chunk `chunk` of image b: the threads' v (four sums, three delta-counts, a pad), summed by
// warp butterflies and then over the warps in a fixed order (deterministic).
__device__ __forceinline__ void write_chunk_partials(int tid, double (&v)[kNPart], double (&red)[kChunkThreads / 32][kNPart],
                                                     double* __restrict__ partials, int b, int chunks, int chunk) {
#pragma unroll
    for (int k = 0; k < kNPart - 1; ++k) v[k] = warp_sum(v[k]);
    const int lane = tid & 31, wrp = tid >> 5;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kNPart; ++k) red[wrp][k] = v[k];
    }
    __syncthreads();
    if (tid < kNPart) {
        double t = 0;
#pragma unroll
        for (int w = 0; w < kChunkThreads / 32; ++w) t += red[w][tid];
        partials[((size_t)b * chunks + chunk) * kNPart + tid] = t;
    }
}

template <bool GENERAL>
__global__ void __launch_bounds__(kChunkThreads, 4)
metrics_sum_kernel(const float* __restrict__ vz, const float* __restrict__ vg,
                   const float* __restrict__ medians, const int* __restrict__ counters, int median_scaling,
                   int n, int chunks, double* __restrict__ partials) {
    __shared__ double red[kChunkThreads / 32][kNPart];
    const int b = blockIdx.y, chunk = blockIdx.x;
    // scale = median(gt) / median(pred)  (utils/metrics.py:47)
    const float s = (median_scaling && counters[8 * b] > 0) ? __fdiv_rn(medians[2 * b], medians[2 * b + 1]) : 1.0f;
    const float* g = vg + (size_t)b * n;
    const float* z = vz + (size_t)b * n;
    double acc[4] = {0, 0, 0, 0};
    int cnt[3] = {0, 0, 0};
    if ((n & 3) == 0) {                       // 128-bit path; fp32 runs of 8 terms folded into fp64
        const int n4 = n >> 2, per = (n4 + chunks - 1) / chunks;
        const int q0 = chunk * per, q1 = min(q0 + per, n4);
        const float4 qnan4 = make_float4(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000),
                                         __int_as_float(0x7fc00000), __int_as_float(0x7fc00000));
        for (int q = q0 + threadIdx.x; q < q1; q += 2 * kChunkThreads) {
            const int q2 = q + kChunkThreads;
            const float4 ga = __ldg(reinterpret_cast<const float4*>(g) + q);
            const float4 za = __ldg(reinterpret_cast<const float4*>(z) + q);
            float4 gb = qnan4, zb = qnan4;
            if (q2 < q1) { gb = __ldg(reinterpret_cast<const float4*>(g) + q2); zb = __ldg(reinterpret_cast<const float4*>(z) + q2); }
            const float gt[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
            float pr[8] = {za.x, za.y, za.z, za.w, zb.x, zb.y, zb.z, zb.w};
            float accf[4] = {0.f, 0.f, 0.f, 0.f};
            float lowest = 1.0f;                                                         // NaN-propagating min of the scaled predictions
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                pr[e] = __fmul_rn(pr[e], s);                                             // pred *= scale   (:48)
                const float m = (gt[e] == gt[e]) ? pr[e] : 1.0f;                         // unselected pixels do not matter
                asm("min.NaN.f32 %0, %0, %1;" : "+f"(lowest) : "f"(m));
            }
            if (!GENERAL && lowest > 0.f) {                                              // all selected predictions positive (not NaN)
#pragma unroll
                for (int e = 0; e < 8; ++e) metric_terms_fast(gt[e], pr[e], accf, cnt);
            } else {
                const float za8[8] = {za.x, za.y, za.z, za.w, zb.x, zb.y, zb.z, zb.w};
#pragma unroll 1
                for (int e = 0; e < 8; ++e) metric_terms<GENERAL>(gt[e], za8[e], s, accf, cnt);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[k] += (double)accf[k];
        }
    } else {
        const int per = (n + chunks - 1) / chunks;
        const int i0 = chunk * per, i1 = min(i0 + per, n);
        for (int i = i0 + threadIdx.x; i < i1; i += kChunkThreads) {
            float accf[4] = {0.f, 0.f, 0.f, 0.f};
            metric_terms<GENERAL>(__ldg(g + i), __ldg(z + i), s, accf, cnt);
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[k] += (double)accf[k];
        }
    }
    double v[kNPart] = {acc[0], acc[1], acc[2], acc[3], (double)cnt[0], (double)cnt[1], (double)cnt[2], 0.0};
    write_chunk_partials(threadIdx.x, v, red, partials, b, chunks, chunk);
}

// Fast form of the sum pass (pairs with depth_extract_fast_kernel): GT straight from the caller's array (nearest-
// resampled through the same index tables), validity re-derived from it, Z from the planar copy the extraction pass
// left in the L2 (or the caller's planar prediction).  Same arithmetic and summation order as metrics_sum_kernel<false>.
template <bool RESAMPLE>
__global__ void __launch_bounds__(kChunkThreads, 4)
metrics_sum_fast_kernel(const float* __restrict__ zplane, const float* __restrict__ gt,
                        const float* __restrict__ medians, const int* __restrict__ counters, int median_scaling,
                        int n, int chunks, double* __restrict__ partials, int H, int W, int gt_h, int gt_w) {
    __shared__ double red[kChunkThreads / 32][kNPart];
    __shared__ int stab[RESAMPLE ? kResampleMaxDim : 1];
    const int b = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
    if (RESAMPLE) {
        fill_nearest_tables(stab, tid, H, W, gt_h, gt_w);
        __syncthreads();
    }
    // scale = median(gt) / median(pred)  (utils/metrics.py:47)
    const float s = (median_scaling && counters[8 * b] > 0) ? __fdiv_rn(medians[2 * b], medians[2 * b + 1]) : 1.0f;
    const float* gimg = gt + (size_t)b * gt_h * gt_w;
    const float* z = zplane + (size_t)b * n;
    const uint64_t keep = l2_policy_evict_last();
    const float qnan = __int_as_float(0x7fc00000);
    auto load_g = [&](int q) {
        if (RESAMPLE) {                                   // W % 4 == 0: the quad lies in one row
            const int y = (4 * q) / W, x = 4 * q - y * W;
            const float* row = gimg + stab[W + y];
            if (gt_w == W) return __ldg(reinterpret_cast<const float4*>(row + x));         // identity column map
            return make_float4(__ldg(row + stab[x]), __ldg(row + stab[x + 1]), __ldg(row + stab[x + 2]), __ldg(row + stab[x + 3]));
        }
        return ldg_stream_f4(gimg + 4 * (size_t)q);
    };
    double acc[4] = {0, 0, 0, 0};
    int cnt[3] = {0, 0, 0};
    const int n4 = n >> 2, per = (n4 + chunks - 1) / chunks;
    const int q0 = chunk * per, q1 = min(q0 + per, n4);
    for (int q = q0 + tid; q < q1; q += 2 * kChunkThreads) {
        const int q2 = q + kChunkThreads;
        const bool two = q2 < q1;
        const float4 ga = load_g(q);
        const float4 za = ldg_f4_l2hint(z + 4 * (size_t)q, keep);
        float4 gb = make_float4(qnan, qnan, qnan, qnan), zb = gb;
        if (two) { gb = load_g(q2); zb = ldg_f4_l2hint(z + 4 * (size_t)q2, keep); }
        float gtv[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
        const float za8[8] = {za.x, za.y, za.z, za.w, zb.x, zb.y, zb.z, zb.w};
        float pr[8];
        bool ok[8];
        bool all_normal = true;        // every selected pixel: gt and scaled prediction positive, normal, finite
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            pr[e] = __fmul_rn(za8[e], s);                                            // pred *= scale   (:48)
            const unsigned int gbits = __float_as_uint(gtv[e]), pbits = __float_as_uint(pr[e]);
            ok[e] = (gbits - 1u) < 0x7f7fffffu;                                      // gt > 0 & finite (:27)
            const bool normal = ((gbits - 0x00800000u) < 0x7f000000u) && ((pbits - 0x00800000u) < 0x7f000000u);
            all_normal = all_normal && (normal || !ok[e]);
        }
        float accf[4] = {0.f, 0.f, 0.f, 0.f};
        if (all_normal) {
            float accl2 = 0.f;
            int unselected = 0;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                metric_terms_nodiv(ok[e] ? gtv[e] : 1.0f, ok[e] ? pr[e] : 1.0f, accf, accl2, cnt);
                unselected += ok[e] ? 0 : 1;
            }
            cnt[0] -= unselected; cnt[1] -= unselected; cnt[2] -= unselected;        // g = q = 1 counted as "inside"
            accf[3] = accl2 * 0.48045301391820144f;                                  // ln(2)^2
        } else {                                                                     // zero / negative / NaN / Inf / subnormal: literal formulas
#pragma unroll 1
            for (int e = 0; e < 8; ++e) metric_terms<false>(ok[e] ? gtv[e] : qnan, za8[e], s, accf, cnt);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[k] += (double)accf[k];
    }
    double v[kNPart] = {acc[0], acc[1], acc[2], acc[3], (double)cnt[0], (double)cnt[1], (double)cnt[2], 0.0};
    write_chunk_partials(tid, v, red, partials, b, chunks, chunk);
}

// ------------------------------------------------------------------ M4: finalize
// out[b] = abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n_valid  (float32 like numpy's results;
// out_f64 keeps a_k = count / n in fp64 as numpy returns them)
__global__ void __launch_bounds__(32 * kNPart) metrics_finalize_kernel(const double* __restrict__ partials, const int* __restrict__ counters,
                                        int chunks, float* __restrict__ out, double* __restrict__ out_f64) {
    // one warp per metric: lane c owns the chunks c, c + 32, ... (all loads in flight at once), fixed butterfly
    const int b = blockIdx.x, k = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double s = 0;
    for (int c = lane; c < chunks; c += 32) s += partials[((size_t)b * chunks + c) * kNPart + k];
    s = warp_sum(s);
    if (lane != 0) return;
    const int nv = counters[8 * b];
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    if (counters[8 * b + 2] > 0 && k < 4) s = qnan;                              // a selected NaN GT poisons every mean
    double r;
    if (k == 7) r = (double)nv;
    else if (nv == 0) r = (k < 4) ? qnan : 0.0;                                  // utils/metrics.py:34-43
    else if (k < 2) r = (double)(float)(s / nv);
    else if (k < 4) r = (double)sqrtf((float)(s / nv));                          // np.sqrt(np.mean(.)) in fp32
    else r = s / nv;                                                             // (thresh < t).mean() -> fp64
    out[(size_t)b * 8 + k] = (float)r;
    if (out_f64) out_f64[(size_t)b * 8 + k] = r;
}

// Dataset accumulator of utils/metrics.py:128-136: state[0..6] += finite per-image metrics, state[7] += images.
// One warp per metric, fixed lane order (deterministic).
__global__ void metrics_accumulate_kernel(const double* __restrict__ m, int B, double* __restrict__ state) {
    const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double s = 0;
    if (k < 7) for (int b = lane; b < B; b += 32) { const double v = m[(size_t)b * 8 + k]; if (isfinite(v)) s += v; }
    s = warp_sum(s);
    if (lane == 0) state[k] += (k < 7) ? s : (double)B;
}

// ------------------------------------------------------------------ intrinsics: median focal estimate
// scripts/pseudo_gt.py:151-184: fx = median((u - W/2) / (X/Z)), fy = median((v - H/2) / (Y/Z)) over Z > 0, fp32
__global__ void __launch_bounds__(t3d_select::kThreads, 1)
focal_estimate_kernel(const float* __restrict__ pointmap, const float* __restrict__ depth, int H, int W,
                      double* __restrict__ out_K) {
    __shared__ t3d_select::Smem sm;
    __shared__ int s_cnt[3];
    const int b = blockIdx.x, n = H * W;
    const float* pm = pointmap + (size_t)b * n * 3;
    const float* dz = depth ? depth + (size_t)b * n : nullptr;
    auto Z = [&](int i) { return dz ? dz[i] : pm[(size_t)i * 3 + 2]; };
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const float hw = (float)((double)W / 2.0), hh = (float)((double)H / 2.0);
    auto ratio = [&](int i, int axis) {
        const float z = Z(i);
        const float c = pm[(size_t)i * 3 + axis];
        const int y = i / W, x = i - y * W;
        // numpy: (u - W/2) is float64 (int64 - python float), X/Z float32 -> division in float64
        const double num = axis == 0 ? ((double)x - (double)W / 2.0) : ((double)y - (double)H / 2.0);
        return num / (double)__fdiv_rn(c, z);
    };
    (void)hw; (void)hh;
    // float64 medians: select on the fp32-rounded keys is not exact for fp64 data, so do a
    // 2-level refinement: this helper is a convenience, not a hot path -> simple O(passes * n) search
    // on the monotone 64-bit key, 16 bits per pass.
    double med[2];
    for (int axis = 0; axis < 2; ++axis) {
        int nv = 0, nn = 0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            if (Z(i) > 0.f) { ++nv; nn += isnan(ratio(i, axis)); }
        }
        atomicAdd(&s_cnt[0], nv); atomicAdd(&s_cnt[1], nn);
        __syncthreads();
        const int total = s_cnt[0], nans = s_cnt[1];
        __syncthreads();
        if (threadIdx.x == 0) { s_cnt[0] = 0; s_cnt[1] = 0; }
        __syncthreads();
        if (total == 0 || nans > 0) { med[axis] = __longlong_as_double(0x7ff8000000000000LL); continue; }
        auto key64 = [&](double d) {
            unsigned long long u = (unsigned long long)__double_as_longlong(d);
            return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
        };
        double vals[2];
        const unsigned int ranks[2] = {(unsigned)(total - 1) / 2, (unsigned)total / 2};
        for (int rr = 0; rr < 2; ++rr) {
            if (rr == 1 && ranks[1] == ranks[0]) { vals[1] = vals[0]; break; }
            unsigned long long prefix = 0, fixed = 0;
            unsigned int rank = ranks[rr];
            for (int pass = 0; pass < 6; ++pass) {      // 11,11,11,11,11,9 bits
                const int width = pass < 5 ? 11 : 9;
                const int sh = 64 - 11 * pass - width;
                for (int i = threadIdx.x; i < t3d_select::kBins; i += blockDim.x) sm.hist[i] = 0u;
                __syncthreads();
                for (int i = threadIdx.x; i < n; i += blockDim.x) {
                    if (Z(i) > 0.f) {
                        const unsigned long long k = key64(ratio(i, axis));
                        if ((k & fixed) == prefix) atomicAdd(&sm.hist[(k >> sh) & ((1u << width) - 1)], 1u);
                    }
                }
                __syncthreads();
                t3d_select::pick_bin(sm, rank, 1 << width);
                prefix |= (unsigned long long)sm.sel_bin << sh;
                fixed |= (unsigned long long)((1u << width) - 1) << sh;
                rank = sm.sel_rank;
                __syncthreads();
            }
            const unsigned long long u = (prefix >> 63) ? (prefix & 0x7fffffffffffffffULL) : ~prefix;
            vals[rr] = __longlong_as_double((long long)u);
        }
        med[axis] = (ranks[0] == ranks[1]) ? vals[0] : (vals[0] + vals[1]) / 2.0;   // np.median: mean of the two
    }
    if (threadIdx.x == 0) {
        double* K = out_K + (size_t)b * 9;
        K[0] = med[0]; K[1] = 0; K[2] = (double)W / 2.0;
        K[3] = 0; K[4] = med[1]; K[5] = (double)H / 2.0;
        K[6] = 0; K[7] = 0; K[8] = 1;
    }
}

// pointmap -> dense depth map (when a caller really wants the [H,W] array, e.g. np.save in inference)
__global__ void __launch_bounds__(256) pointmap_to_depth_kernel(const float* __restrict__ pm, float* __restrict__ depth, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        depth[i] = __ldg(pm + i * 3 + 2);
}

// EXTENSION (not in the reference): u = fx X/Z + cx, v = fy Y/Z + cy
__global__ void __launch_bounds__(256) project_points_kernel(const float* __restrict__ pm, float fx, float fy, float cx,
                                                             float cy, float* __restrict__ uv, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float X = pm[i * 3], Y = pm[i * 3 + 1], Z = pm[i * 3 + 2];
        uv[2 * i] = __fadd_rn(__fmul_rn(fx, __fdiv_rn(X, Z)), cx);
        uv[2 * i + 1] = __fadd_rn(__fmul_rn(fy, __fdiv_rn(Y, Z)), cy);
    }
}

// The extraction / sum kernel pair of a call; choose_metrics_path picks one.
enum class MetricsPath {
    kFastAos,       // depth_extract_fast_kernel<3> + metrics_sum_fast_kernel: the Z channel of an AoS pointmap
    kFastPlanar,    // depth_extract_fast_kernel<1> + metrics_sum_fast_kernel: a planar prediction
    kMasked,        // depth_extract_kernel<true> + metrics_sum_kernel<true>: a caller mask
    kResampled,     // depth_extract_kernel<true> + metrics_sum_kernel<false>: a GT at another size, read per pixel
    kPlain,         // depth_extract_kernel<false> + metrics_sum_kernel<false>: every other call
};
struct MetricsPathChoice { MetricsPath path; bool resample; };   // resample: the GT is nearest-resampled

// aligned: the prediction and the GT are 16-byte aligned.
MetricsPathChoice choose_metrics_path(int H, int W, int gt_h, int gt_w, bool mask, bool aligned, int pred_stride,
                                      int pred_offset) {
    const bool resample = gt_h != H || gt_w != W;
    // The fast kernels derive the validity from the GT (no caller mask), take 4 pixels per thread with 128-bit loads
    // (W % 4 == 0, so a quad lies in one row, also of the resampled GT; aligned arrays) and resample through index
    // tables in shared memory (H + W <= kResampleMaxDim).  They read an AoS pointmap's Z channel or a planar prediction.
    if (!mask && W % 4 == 0 && aligned && (!resample || H + W <= kResampleMaxDim)) {
        if (pred_stride == 3 && pred_offset == 2) return {MetricsPath::kFastAos, resample};
        if (pred_stride == 1 && pred_offset == 0) return {MetricsPath::kFastPlanar, resample};
    }
    // A caller mask may select non-positive or non-finite GT: the masked sum evaluates the literal formulas.
    if (mask) return {MetricsPath::kMasked, resample};
    return {resample ? MetricsPath::kResampled : MetricsPath::kPlain, resample};
}

}  // namespace

extern "C" {

size_t t3d_depth_metrics_workspace_bytes(int B, int H, int W) {
    if (B < 1 || H < 1 || W < 1) return 0;
    return metrics_ws(nullptr, B, H * W, chunks_for(H * W)).total;
}

size_t t3d_depth_metrics_state_bytes(int B) {
    if (B < 1) return 0;
    return (size_t)B * 12 * sizeof(int);          // [B][8] counters, [B][4] bracket keys
}

int t3d_depth_metrics(const float* pred, int pred_stride, int pred_offset,
                      const float* gt, int gt_h, int gt_w, const unsigned char* mask,
                      int B, int H, int W, int median_scaling,
                      float* out, double* out_f64, float* out_medians,
                      void* workspace, size_t workspace_bytes, void* state, int phase, void* stream) {
    T3D_REQUIRE(phase == T3D_PHASE_ALL || phase == T3D_PHASE_SAMPLE || phase == T3D_PHASE_REST, "bad phase %d", phase);
    T3D_REQUIRE(pred && gt && (out || phase == T3D_PHASE_SAMPLE) && workspace, "NULL pointer");
    T3D_REQUIRE(B >= 1 && H >= 1 && W >= 1 && gt_h >= 1 && gt_w >= 1, "bad dims");
    T3D_REQUIRE(pred_stride >= 1 && pred_offset >= 0 && pred_offset < pred_stride, "bad pred stride/offset");
    T3D_REQUIRE((double)H * W < 1.0e9, "image too large");
    const int n = H * W, chunks = chunks_for(n);
    MetricsWs w = metrics_ws(workspace, B, n, chunks);
    if (workspace_bytes < w.total) { t3d_set_error("workspace too small"); return T3D_ERR_WORKSPACE; }
    if (state) {        // the sampling pass's outputs live in the caller's per-step state instead of the (shared) workspace
        T3D_REQUIRE(t3d_aligned16(state), "state must be 16-byte aligned");
        w.counters = reinterpret_cast<int*>(state);
        w.bracket = reinterpret_cast<unsigned int*>(state) + (size_t)B * 8;
    }
    const MetricsPathChoice choice = choose_metrics_path(H, W, gt_h, gt_w, mask != nullptr,
                                                         t3d_aligned16(pred) && t3d_aligned16(gt), pred_stride, pred_offset);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    PixelSrc src;
    src.pred = pred; src.gt = gt; src.mask = mask; src.pred_stride = pred_stride;
    src.gt_h = gt_h; src.gt_w = gt_w; src.H = H; src.W = W; src.resample = choice.resample;
    src.fx = (double)gt_w / (double)W; src.fy = (double)gt_h / (double)H;
    dim3 g((unsigned)chunks, (unsigned)B);
    if (int rc = t3d_set_max_dynamic_smem<median_scale_kernel>(kCandCap * (int)sizeof(unsigned int))) return rc;
    if (phase != T3D_PHASE_REST) {
        if (median_scaling && phase == T3D_PHASE_SAMPLE)      // ahead of time, beside other kernels: the thin form
            T3D_LAUNCH("metrics_sample_kernel", st, metrics_sample_kernel<256><<<dim3(2, B), 256, 0, st>>>(src, pred_offset, w.bracket, w.counters));
        else if (median_scaling)
            T3D_LAUNCH("metrics_sample_kernel", st, metrics_sample_kernel<1024><<<dim3(2, B), 1024, 0, st>>>(src, pred_offset, w.bracket, w.counters));
        else {
            T3D_CUDA(cudaMemsetAsync(w.counters, 0, (size_t)B * 8 * sizeof(int), st));
            T3D_CUDA(cudaMemsetAsync(w.bracket, 0xff, (size_t)B * 4 * sizeof(unsigned int), st));   // empty brackets
        }
        if (phase == T3D_PHASE_SAMPLE) return T3D_OK;
    }
    float* medians = out_medians ? out_medians : w.scale;           // [B][2]: median(gt), median(pred)
    // vg = nullptr: the fast paths keep no planar GT copy, an image whose bracket missed re-reads the caller's arrays
    auto fast = [&](auto extract, const float* zplane) {
        const auto sum = choice.resample ? metrics_sum_fast_kernel<true> : metrics_sum_fast_kernel<false>;
        T3D_LAUNCH("depth_extract_fast_kernel", st, extract<<<g, kChunkThreads, 0, st>>>(
            pred, gt, n, w.vz, w.counters, w.bracket, w.cand, H, W, gt_h, gt_w));
        T3D_LAUNCH("median_scale_kernel", st, median_scale_kernel<<<dim3(2, B), kMedThreads, kCandCap * sizeof(unsigned int), st>>>(
            w.vz, nullptr, w.counters, w.cand, w.bracket, n, median_scaling, medians, src, pred_offset));
        T3D_LAUNCH("metrics_sum_fast_kernel", st, sum<<<g, kChunkThreads, 0, st>>>(
            zplane, gt, medians, w.counters, median_scaling, n, chunks, w.partials, H, W, gt_h, gt_w));
        return T3D_OK;
    };
    auto general = [&](auto extract, auto sum) {
        T3D_LAUNCH("depth_extract_kernel", st, extract<<<g, kChunkThreads, 0, st>>>(
            src, pred_offset, w.vz, w.vg, w.counters, w.bracket, w.cand));
        T3D_LAUNCH("median_scale_kernel", st, median_scale_kernel<<<dim3(2, B), kMedThreads, kCandCap * sizeof(unsigned int), st>>>(
            w.vz, w.vg, w.counters, w.cand, w.bracket, n, median_scaling, medians, src, pred_offset));
        T3D_LAUNCH("metrics_sum_kernel", st, sum<<<g, kChunkThreads, 0, st>>>(
            w.vz, w.vg, medians, w.counters, median_scaling, n, chunks, w.partials));
        return T3D_OK;
    };
    const bool rs = choice.resample;
    int rc = T3D_OK;
    switch (choice.path) {
    case MetricsPath::kFastAos:
        rc = fast(rs ? depth_extract_fast_kernel<3, true> : depth_extract_fast_kernel<3, false>, w.vz);
        break;
    case MetricsPath::kFastPlanar:                                    // a planar prediction is its own Z plane
        rc = fast(rs ? depth_extract_fast_kernel<1, true> : depth_extract_fast_kernel<1, false>, pred);
        break;
    case MetricsPath::kMasked: rc = general(depth_extract_kernel<true>, metrics_sum_kernel<true>); break;
    case MetricsPath::kResampled: rc = general(depth_extract_kernel<true>, metrics_sum_kernel<false>); break;
    case MetricsPath::kPlain: rc = general(depth_extract_kernel<false>, metrics_sum_kernel<false>); break;
    }
    if (rc) return rc;
    T3D_LAUNCH("metrics_finalize_kernel", st, metrics_finalize_kernel<<<B, 32 * kNPart, 0, st>>>(w.partials, w.counters, chunks, out, out_f64));
    return T3D_OK;
}

int t3d_metrics_accumulate(const double* metrics_f64, int B, double* state, void* stream) {
    T3D_REQUIRE(metrics_f64 && state, "NULL pointer");
    T3D_REQUIRE(B >= 1, "bad dims");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("metrics_accumulate_kernel", st, metrics_accumulate_kernel<<<1, 256, 0, st>>>(metrics_f64, B, state));
    return T3D_OK;
}

int t3d_pointmap_to_depth(const float* pointmap, float* depth, size_t n_pixels, void* stream) {
    T3D_REQUIRE(pointmap && depth, "NULL pointer");
    if (n_pixels == 0) return T3D_OK;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t blocks = (n_pixels + 255) / 256;
    const int grid = (int)(blocks < (size_t)t3d_sm_count() * 8 ? blocks : (size_t)t3d_sm_count() * 8);
    T3D_LAUNCH("pointmap_to_depth_kernel", st, pointmap_to_depth_kernel<<<grid, 256, 0, st>>>(pointmap, depth, n_pixels));
    return T3D_OK;
}

int t3d_estimate_focal(const float* pointmap, const float* depth, int B, int H, int W, double* out_K, void* stream) {
    T3D_REQUIRE(pointmap && out_K, "NULL pointer");
    T3D_REQUIRE(B >= 1 && H >= 1 && W >= 1, "bad dims");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("focal_estimate_kernel", st, focal_estimate_kernel<<<B, t3d_select::kThreads, 0, st>>>(pointmap, depth, H, W, out_K));
    return T3D_OK;
}

int t3d_project_points(const float* pointmap, float fx, float fy, float cx, float cy, float* uv, size_t n_pixels,
                       void* stream) {
    T3D_REQUIRE(pointmap && uv, "NULL pointer");
    if (n_pixels == 0) return T3D_OK;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t blocks = (n_pixels + 255) / 256;
    const int grid = (int)(blocks < (size_t)t3d_sm_count() * 8 ? blocks : (size_t)t3d_sm_count() * 8);
    T3D_LAUNCH("project_points_kernel", st, project_points_kernel<<<grid, 256, 0, st>>>(pointmap, fx, fy, cx, cy, uv, n_pixels));
    return T3D_OK;
}

}  // extern "C"
