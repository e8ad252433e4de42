// t3d_preprocess_bracket.cu -- p2 / p98 of the resized 16-bit frame WITHOUT a per-pixel histogram atomic.
//
// np.percentile(x, (2, 98)) (utils/preprocessing.py:22) needs four order statistics of the frame
// (ranks k and k+1 around each quantile).  The exact-histogram path of t3d_preprocess.cu pays one
// shared-memory atomic per pixel, which is what bounds it (ATOMS retires about one lane per clock per SM).
// Here:
//   S  bracket_sample_kernel: 4096 samples (1024 jittered-stride quads) of the RESIZED frame (evaluated on the fly from
//      the raw frame) -> sample order statistics 9 sigma either side of each quantile rank -> two inclusive
//      value windows [lo2, hi2], [lo98, hi98] (integers: at most kBrBins values each);
//   A  resize_march_kernel: the cv2-exact bilinear resize (data/dataset_loader.py:242), fused with the
//      classification of every output pixel: count(v < lo) per window in registers, and a histogram of only
//      the ~5 % of pixels that fall inside a window (global integer atomics into [B][2][kBrBins]);
//   P  percentile_from_brackets_kernel: one CTA per frame: prefix-scan the two small windows, pick the four
//      order statistics, np.percentile's fp64 lerp, then tabulate the frame's normalisation LUT.  If a rank
//      falls outside its window (probability ~1e-8 per frame, or adversarial data) the same CTA falls back
//      to an exact two-level radix select over the frame: slower, same bits.
// Integer counting only: bit-exact and deterministic.
#include "t3d_preprocess_internal.cuh"
#include "t3d_select.cuh"

namespace {

constexpr int kSamp = 4096;
constexpr int kBrStride = kBrSlots;          // uints per windowed histogram (window bins + the below / above slot)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst_saddr, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst_saddr), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ unsigned int lds_u16(uint32_t saddr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr));
    return v;
}

// exact u16 -> fp32 without the conversion pipe: 0x4B000000 | v is the float 2^23 + v
__device__ __forceinline__ float u16_to_float(unsigned int v) { return __fsub_rn(__uint_as_float(0x4B000000u | v), 8388608.0f); }
// round-half-even of 0 <= x < 2^22 to an integer (what cvt.rni / cv2's saturate_cast<ushort> do): x + 2^23
// has unit ulp, so the addition itself rounds; the integer sits in the low mantissa bits
__device__ __forceinline__ unsigned int round_u16(float x) {
    const unsigned int r = __float_as_uint(__fadd_rn(x, 8388608.0f)) - 0x4B000000u;
    return min(r, 65535u);
}

__device__ __forceinline__ unsigned int bilinear_u16(const uint16_t* __restrict__ s, int sw, const Tap& ty, const Tap& tx) {
    const uint16_t* r0 = s + (size_t)ty.s0 * sw;
    const uint16_t* r1 = s + (size_t)ty.s1 * sw;
    const float h0 = __fadd_rn(__fmul_rn((float)__ldg(r0 + tx.s0), tx.c0), __fmul_rn((float)__ldg(r0 + tx.s1), tx.c1));
    const float h1 = __fadd_rn(__fmul_rn((float)__ldg(r1 + tx.s0), tx.c0), __fmul_rn((float)__ldg(r1 + tx.s1), tx.c1));
    return sat_u16(__fadd_rn(__fmul_rn(h0, ty.c0), __fmul_rn(h1, ty.c1)));
}
__device__ __forceinline__ Tap tap_from_tables(const uint2 t) {
    Tap r; r.s0 = (int)(t.x & 0xffffu); r.s1 = (int)(t.x >> 16); r.c1 = __uint_as_float(t.y); r.c0 = __fsub_rn(1.0f, r.c1);
    return r;
}
__device__ __forceinline__ Tap tap_from_tables(const uint4 t) {
    Tap r; r.s0 = (int)t.x; r.s1 = (int)t.y; r.c0 = __uint_as_float(t.z); r.c1 = __uint_as_float(t.w);
    return r;
}

// One warp: bin b of a 256-bin histogram with cum(b-1) <= rank < cum(b); returns b (255 if rank is past the end)
// and the residual rank inside the bin.
__device__ __forceinline__ int warp_find256(const unsigned int* __restrict__ h, unsigned int rank, unsigned int* resid) {
    const int lane = threadIdx.x & 31;
    unsigned int c[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { c[j] = h[8 * lane + j]; sum += c[j]; }
    unsigned int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    unsigned int excl = incl - sum;
    const bool mine = rank >= excl && rank < incl;
    int bin = 255; unsigned int rr = 0;
    if (mine) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (rank >= excl && rank < excl + c[j]) { bin = 8 * lane + j; rr = rank - excl; }
            excl += c[j];
        }
    }
    const unsigned int owner = __ballot_sync(0xffffffffu, mine);
    const int src = owner ? (__ffs(owner) - 1) : 0;
    bin = __shfl_sync(0xffffffffu, bin, src); rr = __shfl_sync(0xffffffffu, rr, src);
    *resid = rr;
    return owner ? bin : 255;
}

// Exact order statistics of u16 data at up to 4 ranks by a two-level (8 + 8 bit) radix select.
// `n` items produced by key(i) -> int (negative = skip).  All 1024 threads of the CTA; results in os[0..3].
struct Select16 {
    unsigned int h256[256];
    unsigned int hlo[4][256];
    unsigned int resid[4];
    int hb[4];
    unsigned int os[4];
};
template <typename Key>
__device__ __forceinline__ void select16_x4(Select16& sm, int n, const unsigned int ranks[4], Key key) {
    const int tid = threadIdx.x, wrp = tid >> 5;
    for (int i = tid; i < 256; i += blockDim.x) { sm.h256[i] = 0u; sm.hlo[0][i] = 0u; sm.hlo[1][i] = 0u; sm.hlo[2][i] = 0u; sm.hlo[3][i] = 0u; }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) { const int v = key(i); if (v >= 0) atomicAdd(&sm.h256[v >> 8], 1u); }
    __syncthreads();
    if (wrp < 4) {
        unsigned int rr;
        const int bin = warp_find256(sm.h256, ranks[wrp], &rr);
        if ((tid & 31) == 0) { sm.hb[wrp] = bin; sm.resid[wrp] = rr; }
    }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) {
        const int v = key(i);
        if (v >= 0) {
#pragma unroll
            for (int r = 0; r < 4; ++r) if ((v >> 8) == sm.hb[r]) atomicAdd(&sm.hlo[r][v & 255], 1u);
        }
    }
    __syncthreads();
    if (wrp < 4) {
        unsigned int rr;
        const int bin = warp_find256(sm.hlo[wrp], sm.resid[wrp], &rr);
        if ((tid & 31) == 0) sm.os[wrp] = ((unsigned)sm.hb[wrp] << 8) | (unsigned)bin;
    }
    __syncthreads();
}

// ------------------------------------------------------------------ S: sample -> value windows (+ tap tables)
// bracket[b] = {lo2, hi2, lo98, hi98}: window A = [lo2, hi2] around the p2 ranks, window B = [lo98, hi98] around
// the p98 ranks.  When the two would touch or overlap (nearly constant frames) they are merged into A and B is
// empty (lo98 = 65536), so a pixel is in at most one window.  CTA 0 also publishes the resize tap tables.
// THREADS = 1024: one CTA fills an SM and is done after one exposed memory latency (the chain is waiting for it);
// THREADS = 256: the thin form for sampling AHEAD of time (T3D_PHASE_SAMPLE): few enough registers to run beside any
// other kernel, four latencies.  Same samples, same windows.
template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 1024 ? 1 : 4)
bracket_sample_kernel(const uint16_t* __restrict__ src, int sh, int sw, int dh, int dw, int same,
                      unsigned int* __restrict__ bracket, uint2* __restrict__ gxt, uint4* __restrict__ gyt,
                      unsigned int* __restrict__ brhist, int B) {
    __shared__ short key[kSamp];
    __shared__ Select16 sel;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int n = dh * dw, m = min(n, kSamp);
    const double scx = (double)sw / (double)dw, scy = (double)sh / (double)dh;
    if (!same && b == 0) {
        for (int i = tid; i < max(dw, dh); i += THREADS) {
            if (i < dw) { const Tap t = linear_tap(i, sw, scx); gxt[i] = make_uint2((unsigned)t.s0 | ((unsigned)t.s1 << 16), __float_as_uint(t.c1)); }
            if (i < dh) { const Tap t = linear_tap(i, sh, scy); gyt[i] = make_uint4((unsigned)t.s0, (unsigned)t.s1, __float_as_uint(t.c0), __float_as_uint(t.c1)); }
        }
    }
    // zero this frame's windowed histograms (and, CTA 0, the fallback counter) for the classification pass
    for (int i = tid; i < 2 * kBrStride; i += THREADS) brhist[(size_t)b * 2 * kBrStride + i] = 0u;
    if (b == 0 && tid == 0) brhist[(size_t)B * 2 * kBrStride] = 0u;
    const uint16_t* s = src + (size_t)b * sh * sw;
    // 1024 jittered-stride locations x 4 consecutive pixels: the 4 pixels share their source cache lines
    // (a quarter of the scattered DRAM reads of 4096 single pixels); a plain stride would alias with
    // column-periodic images.  Neighbours are correlated, hence the wider (9 sigma) windows below.
    // All taps of a round's samples are loaded before the first one is used: ONE exposed DRAM latency per round.
    constexpr int kQ = 4, kRounds = kSamp / (kQ * THREADS);
#pragma unroll 1
    for (int round = 0; round < kRounds; ++round) {
        Tap ty[kQ], tx[kQ];
        unsigned int raw[kQ][4];
#pragma unroll
        for (int q = 0; q < kQ; ++q) {
            const int k = min((round * kQ + q) * THREADS + tid, m - 1);
            int i = k;
            if (n > kSamp) {
                const int l = k >> 2, qstride = (n >> 2) / (kSamp >> 2);
                i = 4 * (l * qstride + (int)((((unsigned)l * 2654435761u) >> 8) % (unsigned)qstride)) + (k & 3);
            }
            if (same) {
                raw[q][0] = __ldg(s + i);
            } else {
                const int y = i / dw, x = i - y * dw;
                ty[q] = linear_tap(y, sh, scy); tx[q] = linear_tap(x, sw, scx);
                const uint16_t* r0 = s + (size_t)ty[q].s0 * sw;
                const uint16_t* r1 = s + (size_t)ty[q].s1 * sw;
                raw[q][0] = __ldg(r0 + tx[q].s0); raw[q][1] = __ldg(r0 + tx[q].s1);
                raw[q][2] = __ldg(r1 + tx[q].s0); raw[q][3] = __ldg(r1 + tx[q].s1);
            }
        }
        if (!same) {
            // make every use depend on every load, or ptxas schedules the first conversion (and its stall) between
            // the loads of consecutive samples; raw values are u16, so the fold can never equal the constant
            unsigned int fold = 0u;
#pragma unroll
            for (int q = 0; q < kQ; ++q) fold |= raw[q][0] | raw[q][1] | raw[q][2] | raw[q][3];
            if (fold == 0xffffffffu) raw[0][0] = 0u;
        }
#pragma unroll
        for (int q = 0; q < kQ; ++q) {
            const int k = (round * kQ + q) * THREADS + tid;
            unsigned int v = raw[q][0];
            if (!same) {                                         // bilinear_u16 on the loaded taps
                const float h0 = __fadd_rn(__fmul_rn((float)raw[q][0], tx[q].c0), __fmul_rn((float)raw[q][1], tx[q].c1));
                const float h1 = __fadd_rn(__fmul_rn((float)raw[q][2], tx[q].c0), __fmul_rn((float)raw[q][3], tx[q].c1));
                v = sat_u16(__fadd_rn(__fmul_rn(h0, ty[q].c0), __fmul_rn(h1, ty[q].c1)));
            }
            if (k < m) key[k] = (short)v;                        // bit pattern of the u16
        }
    }
    __syncthreads();
    // sample ranks 9 sigma either side of each quantile's rank
    // (clamped to the sample's extremes: pixels beyond them are simply counted as below / above the window)
    unsigned int ranks[4];
#pragma unroll
    for (int w = 0; w < 2; ++w) {
        const float q = w ? 0.98f : 0.02f;
        const int r = (int)(q * (float)(m - 1) + 0.5f);
        const int d = (int)ceilf(9.0f * sqrtf((float)m * q * (1.0f - q))) + 2;
        ranks[2 * w] = (unsigned)max(r - d, 0); ranks[2 * w + 1] = (unsigned)min(r + d, m - 1);
    }
    select16_x4(sel, m, ranks, [&](int i) { return (int)(unsigned short)key[i]; });
    if (tid == 0) {
        unsigned int lo2 = sel.os[0], hi2 = sel.os[1], lo98 = sel.os[2], hi98 = sel.os[3];
        if (lo98 <= hi2 + 1) { hi2 = max(hi2, hi98); lo98 = 65536u; hi98 = 65535u; }      // merged into A, B empty
        if (hi2 - lo2 + 1 > (unsigned)kBrBins) hi2 = lo2 + kBrBins - 1;                    // too wide: P falls back if it matters
        if (lo98 <= 65535u && hi98 - lo98 + 1 > (unsigned)kBrBins) hi98 = lo98 + kBrBins - 1;
        reinterpret_cast<uint4*>(bracket)[b] = make_uint4(lo2, hi2, lo98, hi98);
    }
}

// ------------------------------------------------------------------ classification of one output value
// hA: slot 0 counts v < lo2, slot 1 + (v - lo2) the window; hB = hA + kBrStride: slot v - lo98 the window,
// slot hi98 + 1 - lo98 counts v > hi98.  Pixels strictly between the windows (~94 %) cost one subtract + compare.
struct Windows { int kA, kB, capB, lo98; unsigned int mid0, midw; };

__device__ __forceinline__ Windows load_windows(const unsigned int* __restrict__ bracket, int b) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(bracket) + b);
    Windows w;
    w.kA = 1 - (int)t.x;                                  // slot of v on the A side: max(v + kA, 0)
    w.lo98 = (int)t.z;
    w.kB = kBrStride - (int)t.z;                          // slot of v on the B side: min(v + kB, capB)
    w.capB = (int)t.w + 1 + w.kB;
    w.mid0 = t.y + 1; w.midw = t.z - t.y - 1;             // mid: hi2 < v < lo98
    return w;
}
__device__ __forceinline__ bool is_mid(unsigned int v, const Windows& w) { return (v - w.mid0) < w.midw; }
__device__ __forceinline__ void count_edge(unsigned int v, const Windows& w, unsigned int* __restrict__ hA) {
    const int iv = (int)v;
    const int ia = max(iv + w.kA, 0), ib = min(iv + w.kB, w.capB);
    atomicAdd(hA + ((iv >= w.lo98) ? ib : ia), 1u);
}

// ------------------------------------------------------------------ A (general): any shape, scalar loads
template <bool RESIZE>
__global__ void __launch_bounds__(256) resize_classify_generic_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ resized,
                                                                      const uint2* __restrict__ gxt, const uint4* __restrict__ gyt,
                                                                      const unsigned int* __restrict__ bracket,
                                                                      unsigned int* __restrict__ brhist, int sh, int sw, int dh, int dw) {
    const int b = blockIdx.y, n = dh * dw;
    const Windows w = load_windows(bracket, b);
    unsigned int* hA = brhist + (size_t)b * 2 * kBrStride;
    const uint16_t* s = src + (size_t)b * sh * sw;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned int v;
        if (RESIZE) {
            const int y = i / dw, x = i - y * dw;
            v = bilinear_u16(s, sw, tap_from_tables(__ldg(gyt + y)), tap_from_tables(__ldg(gxt + x)));
            resized[(size_t)b * n + i] = (uint16_t)v;
        } else {
            v = __ldg(s + i);
        }
        if (!is_mid(v, w)) count_edge(v, w, hA);
    }
}

// ------------------------------------------------------------------ A (fast): warp-marching resize + classification
// Requirements (checked by the launcher): dw % 4 == 0, sw % 8 == 0, raw frames 16-byte aligned.
// Work is cut into "strip-rows": 128 output columns x 1 output row; the strip-rows of the whole batch are
// numbered frame-major, strip, row, and every warp of the grid takes one contiguous range (equal cost per
// strip-row -> balanced to within one row, no queue, no tail wave).  A warp marches down its rows:
//   * lane = 4 consecutive output pixels; their x taps (two offsets + weight each) live in registers;
//   * the source rows the march needs (a strictly increasing sequence) stream through a warp-private ring in
//     shared memory with cp.async, kRing - 1 rows in flight; DENSE (scale <= 2: every source row between the
//     first and the last is used) just counts rows up, otherwise the y-tap table is walked;
//   * the horizontal pass of a source row is evaluated once and kept in registers for the (up to two) output
//     rows that use it -- what cv2's row cache does; every product is rounded separately (no FMA), u16 -> fp32
//     and the final round-half-even go through the FP32 pipe (magic-number adds), not the conversion pipe.
constexpr int kRzThreads = 256;
constexpr int kRzWarps = kRzThreads / 32;
constexpr int kRzU = 8;                 // consecutive output pixels per lane
constexpr int kRzStrip = 32 * kRzU;
constexpr int kRing = 4;

// H54 -- the dataset's horizontal geometry.  640 -> 512 columns (data/dataset_loader.py:242 with the training size of
// train_thermal_dustr.py) is a 5:4 reduction: scale = 1.25 exactly, so cv2's x taps are periodic -- 4 outputs from 5
// inputs, weights {1/8, 3/8, 5/8, 7/8}, no border clamping -- and become compile-time constants: a lane's 8 output
// pixels read 10 consecutive source pixels (five 32-bit shared loads instead of sixteen 16-bit ones, no tap
// registers).  Same arithmetic, same order, same bits.  (The vertical 512 -> 384 is 4:3: its taps are not exactly
// periodic in floating point and stay in the table.)
template <int K> struct W54 { static constexpr float f = (2 * (K & 3) + 1) * 0.125f; static constexpr float c = 1.0f - f; };

__device__ __forceinline__ void hpass54(uint32_t saddr, float h[8]) {
    unsigned int w[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w[i]) : "r"(saddr + 4u * i));
    float p[10];
#pragma unroll
    for (int i = 0; i < 5; ++i) { p[2 * i] = (float)(w[i] & 0xffffu); p[2 * i + 1] = (float)(w[i] >> 16); }
    // output u reads source pixels u + u / 4 and the next one
    h[0] = __fadd_rn(__fmul_rn(p[0], W54<0>::c), __fmul_rn(p[1], W54<0>::f));
    h[1] = __fadd_rn(__fmul_rn(p[1], W54<1>::c), __fmul_rn(p[2], W54<1>::f));
    h[2] = __fadd_rn(__fmul_rn(p[2], W54<2>::c), __fmul_rn(p[3], W54<2>::f));
    h[3] = __fadd_rn(__fmul_rn(p[3], W54<3>::c), __fmul_rn(p[4], W54<3>::f));
    h[4] = __fadd_rn(__fmul_rn(p[5], W54<0>::c), __fmul_rn(p[6], W54<0>::f));
    h[5] = __fadd_rn(__fmul_rn(p[6], W54<1>::c), __fmul_rn(p[7], W54<1>::f));
    h[6] = __fadd_rn(__fmul_rn(p[7], W54<2>::c), __fmul_rn(p[8], W54<2>::f));
    h[7] = __fadd_rn(__fmul_rn(p[8], W54<3>::c), __fmul_rn(p[9], W54<3>::f));
}

// one warp: resize + classify output rows [ya, yb) of strip `strip` of frame `f`
template <bool DENSE, bool H54>
__device__ __forceinline__ void resize_march_rows(const uint16_t* __restrict__ src, uint16_t* __restrict__ resized,
                                                  const uint2* __restrict__ gxt, const uint4* __restrict__ gyt,
                                                  const unsigned int* __restrict__ bracket, unsigned int* __restrict__ brhist,
                                                  int sh, int sw, int dh, int dw, int f, int strip, int ya, int yb,
                                                  uint32_t ring, uint32_t slot_bytes, int lane, unsigned short* __restrict__ wcand) {
    const int X0 = strip * kRzStrip;
    const int x0 = X0 + kRzU * lane;
    const bool active = x0 < dw;
    // ---- x taps of this lane's 4 pixels as shared-memory byte offsets inside a ring slot
    const int xl = min(X0 + kRzStrip, dw) - 1;
    const int span0 = H54 ? (X0 >> 2) * 5 : ((int)(__ldg(gxt + X0).x & 0xffffu) & ~7);          // 8-aligned first source column
    const int span1 = H54 ? ((xl + 1) >> 2) * 5 : ((int)(__ldg(gxt + xl).x >> 16) + 1);         // one past the last source column used
    const int nvec = (span1 - span0 + 7) >> 3;                          // <= 64 16-byte chunks per source row (launcher)
    const bool copier = lane < nvec, copier2 = lane + 32 < nvec;
    // the second tap is the next source pixel; where cv2 clamps it to the same pixel (right border) its weight
    // is exactly 0, so reading the (finite) u16 after the row's last pixel instead changes nothing
    uint32_t o0[kRzU]; float fx[kRzU], cx[kRzU];
    if (!H54) {
#pragma unroll
        for (int u = 0; u < kRzU; ++u) {
            const uint2 t = __ldg(gxt + min(x0 + u, dw - 1));
            o0[u] = ring + 2u * (uint32_t)((int)(t.x & 0xffffu) - span0);
            fx[u] = __uint_as_float(t.y); cx[u] = __fsub_rn(1.0f, fx[u]);
        }
    }
    const uint32_t lane_ld = ring + 20u * lane;                         // H54: this lane's 10 source pixels inside a slot
    const Windows w = load_windows(bracket, f);
    const unsigned int mid0b = w.mid0 + 0x4B000000u;                    // is_mid on the magic-biased value
    unsigned int* hA = brhist + (size_t)f * 2 * kBrStride;
    const char* lane_src = reinterpret_cast<const char*>(src + (size_t)f * sh * sw + span0 + 8 * lane);
    const uint32_t lane_dst = ring + 16u * lane;
    const size_t src_rowb = (size_t)sw * sizeof(uint16_t);

    // ---- source-row stream: ring slot of the i-th streamed row is i % kRing
    uint32_t issue_off = 0, load_off = 0;                               // byte offsets of the next slot to fill / to read
    const uint32_t ring_bytes = kRing * slot_bytes;
    int inext = (int)__ldg(gyt + ya).x;                                 // DENSE: next source row to issue
    const int rlast = (int)__ldg(gyt + (yb - 1)).y;                     //        last source row needed
    const char* next_src = lane_src + (size_t)inext * src_rowb;         //        and where it starts for this lane
    int iy = ya, ilast = -1;                                            // !DENSE: y-tap walker
    auto issue_next = [&]() {
        int r = -1;
        if (DENSE) {
            if (inext <= rlast) {
                if (copier) cp_async16(lane_dst + issue_off, next_src);
                if (copier2) cp_async16(lane_dst + issue_off + 512u, next_src + 512);
                next_src += src_rowb; ++inext;
                issue_off += slot_bytes; if (issue_off == ring_bytes) issue_off = 0;
            }
        } else {
            while (iy < yb) {
                const uint4 t = __ldg(gyt + iy);
                if ((int)t.x > ilast) { r = (int)t.x; break; }
                if ((int)t.y > ilast) { r = (int)t.y; ++iy; break; }
                ++iy;
            }
            if (r >= 0) {
                ilast = r;
                if (copier) cp_async16(lane_dst + issue_off, lane_src + (size_t)r * src_rowb);
                if (copier2) cp_async16(lane_dst + issue_off + 512u, lane_src + (size_t)r * src_rowb + 512);
                issue_off += slot_bytes; if (issue_off == ring_bytes) issue_off = 0;
            }
        }
        cp_async_commit();                                              // possibly empty: keeps the group count in step
    };
    auto load_h = [&](float h[kRzU]) {
        cp_async_wait<kRing - 2>();
        __syncwarp();                 // the row has landed for every lane; everyone is done with the previous row
        issue_next();                 // ... whose slot is the one this issue refills
        if (H54) hpass54(lane_ld + load_off, h);
        else {
#pragma unroll
            for (int u = 0; u < kRzU; ++u) {
                const uint32_t ad = o0[u] + load_off;
                const float a = (float)lds_u16(ad), bq = (float)lds_u16(ad + 2u);
                h[u] = __fadd_rn(__fmul_rn(a, cx[u]), __fmul_rn(bq, fx[u]));
            }
        }
        load_off += slot_bytes; if (load_off == ring_bytes) load_off = 0;
    };
    __syncwarp();
#pragma unroll
    for (int p = 0; p < kRing - 1; ++p) issue_next();

    float hA_[kRzU], hB_[kRzU];
    int tagA = -1, tagB = -1;
    uint16_t* out = resized + ((size_t)f * dh + ya) * dw + x0;
    uint4 ty = __ldg(gyt + ya);
#pragma unroll 1
    for (int y = ya; y < yb; ++y, out += dw) {
        const int s0 = (int)ty.x, s1 = (int)ty.y;
        const float cy0 = __uint_as_float(ty.z), cy1 = __uint_as_float(ty.w);
        if (y + 1 < yb) ty = __ldg(gyt + y + 1);                        // next row's taps: off the critical path
        if (s0 != tagA) {
            if (s0 == tagB) {
#pragma unroll
                for (int u = 0; u < kRzU; ++u) hA_[u] = hB_[u];
            } else load_h(hA_);
            tagA = s0;
        }
        if (s1 != tagB) {
            if (s1 == tagA) {
#pragma unroll
                for (int u = 0; u < kRzU; ++u) hB_[u] = hA_[u];
            } else load_h(hB_);
            tagB = s1;
        }
        // round-half-even by the magic-number add: the float 2^23 + x has unit ulp, its low mantissa bits ARE the
        // integer.  A convex combination of u16 values cannot exceed 65535.03 (weights sum to 1 within one ulp, two
        // roundings of 2^-8 each), so cv2's saturation never binds and the low 16 bits of the float are the pixel:
        // packed straight out of the bit patterns, classified on the biased value.
        unsigned int vb[kRzU];
#pragma unroll
        for (int u = 0; u < kRzU; ++u)
            vb[u] = __float_as_uint(__fadd_rn(__fadd_rn(__fmul_rn(hA_[u], cy0), __fmul_rn(hB_[u], cy1)), 8388608.0f));
        if (active) {
            *reinterpret_cast<uint4*>(out) = make_uint4(__byte_perm(vb[0], vb[1], 0x5410), __byte_perm(vb[2], vb[3], 0x5410),
                                                        __byte_perm(vb[4], vb[5], 0x5410), __byte_perm(vb[6], vb[7], 0x5410));
        }
        // ~6 % of the pixels lie outside the mid range: instead of eight thinly populated atomic sites per row, the
        // warp compacts them into its shared-memory list (ballot + popc) and counts them with ONE site, all lanes busy
        const unsigned int lt_mask = (1u << lane) - 1u;
        int ncand = 0;
#pragma unroll
        for (int u = 0; u < kRzU; ++u) {
            const bool c = active && ((vb[u] - mid0b) >= w.midw);
            const unsigned int bal = __ballot_sync(0xffffffffu, c);
            if (c) wcand[ncand + __popc(bal & lt_mask)] = (unsigned short)vb[u];     // low 16 bits: the pixel
            ncand += __popc(bal);
        }
        __syncwarp();
        for (int k = lane; k < ncand; k += 32) count_edge((unsigned int)wcand[k], w, hA);
        __syncwarp();
    }
    cp_async_wait<0>();
}

template <bool DENSE, bool H54>
__global__ void __launch_bounds__(kRzThreads, 3)
resize_march_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ resized,
                    const uint2* __restrict__ gxt, const uint4* __restrict__ gyt,
                    const unsigned int* __restrict__ bracket, unsigned int* __restrict__ brhist,
                    int B, int sh, int sw, int dh, int dw, int nstrips, int slot_bytes /* multiple of 16 */) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    __shared__ unsigned short s_cand[kRzWarps][kRzStrip];             // per warp: the row's pixels outside the mid range
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const uint32_t ring = smem_u32(rz_smem) + (uint32_t)(wrp * kRing * slot_bytes);
    // strip-rows [L, L1) of this warp (total < 2^31 / warps: checked by the launcher)
    const unsigned int total = (unsigned)B * nstrips * dh;
    const unsigned int gw = blockIdx.x * kRzWarps + wrp, nw = gridDim.x * kRzWarps;
    unsigned int L = (unsigned int)((unsigned long long)gw * total / nw);
    const unsigned int L1 = (unsigned int)((unsigned long long)(gw + 1) * total / nw);
    while (L < L1) {
        const unsigned int col = L / (unsigned)dh;
        const int ya = (int)(L - col * dh);
        const int yb = (int)min((unsigned)dh, ya + (L1 - L));
        L += yb - ya;
        const int f = (int)(col / (unsigned)nstrips), strip = (int)(col - f * nstrips);
        resize_march_rows<DENSE, H54>(src, resized, gxt, gyt, bracket, brhist, sh, sw, dh, dw, f, strip, ya, yb,
                                 ring, (uint32_t)slot_bytes, lane, s_cand[wrp]);
    }
}

// ------------------------------------------------------------------ P: order statistics -> percentiles -> LUT
__global__ void __launch_bounds__(1024, 1)
percentile_from_brackets_kernel(const uint16_t* __restrict__ frames, int n, const unsigned int* __restrict__ bracket,
                                const unsigned int* __restrict__ brhist, int rep3, double* __restrict__ out_p,
                                float2* __restrict__ glut, int2* __restrict__ lutmeta, unsigned int* __restrict__ n_fallback) {
    __shared__ unsigned int warp_tot[33];
    __shared__ int found[4];
    __shared__ Select16 sel;
    __shared__ double s_p[2];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    unsigned int k[2]; double g[2];
    percentile_ranks(n, 2.0, &k[0], &g[0]);
    percentile_ranks(n, 98.0, &k[1], &g[1]);
    const unsigned int ranks[4] = {k[0], min(k[0] + 1, (unsigned)n - 1), k[1], min(k[1] + 1, (unsigned)n - 1)};
    if (tid < 4) found[tid] = -1;
    __syncthreads();
    static_assert(kBrBins == 2048, "two bins per thread");
    const uint4 br = reinterpret_cast<const uint4*>(bracket)[b];
    for (int w = 0; w < 2; ++w) {
        const unsigned int lo = w ? br.z : br.x, hi = w ? br.w : br.y;
        const int nb = (lo <= 65535u && hi >= lo) ? (int)(hi - lo + 1) : 0;
        const unsigned int* h = brhist + ((size_t)b * 2 + w) * kBrStride + (w ? 0 : 1);     // first window bin
        const unsigned int c0 = (2 * tid < nb) ? h[2 * tid] : 0u, c1 = (2 * tid + 1 < nb) ? h[2 * tid + 1] : 0u;
        const unsigned int sum = c0 + c1;
        unsigned int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[wrp] = incl;
        __syncthreads();
        if (wrp == 0) {
            unsigned int x = warp_tot[lane], xi = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int t = __shfl_up_sync(0xffffffffu, xi, o);
                if (lane >= o) xi += t;
            }
            warp_tot[lane] = xi - x;
            if (lane == 31) warp_tot[32] = xi;                  // pixels inside the window
        }
        __syncthreads();
        // pixels below the window: counted directly (A) or n - inside - above (B)
        const unsigned int below = w ? ((unsigned)n - warp_tot[32] - h[nb]) : h[-1];
        const unsigned int excl = below + warp_tot[wrp] + incl - sum;
        if (nb > 0) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                if (ranks[r] >= excl && ranks[r] < excl + c0) found[r] = (int)lo + 2 * tid;
                else if (ranks[r] >= excl + c0 && ranks[r] < excl + sum) found[r] = (int)lo + 2 * tid + 1;
            }
        }
        __syncthreads();
    }
    if (found[0] < 0 || found[1] < 0 || found[2] < 0 || found[3] < 0) {
        // a rank fell outside the windows: exact two-level radix select over the frame (block-uniform branch)
        const uint16_t* x = frames + (size_t)b * n;
        if (tid == 0) atomicAdd(n_fallback, 1u);
        select16_x4(sel, n, ranks, [&](int i) { return (int)__ldg(x + i); });
        if (tid < 4) found[tid] = (int)sel.os[tid];
        __syncthreads();
    }
    if (tid == 0) {
        s_p[0] = lerp_percentile((float)found[0], (float)found[1], g[0]);
        s_p[1] = lerp_percentile((float)found[2], (float)found[3], g[1]);
        out_p[2 * b] = s_p[0]; out_p[2 * b + 1] = s_p[1];
    }
    __syncthreads();
    build_norm_lut(b, s_p[0], s_p[1], rep3, glut, lutmeta);
}

}  // namespace

int t3d_launch_bracket_percentiles(const uint16_t* raw, int B, int sh, int sw, int dh, int dw, bool same,
                                   const PreWs& w, int rep3, double* percentiles, bool shared, int phase, cudaStream_t st) {
    const int n = dh * dw;
    if (phase == T3D_PHASE_SAMPLE) {            // ahead of time, beside other kernels: the thin form
        T3D_LAUNCH("bracket_sample_kernel", st, bracket_sample_kernel<256><<<B, 256, 0, st>>>(
            raw, sh, sw, dh, dw, same ? 1 : 0, w.bracket, w.gxt, w.gyt, w.brhist, B));
        return T3D_OK;
    }
    if (phase != T3D_PHASE_REST)
        T3D_LAUNCH("bracket_sample_kernel", st, bracket_sample_kernel<1024><<<B, 1024, 0, st>>>(
            raw, sh, sw, dh, dw, same ? 1 : 0, w.bracket, w.gxt, w.gyt, w.brhist, B));
    const bool fast = !same && (dw % 8 == 0) && (sw % 8 == 0) && t3d_aligned16(raw);
    bool launched = false;
    if (fast) {
        const int nstrips = (dw + kRzStrip - 1) / kRzStrip;
        // widest source span of a strip (+ alignment slack), from the resize ratio
        const double scale = (double)sw / (double)dw;
        int slot_px = (int)(kRzStrip * scale) + 24;
        slot_px = min((slot_px + 7) & ~7, ((sw + 7) & ~7) + 8);    // + 8: the pixel after the row's last one is read (weight 0)
        const int slot_bytes = slot_px * (int)sizeof(uint16_t);
        const size_t smem = (size_t)kRzWarps * kRing * slot_bytes;
        const bool dense = sh <= 2 * dh;
        if (smem <= 96 * 1024 && slot_px <= 512 && (long long)B * nstrips * dh < (1ll << 31)) {
            static int max_ctas_dev[kT3dMaxDevices][3] = {};
            static size_t attr_smem_dev[kT3dMaxDevices][3] = {};
            const int slot = t3d_device_slot();
            int* max_ctas = max_ctas_dev[slot];
            size_t* attr_smem = attr_smem_dev[slot];
            // the dataset's 5:4 horizontal geometry: compile-time x taps (dense only: 5:4 implies scale < 2)
            const bool h54 = dense && sw * 4 == dw * 5 && (dw & 31) == 0;
            const int di = h54 ? 2 : (dense ? 1 : 0);
            const void* fn = h54 ? (const void*)resize_march_kernel<true, true> :
                             dense ? (const void*)resize_march_kernel<true, false> : (const void*)resize_march_kernel<false, false>;
            if (smem > attr_smem[di] || max_ctas[di] == 0) {
                T3D_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                attr_smem[di] = smem;
                T3D_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_ctas[di], fn, kRzThreads, smem));
                if (max_ctas[di] < 1) max_ctas[di] = 1;
            }
            // Shared machine (`shared`: the caller runs other kernels concurrently, as
            // pipeline.HotPathStep does with the metric pipeline): 2 of the 3 CTAs per SM that fit -- the registers
            // left over let the memory-bound kernels of the other stream co-reside with this issue-bound one
            // (436.6 -> 432.9 us per step); alone, 3 CTAs per SM are faster (56.7 vs 65.8 us).
            const int ctas = min(max_ctas[di], shared ? 2 : max_ctas[di]);
            const long long total = (long long)B * nstrips * dh;
            long long grid = (long long)t3d_sm_count() * ctas;
            if (grid * kRzWarps > total) grid = (total + kRzWarps - 1) / kRzWarps;
            if (h54)
                T3D_LAUNCH("resize_march_kernel", st, (resize_march_kernel<true, true><<<(unsigned)grid, kRzThreads, smem, st>>>(
                    raw, w.resized, w.gxt, w.gyt, w.bracket, w.brhist, B, sh, sw, dh, dw, nstrips, slot_bytes)));
            else if (dense)
                T3D_LAUNCH("resize_march_kernel", st, (resize_march_kernel<true, false><<<(unsigned)grid, kRzThreads, smem, st>>>(
                    raw, w.resized, w.gxt, w.gyt, w.bracket, w.brhist, B, sh, sw, dh, dw, nstrips, slot_bytes)));
            else
                T3D_LAUNCH("resize_march_kernel", st, (resize_march_kernel<false, false><<<(unsigned)grid, kRzThreads, smem, st>>>(
                    raw, w.resized, w.gxt, w.gyt, w.bracket, w.brhist, B, sh, sw, dh, dw, nstrips, slot_bytes)));
            launched = true;
        }
    }
    if (!launched) {
        dim3 grid((unsigned)max(1, min((n + 255) / 256, 4 * t3d_sm_count() / max(B, 1) + 1)), (unsigned)B);
        if (same) T3D_LAUNCH("resize_classify_generic_kernel", st, resize_classify_generic_kernel<false><<<grid, 256, 0, st>>>(
            raw, w.resized, w.gxt, w.gyt, w.bracket, w.brhist, sh, sw, dh, dw));
        else T3D_LAUNCH("resize_classify_generic_kernel", st, resize_classify_generic_kernel<true><<<grid, 256, 0, st>>>(
            raw, w.resized, w.gxt, w.gyt, w.bracket, w.brhist, sh, sw, dh, dw));
    }
    T3D_LAUNCH("percentile_from_brackets_kernel", st, percentile_from_brackets_kernel<<<B, 1024, 0, st>>>(
        same ? raw : w.resized, n, w.bracket, w.brhist, rep3, percentiles, w.lut, w.lutmeta, w.brhist + (size_t)B * 2 * kBrStride));
    return T3D_OK;
}
