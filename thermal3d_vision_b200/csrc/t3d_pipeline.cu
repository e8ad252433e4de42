// t3d_pipeline.cu -- packs the per-step scalars of the hot path into the one
// small vector that is all-reduced across ranks (SURVEY.md section 8e):
// training [sum valid loss, sum basic, edge, smooth, detail, n_valid, B] as
// train_thermal_dustr.py:320,359 accumulates them, evaluation [7 metric sums,
// n_images] as utils/metrics.py:128-136 does (non-finite metrics skipped but
// the image still counted).
#include "t3d_common.cuh"

namespace {

// pack + the validity fix-up of the loss gradients (scale_grads_kernel<0> of t3d_loss.cu) as ONE launch: block 0
// packs, every block then checks the batch's valid count and returns at once when all samples are valid.
// Peer-memory exchange of the packed vector (one process per GPU on one NVLink / NVSwitch node): every rank owns a
// mailbox  { double slots[2][T3D_MAX_PEERS][T3D_RESULT_SIZE]; unsigned long long flags[2][T3D_MAX_PEERS]; }  in memory its peers
// can address (CUDA IPC / symmetric memory).  Step s uses parity p = s & 1: rank r's epilogue stores its doubles
// into slot [p][r] of EVERY rank's mailbox (128-byte peer stores), fences, then publishes flags[p][r] = s + 1 with
// release semantics; mailbox_reduce_kernel on each rank waits for the world's flags and adds the slots in rank order
// (the same bits on every rank).  No NCCL call and no host work per step beyond the two launches.
// Slot reuse: a rank runs reduce(s) before its epilogue(s + 1) in stream order, so by the time a peer may write
// step s + 2 into parity p (after its own reduce(s + 1), which needed this rank's epilogue(s + 1)) the step-s slots
// have been read here.
constexpr int kMaxPeers = T3D_MAX_PEERS;
constexpr int kVec = T3D_RESULT_SIZE;      // doubles in the packed step vector
struct Mailbox { double slots[2][kMaxPeers][kVec]; unsigned long long flags[2][kMaxPeers]; };
static_assert(kVec <= 32 && kVec >= 16 && kMaxPeers <= kVec, "one warp handles the vector and the flags");
struct PeerArgs { Mailbox* box[kMaxPeers]; int world, rank; unsigned long long step; };

struct EpilogueArgs {
    float* dpred[2]; float* dconf[2];
    const float* out_sample; const float* out_batch; const double* metrics_f64;
    int B, n_images; size_t plane; double* out16;
    int defer_rescale;      // data parallel: only zero the invalid samples here, the global factor comes later
    const float* param_grads; int n_param_grads;     // parameter gradients riding along in slots 16.. (or NULL)
};

// gradients of sample b *= valid_b ? scale : 0 (exact zeros: an invalid sample's gradients may hold NaN / Inf)
__device__ __forceinline__ void rescale_samples(float* const dpred[2], float* const dconf[2], const float* __restrict__ out_sample,
                                                int B, size_t plane, float scale) {
    const size_t per_sample[2] = {plane * 3, plane};
#pragma unroll
    for (int which = 0; which < 4; ++which) {
        float* base = (which < 2) ? dpred[which] : dconf[which - 2];
        if (!base) continue;
        const size_t n = per_sample[which >> 1];
        const size_t total = n * B;
        for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
            const int b = (int)(idx / n);
            const bool valid = out_sample[(size_t)b * T3D_LOSS_OUT_STRIDE + 5] != 0.f;
            const float f = valid ? scale : 0.f;
            base[idx] = (f == 0.f) ? 0.f : ((f == 1.0f) ? base[idx] : base[idx] * f);
        }
    }
}

template <bool PEERS>
__global__ void __launch_bounds__(128) step_epilogue_kernel(const EpilogueArgs a, const PeerArgs pa) {
    if (blockIdx.x == 0) {
        __shared__ double red[4][14];
        const int tid = threadIdx.x;
        double v[14];
#pragma unroll
        for (int k = 0; k < 14; ++k) v[k] = 0.0;
        for (int b = tid; b < a.B; b += 128) {
            const float* o = a.out_sample + (size_t)b * T3D_LOSS_OUT_STRIDE;
            if (o[5] != 0.f) {
#pragma unroll
                for (int k = 0; k < 5; ++k) v[k] += (double)o[k];
                v[5] += 1.0;
            }
        }
        if (a.metrics_f64) {
            for (int b = tid; b < a.n_images; b += 128) {
                const double* m = a.metrics_f64 + (size_t)b * 8;
#pragma unroll
                for (int k = 0; k < 7; ++k) if (isfinite(m[k])) v[7 + k] += m[k];
            }
        }
        const int lane = tid & 31, wrp = tid >> 5;
#pragma unroll
        for (int k = 0; k < 14; ++k) {
            const double r = warp_sum(v[k]);
            if (lane == 0) red[wrp][k] = r;
        }
        __syncthreads();
        if (tid < kVec) {
            double r;
            if (tid == 6) r = (double)a.B;
            else if (tid == 14) r = a.metrics_f64 ? (double)a.n_images : 0.0;
            else if (tid == 15) r = 0.0;
            else if (tid >= 16) r = (a.param_grads && tid - 16 < a.n_param_grads) ? (double)a.param_grads[tid - 16] : 0.0;
            else r = (red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid]);
            a.out16[tid] = r;
            if (PEERS) {
                const int p = (int)(pa.step & 1ull);
                for (int q = 0; q < pa.world; ++q) pa.box[q]->slots[p][pa.rank][tid] = r;       // peer stores (NVLink)
                __threadfence_system();
                __syncwarp(0x00ffffffu);
                if (tid < pa.world) {
                    unsigned long long* f = &pa.box[tid]->flags[p][pa.rank];
                    const unsigned long long v = pa.step + 1ull;
                    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(f), "l"(v) : "memory");
                }
            }
        }
    }
    const float nv = a.out_batch[5];
    if (nv == (float)a.B) return;                      // every sample valid: the a-priori 1/B scale is right
    // single process: valid samples * B / n_valid, invalid samples -> exact zeros.  Data parallel (PEERS): only the
    // zeros here -- the factor is (B * world) / n_valid over the GLOBAL batch (train_thermal_dustr.py:320,357-360
    // applied to the whole batch), which mailbox_reduce_kernel applies once it has the world's counts.
    const float scale = (PEERS || a.defer_rescale) ? 1.0f : ((nv > 0.f) ? (float)a.B / nv : 0.f);
    rescale_samples(a.dpred, a.dconf, a.out_sample, a.B, a.plane, scale);
}

}  // namespace

extern "C" int t3d_step_epilogue(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                                 const float* loss_per_sample, const float* loss_batch, const double* metrics_f64,
                                 int B, int H, int W, int n_images, int defer_rescale,
                                 const float* param_grads, int n_param_grads, double* out16, void* stream) {
    T3D_REQUIRE(loss_per_sample && loss_batch && out16, "NULL pointer");
    T3D_REQUIRE(B >= 1 && H >= 1 && W >= 1 && n_images >= 0, "bad dims");
    EpilogueArgs a;
    a.dpred[0] = dpred1; a.dpred[1] = dpred2; a.dconf[0] = dconf1; a.dconf[1] = dconf2;
    a.out_sample = loss_per_sample; a.out_batch = loss_batch; a.metrics_f64 = metrics_f64;
    T3D_REQUIRE(n_param_grads >= 0 && n_param_grads <= kVec - 16 && (n_param_grads == 0 || param_grads), "at most %d parameter gradients", kVec - 16);
    a.B = B; a.n_images = n_images; a.plane = (size_t)H * W; a.out16 = out16; a.defer_rescale = defer_rescale ? 1 : 0;
    a.param_grads = param_grads; a.n_param_grads = n_param_grads;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    PeerArgs pa;
    pa.world = 0; pa.rank = 0; pa.step = 0;
    T3D_LAUNCH("step_epilogue_kernel", st, step_epilogue_kernel<false><<<t3d_sm_count() * 8, 128, 0, st>>>(a, pa));
    return T3D_OK;
}

struct ReduceArgs {
    const Mailbox* box; int world; unsigned long long step; double* out16;
    float* dpred[2]; float* dconf[2]; const float* out_sample; int B; size_t plane;     // this rank's step-`step` gradients (or NULL)
};

// Waits for the world's vectors of `step`, adds them in rank order (the same bits on every rank) and -- the global
// validity semantics of train_thermal_dustr.py:320,357-360 over the data-parallel batch -- when any sample of ANY rank
// was invalid, rescales this rank's gradients (a-priori scale 1 / (B * world), invalid samples already zeroed by the
// epilogue) by (B * world) / n_valid_global.  Every block reads the flags and the two counts itself (world <= 16
// loads); in the common all-valid case all but block 0 return at once.
__global__ void __launch_bounds__(128) mailbox_reduce_kernel(const ReduceArgs a) {
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, p = (int)(a.step & 1ull);
    __shared__ double counts[2];
    if (wrp == 0) {
        if (lane < a.world) {
            const unsigned long long* f = &a.box->flags[p][lane];
            unsigned long long v;
            do {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
                if (v < a.step + 1ull) __nanosleep(200);
            } while (v < a.step + 1ull);
        }
        __syncwarp();
        if (lane < kVec) {
            double s = 0.0;
            for (int r = 0; r < a.world; ++r) {                       // rank order: the same bits on every rank
                double x;
                asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(x) : "l"(&a.box->slots[p][r][lane]) : "memory");
                s += x;
            }
            if (blockIdx.x == 0) a.out16[lane] = s;
            if (lane == 5) counts[0] = s;                             // n_valid over the world
            if (lane == 6) counts[1] = s;                             // samples over the world
        }
    }
    __syncthreads();
    if (!a.dpred[0] || counts[0] == counts[1]) return;                // every sample of every rank valid
    const float nv = (float)counts[0];
    const float scale = (nv > 0.f) ? (float)counts[1] / nv : 0.f;
    rescale_samples(a.dpred, a.dconf, a.out_sample, a.B, a.plane, scale);
}

extern "C" size_t t3d_mailbox_bytes(void) { return sizeof(Mailbox); }

extern "C" int t3d_step_epilogue_peers(float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                                       const float* loss_per_sample, const float* loss_batch, const double* metrics_f64,
                                       int B, int H, int W, int n_images,
                                       const float* param_grads, int n_param_grads, double* out16_local,
                                       const unsigned long long* peer_mailboxes, int world, int rank,
                                       unsigned long long step, void* stream) {
    T3D_REQUIRE(loss_per_sample && loss_batch && out16_local && peer_mailboxes, "NULL pointer");
    T3D_REQUIRE(B >= 1 && H >= 1 && W >= 1 && n_images >= 0, "bad dims");
    T3D_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "bad world / rank (at most %d peers)", kMaxPeers);
    EpilogueArgs a;
    a.dpred[0] = dpred1; a.dpred[1] = dpred2; a.dconf[0] = dconf1; a.dconf[1] = dconf2;
    a.out_sample = loss_per_sample; a.out_batch = loss_batch; a.metrics_f64 = metrics_f64;
    T3D_REQUIRE(n_param_grads >= 0 && n_param_grads <= kVec - 16 && (n_param_grads == 0 || param_grads), "at most %d parameter gradients", kVec - 16);
    a.B = B; a.n_images = n_images; a.plane = (size_t)H * W; a.out16 = out16_local; a.defer_rescale = 1;
    a.param_grads = param_grads; a.n_param_grads = n_param_grads;
    PeerArgs pa;
    for (int q = 0; q < kMaxPeers; ++q) pa.box[q] = (q < world) ? reinterpret_cast<Mailbox*>(peer_mailboxes[q]) : nullptr;
    pa.world = world; pa.rank = rank; pa.step = step;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("step_epilogue_kernel", st, step_epilogue_kernel<true><<<t3d_sm_count() * 8, 128, 0, st>>>(a, pa));
    return T3D_OK;
}

extern "C" int t3d_mailbox_reduce(const void* my_mailbox, int world, unsigned long long step, double* out16,
                                  float* dpred1, float* dpred2, float* dconf1, float* dconf2,
                                  const float* loss_per_sample, int B, int H, int W, void* stream) {
    T3D_REQUIRE(my_mailbox && out16, "NULL pointer");
    T3D_REQUIRE(world >= 1 && world <= kMaxPeers, "bad world");
    const bool fixup = dpred1 != nullptr;
    if (fixup) T3D_REQUIRE(dpred2 && loss_per_sample && B >= 1 && H >= 1 && W >= 1, "gradient fix-up needs dpred1/2, loss_per_sample and dims");
    ReduceArgs a;
    a.box = reinterpret_cast<const Mailbox*>(my_mailbox); a.world = world; a.step = step; a.out16 = out16;
    a.dpred[0] = dpred1; a.dpred[1] = fixup ? dpred2 : nullptr; a.dconf[0] = fixup ? dconf1 : nullptr; a.dconf[1] = fixup ? dconf2 : nullptr;
    a.out_sample = loss_per_sample; a.B = B; a.plane = fixup ? (size_t)H * W : 0;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int grid = fixup ? t3d_sm_count() * 4 : 1;
    T3D_LAUNCH("mailbox_reduce_kernel", st, mailbox_reduce_kernel<<<grid, 128, 0, st>>>(a));
    return T3D_OK;
}

// the deferred factor of t3d_step_epilogue(defer_rescale = 1) from an already all-reduced vector (NCCL exchange)
__global__ void __launch_bounds__(128) rescale_global_kernel(const ReduceArgs a) {
    const double nv = a.out16[5], tot = a.out16[6];
    if (nv == tot) return;
    const float nvf = (float)nv;
    rescale_samples(a.dpred, a.dconf, a.out_sample, a.B, a.plane, (nvf > 0.f) ? (float)tot / nvf : 0.f);
}

extern "C" int t3d_rescale_global(float* dpred1, float* dpred2, float* dconf1, float* dconf2, const float* loss_per_sample,
                                  const double* out16_global, int B, int H, int W, void* stream) {
    T3D_REQUIRE(dpred1 && dpred2 && loss_per_sample && out16_global, "NULL pointer");
    T3D_REQUIRE(B >= 1 && H >= 1 && W >= 1, "bad dims");
    ReduceArgs a;
    a.box = nullptr; a.world = 0; a.step = 0; a.out16 = const_cast<double*>(out16_global);
    a.dpred[0] = dpred1; a.dpred[1] = dpred2; a.dconf[0] = dconf1; a.dconf[1] = dconf2;
    a.out_sample = loss_per_sample; a.B = B; a.plane = (size_t)H * W;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    T3D_LAUNCH("rescale_global_kernel", st, rescale_global_kernel<<<t3d_sm_count() * 4, 128, 0, st>>>(a));
    return T3D_OK;
}
