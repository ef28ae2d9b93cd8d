// comm.cu — the one collective of the hot path, fused with the optimizer step: a one-shot gradient all-reduce over
// NVLink peer memory inside the clip_grad_norm_ + Adam launch pair (sm_100a, one process per GPU on one NVSwitch box).
//
// Data-parallel PPO sums the flat fp32 gradient (547 KB for ball3d) over the ranks once per minibatch, 320 times per
// iteration, with the next minibatch waiting for the updated weights: the transfer is latency-bound and fully exposed
// (SB3 has no counterpart — the reference trains in one process; this replaces the `dist.all_reduce(grads)` +
// `tmla_adam_clip_fused` pair of the NCCL path, DESIGN.md §7).  Here every rank owns an IPC-exported exchange buffer:
//     reduce_norm_kernel   (1) PUSH: store the local gradient into slot [parity][rank] of EVERY rank's buffer over NVLink
//                              (posted 128-bit stores: one-way latency; double-buffered by step parity),
//                          (2) the last CTA to finish publishes the step number into every peer's flag word (st.release.sys),
//                          (3) every CTA waits until all peers' flags for this step have arrived in LOCAL memory,
//                          (4) reads its slice of all `world` slots from LOCAL memory (ld.relaxed.sys, 128-bit), sums them in
//                              RANK ORDER — identical on every rank, so replicas stay bit-identical — writes the sum back
//                              into the local gradient and emits the squared-norm partials of clip_grad_norm_;
//                          (round 2 began with a PULL exchange — publish locally, read every peer's slot over NVLink after the
//                          handshake: 20.9 us per exchange at 8 ranks; pushing removes the read round trip from the critical path)
//     adam_kernel          (ppo_kernels.cu, unchanged) clips, steps, clears the gradient, refreshes the bf16 operand images.
// No NCCL launch, no extra pass over the gradient for the norm.  Slot reuse is safe with two parities: a rank pushes step
// s+2 only after its wait of step s+1, i.e. after every peer has published s+1, which each peer does only after it has
// finished reading its slots of step s (stream order).  Spins are bounded (TMLA_COMM_TIMEOUT_MS, default 5000): a missing
// peer sets an error word instead of hanging the GPU; tmla_comm_check reports it.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <cuda_bf16.h>
#include "common.cuh"
#include "mlp_common.cuh"

static constexpr int kMaxRanks = 16;
static constexpr int kReduceBlocks = TMLA_NORM_BLOCKS;      // the Adam kernel sums exactly this many partials
static constexpr int kReduceThreads = 256;

struct tmla_comm {
    int rank, world, device;
    int64_t capacity;                // floats per slot
    size_t bytes;                    // allocation: flags page + 2 parities x world slots
    char *local;                     // this rank's allocation
    char *peer[kMaxRanks];           // every rank's allocation as mapped here (peer[rank] == local)
    uint32_t *ticket;                // device: CTA ticket counter
    int *err;                        // device: set when a spin timed out
    long long timeout_ns;
    bool connected;
};

// layout of one rank's allocation: [0, 4096): flags uint32[2][kMaxRanks] ; then slots [parity][source rank] (each capacity floats,
// 256-byte aligned): slot_offset(capacity, parity * world + source)
static constexpr size_t kFlagBytes = 4096;
__host__ __device__ inline size_t slot_offset(int64_t capacity, int slot) {
    return kFlagBytes + (size_t)slot * (((size_t)capacity * 4 + 255) & ~(size_t)255);
}

struct CommPtrs { char *peer[kMaxRanks]; };

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_f4(float4 *p, const float4 &v) {
    asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 ld_relaxed_sys_f4(const float4 *p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ float warp_sum_comm(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int WORLD>
__global__ void __launch_bounds__(kReduceThreads)
reduce_norm_kernel(CommPtrs cp, int rank, int world_rt, int64_t capacity, float *__restrict__ grads, int64_t np, float scale,
                   uint32_t step, uint32_t *ticket, int *err, long long timeout_ns, float *__restrict__ partial) {
    const int world = WORLD > 0 ? WORLD : world_rt;
    const int parity = (int)(step & 1u);
    char *mine = cp.peer[rank];
    const size_t push_off = slot_offset(capacity, parity * world + rank);     // this rank's slot in every rank's buffer
    __shared__ float sh[kReduceThreads / 32];
    __shared__ int s_last;
    const int64_t nvec = np >> 2;                          // float4 body + scalar tail; slices are contiguous per CTA
    const int64_t per = (nvec + gridDim.x - 1) / gridDim.x, v0 = (int64_t)blockIdx.x * per, v1 = min(nvec, v0 + per);
    // (1) push: local gradient -> slot [parity][rank] of every rank (its own included)
    for (int64_t i = v0 + threadIdx.x; i < v1; i += blockDim.x) {
        const float4 gl = reinterpret_cast<const float4 *>(grads)[i];
        for (int q = 0; q < world; ++q) st_relaxed_sys_f4(reinterpret_cast<float4 *>(cp.peer[q] + push_off) + i, gl);
    }
    if (blockIdx.x == gridDim.x - 1)
        for (int64_t i = (nvec << 2) + threadIdx.x; i < np; i += blockDim.x)
            for (int q = 0; q < world; ++q) *reinterpret_cast<volatile float *>(cp.peer[q] + push_off + (size_t)i * 4) = grads[i];
    __threadfence_system();
    __syncthreads();
    // (2) the last CTA to get here tells every peer (and itself) that this rank's slot holds step `step`
    if (threadIdx.x == 0) {
        const uint32_t t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) *ticket = 0u;                           // re-armed for the next launch (stream order)
    }
    __syncthreads();
    if (s_last) {
        __threadfence_system();
        if (threadIdx.x < world)
            st_release_sys(reinterpret_cast<uint32_t *>(cp.peer[threadIdx.x]) + parity * kMaxRanks + rank, step);
    }
    // (3) wait for every rank's flag of this step in local memory (bounded spin)
    if (threadIdx.x < world) {
        const uint32_t *flag = reinterpret_cast<const uint32_t *>(mine) + parity * kMaxRanks + threadIdx.x;
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        uint32_t spins = 0;
        while (ld_acquire_sys(flag) != step) {
            if ((++spins & 1023u) == 0) {
                unsigned long long t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if ((long long)(t1 - t0) > timeout_ns) { *err = 1 + threadIdx.x; break; }
            }
        }
    }
    __syncthreads();
    // (4) sum the slots of all ranks — now in LOCAL memory — in rank order (identical on every rank), write back, squared-norm partial
    float ss = 0.0f;
    const size_t slot_bytes = slot_offset(capacity, 1) - slot_offset(capacity, 0);
    const char *slots = mine + slot_offset(capacity, parity * world);
    for (int64_t i = v0 + threadIdx.x; i < v1; i += blockDim.x) {
        // all loads are issued before the first sum (with the pull exchange this made ONE NVLink round trip per element out of
        // `world` dependent ones: 30 -> 20.9 us per exchange at 8 ranks)
        constexpr int NQ = WORLD > 0 ? WORLD : kMaxRanks;
        float4 x[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q)
            if (q < world) x[q] = ld_relaxed_sys_f4(reinterpret_cast<const float4 *>(slots + (size_t)q * slot_bytes) + i);
        float4 acc = x[0];
#pragma unroll
        for (int q = 1; q < NQ; ++q)
            if (q < world) { acc.x += x[q].x; acc.y += x[q].y; acc.z += x[q].z; acc.w += x[q].w; }
        reinterpret_cast<float4 *>(grads)[i] = acc;
        const float a = acc.x * scale, b = acc.y * scale, c = acc.z * scale, d = acc.w * scale;
        ss += (a * a + b * b) + (c * c + d * d);
    }
    if (blockIdx.x == gridDim.x - 1) {
        for (int64_t i = (nvec << 2) + threadIdx.x; i < np; i += blockDim.x) {
            float acc = 0.0f;
            for (int q = 0; q < world; ++q) acc += *reinterpret_cast<const volatile float *>(slots + (size_t)q * slot_bytes + (size_t)i * 4);
            grads[i] = acc;
            const float a = acc * scale;
            ss += a * a;
        }
    }
    ss = warp_sum_comm(ss);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < kReduceThreads / 32; ++w) t += sh[w];
        partial[blockIdx.x] = t;
    }
}

// ------------------------------------------------------------------ the whole optimizer step in ONE launch
// gradient exchange (WORLD > 1, as reduce_norm_kernel) -> squared-norm partials -> grid barrier -> clip + Adam + zero_grad +
// refresh of the bf16 operand images, with the (summed) gradient held in registers across the barrier: one launch per minibatch
// instead of gradnorm + adam (single GPU) or reduce_norm + adam (data parallel), and one pass over the gradient instead of two.
// Arithmetic per element is adam_kernel's (ppo_kernels.cu); the norm is the fixed-order sum of TMLA_NORM_BLOCKS partials.
// RMS = true is A2C's torch.optim.RMSprop(alpha, eps) step instead (not centred, no momentum, no weight decay): one state
// vector, square_avg, in `v`, with b2 = alpha and b1 = 1 - alpha (formed in double from the caller's double alpha, then rounded: torch's factors); `m` is unused.
struct OptStepArgs {
    CommPtrs cp; int rank, world; int64_t capacity; uint32_t seq; uint32_t *ticket; int *err; long long timeout_ns;   // exchange (WORLD > 1)
    float *p, *g, *m, *v; int64_t np;
    float scale, max_norm, lr, b1, b2, eps, bc1, bc2_sqrt;
    float *norm_out;                 // [0] = norm, [1 .. 1+TMLA_NORM_BLOCKS) = partials
    int zero_grads;
    __nv_bfloat16 *img0, *img1; int64_t w2_off0, w2_off1;
};
static constexpr int kOptVecPerThread = 2;       // float4 per thread: 128 CTAs x 256 threads x 2 x 4 = 262 144 parameters

// Grid barrier for an ORDINARY launch of at most one small CTA per SM (128 x 256 threads: every CTA is resident as soon as the
// grid starts, also beside the weight-gradient kernel when launched as its programmatic dependent).  bar[0] counts arrivals and
// is reset by the last one, bar[1] is the generation the waiters watch; both live in the caller's zero-initialised scratch.
// A cooperative launch + grid.sync() does the same but costs ~10 us more per launch on the stream (measured below).
__device__ __forceinline__ void opt_grid_barrier(uint32_t *bar, unsigned nblocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        volatile uint32_t *gen = bar + 1;
        const uint32_t g0 = *gen;
        __threadfence();
        if (atomicAdd(bar, 1u) == nblocks - 1) {
            *(volatile uint32_t *)bar = 0u;
            __threadfence();
            *gen = g0 + 1u;
        } else {
            unsigned long long t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            uint32_t spins = 0;
            while (*gen == g0) {
                if ((++spins & 4095u) == 0) {
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t1 - t0 > 5000000000ull) __trap();         // 5 s: a CTA of this grid never became resident
                }
            }
        }
        __threadfence();
    }
    __syncthreads();
}

template <int WORLD, bool RMS>
__global__ void __launch_bounds__(kReduceThreads)
opt_step_kernel(const __grid_constant__ OptStepArgs a) {
    __shared__ float sh[kReduceThreads / 32];
    __shared__ int s_last;
    __shared__ float s_norm;
    const int64_t nvec = a.np >> 2;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gsize = (int64_t)gridDim.x * blockDim.x;
    const int64_t tail0 = nvec << 2;                       // scalar tail [tail0, np): threads 0.. of the last CTA
    const bool tail_owner = blockIdx.x == gridDim.x - 1 && tail0 + threadIdx.x < a.np;
    float4 g[kOptVecPerThread];
    float gt = 0.0f;
    // optimizer state of this thread's elements: in flight across the wait for the gradient, the norm reduction and the grid barrier
    float4 p4[kOptVecPerThread], m4[kOptVecPerThread], v4[kOptVecPerThread];
#pragma unroll
    for (int j = 0; j < kOptVecPerThread; ++j) {
        const int64_t i = gtid + j * gsize;
        if (i < nvec) {
            p4[j] = reinterpret_cast<const float4 *>(a.p)[i];
            if constexpr (!RMS) m4[j] = reinterpret_cast<const float4 *>(a.m)[i];
            v4[j] = reinterpret_cast<const float4 *>(a.v)[i];
        }
    }
    // launched as a programmatic dependent of the weight-gradient kernel: everything above ran beside its last CTAs; the
    // gradient is complete once the prerequisite grids have finished (returns at once after an ordinary launch)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if constexpr (WORLD > 1) {
        const int parity = (int)(a.seq & 1u);
        char *mine = a.cp.peer[a.rank];
        const size_t push_off = slot_offset(a.capacity, parity * WORLD + a.rank);   // this rank's slot in every rank's buffer
        const size_t slot_bytes = slot_offset(a.capacity, 1) - slot_offset(a.capacity, 0);
        const char *slots = mine + slot_offset(a.capacity, parity * WORLD);
#pragma unroll
        for (int j = 0; j < kOptVecPerThread; ++j) {       // push: local gradient -> slot [parity][rank] of every rank
            const int64_t i = gtid + j * gsize;
            if (i < nvec) {
                const float4 gl = reinterpret_cast<const float4 *>(a.g)[i];
#pragma unroll
                for (int q = 0; q < WORLD; ++q) st_relaxed_sys_f4(reinterpret_cast<float4 *>(a.cp.peer[q] + push_off) + i, gl);
            }
        }
        if (tail_owner) {
            const float gl = a.g[tail0 + threadIdx.x];
#pragma unroll
            for (int q = 0; q < WORLD; ++q) *reinterpret_cast<volatile float *>(a.cp.peer[q] + push_off + (size_t)(tail0 + threadIdx.x) * 4) = gl;
        }
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t t = atomicAdd(a.ticket, 1u);
            s_last = (t == gridDim.x - 1);
            if (s_last) *a.ticket = 0u;
        }
        __syncthreads();
        if (s_last) {
            __threadfence_system();
            if (threadIdx.x < WORLD) st_release_sys(reinterpret_cast<uint32_t *>(a.cp.peer[threadIdx.x]) + parity * kMaxRanks + a.rank, a.seq);
        }
        if (threadIdx.x < WORLD) {
            const uint32_t *flag = reinterpret_cast<const uint32_t *>(mine) + parity * kMaxRanks + threadIdx.x;
            unsigned long long t0;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            uint32_t spins = 0;
            while (ld_acquire_sys(flag) != a.seq) {
                if ((++spins & 1023u) == 0) {
                    unsigned long long t1;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if ((long long)(t1 - t0) > a.timeout_ns) { *a.err = 1 + threadIdx.x; break; }
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kOptVecPerThread; ++j) {
            const int64_t i = gtid + j * gsize;
            g[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (i < nvec) {
                float4 x[WORLD];
#pragma unroll
                for (int q = 0; q < WORLD; ++q) x[q] = ld_relaxed_sys_f4(reinterpret_cast<const float4 *>(slots + (size_t)q * slot_bytes) + i);
                float4 acc = x[0];
#pragma unroll
                for (int q = 1; q < WORLD; ++q) { acc.x += x[q].x; acc.y += x[q].y; acc.z += x[q].z; acc.w += x[q].w; }
                g[j] = acc;
            }
        }
        if (tail_owner)
            for (int q = 0; q < WORLD; ++q) gt += *reinterpret_cast<const volatile float *>(slots + (size_t)q * slot_bytes + (size_t)(tail0 + threadIdx.x) * 4);
    } else {
#pragma unroll
        for (int j = 0; j < kOptVecPerThread; ++j) {
            const int64_t i = gtid + j * gsize;
            g[j] = i < nvec ? reinterpret_cast<const float4 *>(a.g)[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        if (tail_owner) gt = a.g[tail0 + threadIdx.x];
    }
    float ss = 0.0f;
#pragma unroll
    for (int j = 0; j < kOptVecPerThread; ++j) {
        const float x0 = g[j].x * a.scale, x1 = g[j].y * a.scale, x2 = g[j].z * a.scale, x3 = g[j].w * a.scale;
        ss += (x0 * x0 + x1 * x1) + (x2 * x2 + x3 * x3);
    }
    { const float xt = gt * a.scale; ss += xt * xt; }
    ss = warp_sum_comm(ss);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < kReduceThreads / 32; ++w) t += sh[w];
        a.norm_out[1 + blockIdx.x] = t;
    }
    opt_grid_barrier(reinterpret_cast<uint32_t *>(a.norm_out + 1 + TMLA_NORM_BLOCKS), gridDim.x);
    if (threadIdx.x < 32) {                                // same summation order in every CTA and on every rank
        float t = 0.0f;
        for (int j = threadIdx.x; j < (int)gridDim.x; j += 32) t += __ldcg(a.norm_out + 1 + j);
        t = warp_sum_comm(t);
        if (threadIdx.x == 0) s_norm = sqrtf(t);
    }
    __syncthreads();
    const float norm = s_norm;
    const float coef = a.max_norm > 0.0f ? fminf(a.max_norm / (norm + 1e-6f), 1.0f) : 1.0f;   // torch clip_grad_norm_
    if (gtid == 0) a.norm_out[0] = norm;
    auto step1 = [&](float gi_raw, float &pp, float &mm, float &vv, int64_t idx) {
        const float gi = gi_raw * a.scale * coef;
        float pn;
        if constexpr (RMS) {                                // square_avg = alpha sq + (1 - alpha) g^2;  p -= lr g / (sqrt(sq) + eps)
            const float vi = a.b2 * vv + a.b1 * gi * gi;
            vv = vi;
            pn = pp - a.lr * (gi / (sqrtf(vi) + a.eps));
        } else {
            const float mi = a.b1 * mm + (1.0f - a.b1) * gi;
            const float vi = a.b2 * vv + (1.0f - a.b2) * gi * gi;
            mm = mi; vv = vi;
            const float denom = sqrtf(vi) / a.bc2_sqrt + a.eps;
            pn = pp - (a.lr / a.bc1) * (mi / denom);
        }
        pp = pn;
        if (a.img0) {                                       // hidden-layer weight: refresh its bf16 operand-image entry
            const int64_t e0 = idx - a.w2_off0, e1 = idx - a.w2_off1;
            const bool in0 = e0 >= 0 && e0 < 65536, in1 = e1 >= 0 && e1 < 65536;
            if (in0 || in1) {
                const int e = (int)(in0 ? e0 : e1), r = e >> 8, k = e & 255;
                (in0 ? a.img0 : a.img1)[(r >> 3) * 2048 + (k >> 3) * 64 + (r & 7) * 8 + (k & 7)] = __float2bfloat16_rn(pn);
            }
        }
    };
#pragma unroll
    for (int j = 0; j < kOptVecPerThread; ++j) {
        const int64_t i = gtid + j * gsize;
        if (i < nvec) {
            step1(g[j].x, p4[j].x, m4[j].x, v4[j].x, 4 * i + 0); step1(g[j].y, p4[j].y, m4[j].y, v4[j].y, 4 * i + 1);
            step1(g[j].z, p4[j].z, m4[j].z, v4[j].z, 4 * i + 2); step1(g[j].w, p4[j].w, m4[j].w, v4[j].w, 4 * i + 3);
            reinterpret_cast<float4 *>(a.p)[i] = p4[j];
            if constexpr (!RMS) reinterpret_cast<float4 *>(a.m)[i] = m4[j];
            reinterpret_cast<float4 *>(a.v)[i] = v4[j];
            reinterpret_cast<float4 *>(a.g)[i] = a.zero_grads ? make_float4(0.0f, 0.0f, 0.0f, 0.0f) : g[j];
        }
    }
    if (tail_owner) {
        const int64_t i = tail0 + threadIdx.x;
        float pp = a.p[i], mm = RMS ? 0.0f : a.m[i], vv = a.v[i];
        step1(gt, pp, mm, vv, i);
        a.p[i] = pp;
        if (!RMS) a.m[i] = mm;
        a.v[i] = vv;
        a.g[i] = a.zero_grads ? 0.0f : gt;
    }
}

// one launch (ordinary or programmatic dependent; own grid barrier)
template <int WORLD, bool RMS>
static int opt_step_launch_t(OptStepArgs &a, cudaStream_t st) {
    static const int mode = [] { const char *e = getenv("TMLA_OPT_PDL"); return e ? atoi(e) : 1; }();   // 0: ordinary launch, 1: programmatic dependent
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(kReduceBlocks); cfg.blockDim = dim3(kReduceThreads); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr; cfg.numAttrs = mode ? 1 : 0;
    TMLA_CUDA(cudaLaunchKernelEx(&cfg, opt_step_kernel<WORLD, RMS>, a));
    return TMLA_OK;
}
static bool opt_step_enabled() {      // TMLA_ADAM=split keeps the two-launch path (A/B runs)
    static const bool on = [] { const char *e = getenv("TMLA_ADAM"); return !(e && !strcmp(e, "split")); }();
    return on;
}
static bool opt_step_fits(const float *params, const float *grads, const float *m, const float *v, int64_t num_params) {
    return (num_params >> 2) <= (int64_t)kReduceBlocks * kReduceThreads * kOptVecPerThread && (num_params & 3) < kReduceThreads &&
           !((reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15u);
}
static void opt_step_comm(OptStepArgs &a, const tmla_comm *c, int64_t step) {
    for (int q = 0; q < kMaxRanks; ++q) a.cp.peer[q] = q < c->world ? c->peer[q] : nullptr;
    a.rank = c->rank; a.world = c->world; a.capacity = c->capacity; a.ticket = c->ticket; a.err = c->err; a.timeout_ns = c->timeout_ns;
    a.seq = (uint32_t)(step & 0x7FFFFFFF) | 0x80000000u;
}
static int opt_step_images(OptStepArgs &a, void *wpack, int obs_dim, int hidden, int n_actions, int64_t num_params) {
    if (!wpack) return TMLA_OK;
    if (hidden != 256) return TMLA_EINVAL;
    const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
    if (o.total != num_params) return TMLA_EINVAL;
    a.img0 = reinterpret_cast<__nv_bfloat16 *>(wpack) + (int64_t)4 * 65536; a.img1 = a.img0 + 65536;
    a.w2_off0 = o.w2[0]; a.w2_off1 = o.w2[1];
    return TMLA_OK;
}
template <bool RMS>
static int opt_step_dispatch(const tmla_comm *c, OptStepArgs &a, cudaStream_t st) {
    switch (c ? c->world : 1) {
        case 1: return opt_step_launch_t<1, RMS>(a, st);
        case 2: return opt_step_launch_t<2, RMS>(a, st);
        case 4: return opt_step_launch_t<4, RMS>(a, st);
        case 8: return opt_step_launch_t<8, RMS>(a, st);
        default: return TMLA_EINVAL;
    }
}

// returns TMLA_EINVAL (without an error message) when the shape does not fit so that callers fall back
int opt_step_launch(tmla_comm *c, float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                    float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, int zero_grads, void *wpack, int obs_dim,
                    int hidden, int n_actions, void *stream) {
    if (!opt_step_enabled() || !opt_step_fits(params, grads, m, v, num_params))
        return TMLA_EINVAL;
    OptStepArgs a;
    memset(&a, 0, sizeof(a));
    if (c) opt_step_comm(a, c, step);
    a.p = params; a.g = grads; a.m = m; a.v = v; a.np = num_params;
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    a.scale = grad_scale; a.max_norm = max_grad_norm; a.lr = lr; a.b1 = beta1; a.b2 = beta2; a.eps = eps; a.bc1 = (float)bc1; a.bc2_sqrt = (float)sqrt(bc2);
    a.norm_out = norm_out; a.zero_grads = zero_grads;
    if (opt_step_images(a, wpack, obs_dim, hidden, n_actions, num_params)) return TMLA_EINVAL;
    return opt_step_dispatch<false>(c, a, (cudaStream_t)stream);
}

// clip + RMSprop: this one-launch form only (no two-launch fallback, TMLA_ADAM does not apply)
static int rmsprop_launch(tmla_comm *c, float *params, float *grads, float *sq_avg, int64_t num_params, float grad_scale, float max_grad_norm,
                          float lr, double alpha, float eps, int64_t step, float *norm_out, int zero_grads, void *wpack, int obs_dim, int hidden,
                          int n_actions, void *stream) {
    TMLA_REQUIRE(params && grads && sq_avg && norm_out, "NULL buffer (norm_out doubles as scratch)");
    TMLA_REQUIRE(num_params > 0, "num_params must be positive");
    if (!opt_step_fits(params, grads, sq_avg, sq_avg, num_params)) {
        tmla_set_error("clip + RMSprop runs as one launch only: at most %d parameters in 16-byte aligned buffers (got %lld)",
                       kReduceBlocks * kReduceThreads * kOptVecPerThread * 4, (long long)num_params);
        return TMLA_EINVAL;
    }
    OptStepArgs a;
    memset(&a, 0, sizeof(a));
    if (c) opt_step_comm(a, c, step);
    a.p = params; a.g = grads; a.v = sq_avg; a.np = num_params;
    a.scale = grad_scale; a.max_norm = max_grad_norm; a.lr = lr; a.b2 = (float)alpha; a.b1 = (float)(1.0 - alpha); a.eps = eps;
    a.norm_out = norm_out; a.zero_grads = zero_grads;
    if (opt_step_images(a, wpack, obs_dim, hidden, n_actions, num_params)) {
        tmla_set_error("wpack needs hidden = 256 and num_params matching (obs_dim, n_actions)");
        return TMLA_EINVAL;
    }
    const int rc = opt_step_dispatch<true>(c, a, (cudaStream_t)stream);
    if (rc == TMLA_EINVAL) tmla_set_error("clip + RMSprop with a gradient exchange covers 2, 4 or 8 ranks (got %d)", c ? c->world : 1);
    return rc;
}

extern "C" {

int tmla_comm_create(int rank, int world, int device, int64_t num_floats, tmla_comm **out, void *handle_out) {
    TMLA_REQUIRE(out && handle_out, "out/handle_out is NULL");
    TMLA_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world, "rank/world out of range (at most 16 ranks)");
    TMLA_REQUIRE(num_floats > 0, "num_floats must be positive");
    int prev = -1;
    cudaGetDevice(&prev);
    TMLA_CUDA(cudaSetDevice(device));
    tmla_comm *c = new (std::nothrow) tmla_comm();
    if (!c) { tmla_set_error("out of host memory"); return TMLA_ENOMEM; }
    memset(c, 0, sizeof(*c));
    c->rank = rank; c->world = world; c->device = device; c->capacity = num_floats;
    c->bytes = slot_offset(num_floats, 2 * world);
    const char *e = getenv("TMLA_COMM_TIMEOUT_MS");
    c->timeout_ns = (long long)(e ? atoll(e) : 5000) * 1000000ll;
    if (cudaMalloc((void **)&c->local, c->bytes) != cudaSuccess || cudaMalloc((void **)&c->ticket, sizeof(uint32_t)) != cudaSuccess ||
        cudaMalloc((void **)&c->err, sizeof(int)) != cudaSuccess) {
        tmla_set_error("tmla_comm_create: cudaMalloc: %s", cudaGetErrorString(cudaGetLastError()));
        tmla_comm_destroy(c);
        if (prev >= 0) cudaSetDevice(prev);
        return TMLA_ENOMEM;
    }
    TMLA_CUDA(cudaMemset(c->local, 0, c->bytes));
    TMLA_CUDA(cudaMemset(c->ticket, 0, sizeof(uint32_t)));
    TMLA_CUDA(cudaMemset(c->err, 0, sizeof(int)));
    TMLA_CUDA(cudaDeviceSynchronize());
    c->peer[rank] = c->local;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handles travel as 64 bytes");
    cudaIpcMemHandle_t hnd;
    TMLA_CUDA(cudaIpcGetMemHandle(&hnd, c->local));
    memcpy(handle_out, &hnd, sizeof(hnd));
    *out = c;
    if (prev >= 0) cudaSetDevice(prev);
    return TMLA_OK;
}

// all_handles: world x 64 bytes, rank-major (what every rank's tmla_comm_create returned, gathered by the caller)
int tmla_comm_connect(tmla_comm *c, const void *all_handles) {
    TMLA_REQUIRE(c && all_handles, "comm/handles is NULL");
    int prev = -1;
    cudaGetDevice(&prev);
    TMLA_CUDA(cudaSetDevice(c->device));
    for (int q = 0; q < c->world; ++q) {
        if (q == c->rank) continue;
        cudaIpcMemHandle_t hnd;
        memcpy(&hnd, (const char *)all_handles + (size_t)q * 64, 64);
        void *p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            tmla_set_error("tmla_comm_connect: cudaIpcOpenMemHandle(rank %d): %s", q, cudaGetErrorString(e));
            cudaGetLastError();
            if (prev >= 0) cudaSetDevice(prev);
            return TMLA_ECUDA;
        }
        c->peer[q] = (char *)p;
    }
    c->connected = true;
    if (prev >= 0) cudaSetDevice(prev);
    return TMLA_OK;
}

int tmla_comm_destroy(tmla_comm *c) {
    if (!c) return TMLA_OK;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int q = 0; q < c->world; ++q)
        if (q != c->rank && c->peer[q]) cudaIpcCloseMemHandle(c->peer[q]);
    if (c->local) cudaFree(c->local);
    if (c->ticket) cudaFree(c->ticket);
    if (c->err) cudaFree(c->err);
    delete c;
    if (prev >= 0) cudaSetDevice(prev);
    return TMLA_OK;
}

// reads the error word (synchronises `stream`): TMLA_ECUDA when a peer's flag did not arrive within the timeout
int tmla_comm_check(tmla_comm *c, void *stream) {
    TMLA_REQUIRE(c, "comm is NULL");
    int err = 0;
    TMLA_CUDA(cudaMemcpyAsync(&err, c->err, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    TMLA_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (err) {
        tmla_set_error("gradient exchange: rank %d never published its gradient (waited %lld ms on rank %d)", err - 1,
                       c->timeout_ns / 1000000ll, c->rank);
        return TMLA_ECUDA;
    }
    return TMLA_OK;
}

// grads <- sum over ranks of grads (rank order), then clip_grad_norm_ + Adam exactly as tmla_adam_clip_fused.
// `step` (the 1-based Adam step) doubles as the exchange sequence number: every rank must call with the same step.
int tmla_adam_clip_allreduce(tmla_comm *c, float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale,
                             float max_grad_norm, float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out,
                             int zero_grads, void *wpack, int obs_dim, int hidden, int n_actions, void *stream) {
    TMLA_REQUIRE(c && c->connected, "comm is NULL or not connected (tmla_comm_connect)");
    TMLA_REQUIRE(params && grads && m && v && norm_out, "NULL buffer");
    TMLA_REQUIRE(num_params > 0 && num_params <= c->capacity && step >= 1, "bad arguments (num_params exceeds the comm's capacity?)");
    TMLA_REQUIRE((reinterpret_cast<uintptr_t>(grads) & 15u) == 0, "grads must be 16-byte aligned");
    {   // one launch for exchange + clip + Adam when the shape fits (2, 4, 8 ranks)
        const int rc = opt_step_launch(c, params, grads, m, v, num_params, grad_scale, max_grad_norm, lr, beta1, beta2, eps, step, norm_out,
                                       zero_grads, wpack, obs_dim, hidden, n_actions, stream);
        if (rc != TMLA_EINVAL) return rc;
    }
    CommPtrs cp;
    for (int q = 0; q < kMaxRanks; ++q) cp.peer[q] = q < c->world ? c->peer[q] : nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t seq = (uint32_t)(step & 0x7FFFFFFF) | 0x80000000u;     // never 0 (the cleared flag value)
#define RN(W) reduce_norm_kernel<W><<<kReduceBlocks, kReduceThreads, 0, st>>>(cp, c->rank, c->world, c->capacity, grads, num_params, grad_scale, \
                                                                               seq, c->ticket, c->err, c->timeout_ns, norm_out + 1)
    switch (c->world) {
        case 2: RN(2); break;
        case 4: RN(4); break;
        case 8: RN(8); break;
        default: RN(0); break;
    }
#undef RN
    TMLA_LAUNCH_CHECK();
    return adam_clip_launch(params, grads, m, v, num_params, grad_scale, max_grad_norm, lr, beta1, beta2, eps, step, norm_out, zero_grads,
                            wpack, obs_dim, hidden, n_actions, stream, true);
}

// torch.nn.utils.clip_grad_norm_ + torch.optim.RMSprop.step (A2C), as tmla_adam_clip_fused with one state vector
int tmla_rmsprop_clip_fused(float *params, float *grads, float *sq_avg, int64_t num_params, float grad_scale, float max_grad_norm, float lr,
                            double alpha, float eps, float *norm_out, int zero_grads, void *wpack, int obs_dim, int hidden, int n_actions,
                            void *stream) {
    return rmsprop_launch(nullptr, params, grads, sq_avg, num_params, grad_scale, max_grad_norm, lr, alpha, eps, 1, norm_out, zero_grads, wpack,
                          obs_dim, hidden, n_actions, stream);
}

// grads <- sum over ranks (rank order), then clip + RMSprop in the same launch; `step` is the exchange sequence number
int tmla_rmsprop_clip_allreduce(tmla_comm *c, float *params, float *grads, float *sq_avg, int64_t num_params, float grad_scale,
                                float max_grad_norm, float lr, double alpha, float eps, int64_t step, float *norm_out, int zero_grads,
                                void *wpack, int obs_dim, int hidden, int n_actions, void *stream) {
    TMLA_REQUIRE(c && c->connected, "comm is NULL or not connected (tmla_comm_connect)");
    TMLA_REQUIRE(num_params <= c->capacity && step >= 1, "bad arguments (num_params exceeds the comm's capacity?)");
    return rmsprop_launch(c, params, grads, sq_avg, num_params, grad_scale, max_grad_norm, lr, alpha, eps, step, norm_out, zero_grads, wpack,
                          obs_dim, hidden, n_actions, stream);
}

}  // extern "C"
