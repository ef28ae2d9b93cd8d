// mlp_train.cu — one PPO minibatch of one tower (policy or value), forward + loss + backward in ONE kernel.
//
// Replaces, for the minibatch loop of SB3's PPO.train (reached from backend/mlagents/training.py:166 with the
// hyper-parameters of training.py:379-389), the chain
//     evaluate_actions (tower forward) -> advantage normalisation -> clipped surrogate / value MSE / entropy
//     -> autograd backward through head, layer 2 and layer 1
// that the unfused path runs as 9 kernels with every [rows,256] activation making a round trip through HBM
// (10 KB per sample).  Here one persistent CTA per SM walks 128-row tiles and keeps everything on chip.
// CUDA cores do only the element-wise work, one thread = (row, 64-column quarter); every reduction over the
// rows of a tile is a tcgen05.mma whose accumulator lives in TMEM for the whole kernel.  17 warps: 16 workers run the
// P phases, one DRIVER warp issues every MMA group (M*) and bulk-TMA store — tcgen05.mma issue blocks while the tensor
// core's queue is full, which would otherwise stall a worker warp (and with it every CTA barrier) for the length of
// the group.  Workers signal "operands staged" on one mbarrier, the driver commits each group to a "done" mbarrier:
//
//   P1  layer 1 (K = obs_dim) on CUDA cores -> H1 (bf16): shared-memory tile (K-major) + a TMEM stash for P7
//   M1  Z2 = H1 . W2^T            16 x (M128 N256 K16), W2 resident in shared memory          -> ACC (TMEM)
//   P3  ACC -> bias + tanh -> H2 (bf16) overwrites the tile
//   MH  head outputs = H2 . WHT  (N = 16: hi | hi | lo parts of Wh, WHT read MN-major)        -> HEAD (TMEM)
//   P4  loss per row, d(loss)/d(head) written as a [128][16] bf16 hi/lo tile DOUT
//   M2  dH2 = DOUT . Wh (one K=16 MMA) -> ACC;   dWh += H2^T . DOUT (H2 tile read MN-major)  -> GWH (TMEM)
//   P5  dZ2 = ACC * (1 - H2^2) -> tile
//   M3  dH1 = dZ2 . W2 — the SAME resident W2 bytes through an MN-major descriptor              -> ACC
//       db2 += dZ2^T . 1 (ones column of the XB tile)                                           -> GB2 (TMEM)
//       meanwhile the CUDA cores compute layer 1 of the NEXT tile into registers
//   P7  dZ1 = ACC * (1 - H1^2) (H1 from the TMEM stash) -> tile
//   M4  dW1|db1 += dZ1^T . [x_hi | x_lo | 1]  (XB tile, bf16 hi/lo split of the fp32 observations)  -> GW1 (TMEM)
//
// Only H1 and dZ2 (2 x 512 B per sample) are written out, for the split-K weight-gradient GEMM
// dW2 = dZ2^T . H1 whose 256x256 fp32 accumulator needs all 512 TMEM columns (tc_wgrad_tiled_kernel below).
// They leave as whole 64 KB tile IMAGES (the shared-memory operand layout, byte for byte) through one bulk-TMA
// store per tile (cp.async.bulk.global.shared::cta) and come back the same way, so neither kernel spends a
// single LSU instruction on them.
//
// MN-major trick: a [rows][C] bf16 tile staged in the canonical K-major SWIZZLE_NONE layout
// (16-byte chunk (r, cb) at (r/8)*G + cb*S + (r%8)*16) is, byte for byte, also the canonical MN-major layout of
// its transpose with SBO = S (stride between 8-element groups along MN) and LBO = G (stride between 8-row groups
// along K) — cute::UMMA "((1,n),(8,k)):((X,SBO),(1,LBO))" in uint128 units.  So one staged tile serves as the
// K-major A operand of one GEMM and the MN-major A/B operand of the next, and W2 needs no transposed copy.
#include <algorithm>
#include <stdlib.h>
#include <string.h>
#include <cuda_bf16.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "mlp_common.cuh"

static constexpr int kTrainThreads = 512;                  // 16 worker warps: row = (warp%4)*32 + lane, column quarter = warp/4 (+ 1 driver warp)

__host__ __device__ constexpr uint32_t make_idesc_major(int M, int N, int a_mn, int b_mn) {
    return make_idesc(M, N) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16);
}

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// 32 lanes x 16 consecutive columns, issue only (pair with tmem_wait_ld)
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t *r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t *r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void launder8(uint32_t *r) {
    asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// pins 16 registers behind the preceding (volatile) wait: their consumers cannot be scheduled above it
__device__ __forceinline__ void launder16(uint32_t *r) {
    asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t *r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// bulk TMA (1-D, no tensor map): shared -> global store tracked by bulk async-groups, global -> shared load
// tracked by an mbarrier transaction count
__device__ __forceinline__ void bulk_store(void *gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}
// the same load with an L2 eviction-priority hint (createpolicy): image chunks are read exactly once
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_load_hint(uint32_t sdst, const void *gsrc, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(sdst), "l"(gsrc),
                 "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// per-thread asynchronous global -> shared copies (LDGSTS): the prefetched rows never occupy registers
template <int BYTES>
__device__ __forceinline__ void cp_async_ca(uint32_t dst, const void *src, uint32_t src_bytes) {   // src_bytes 0 = zero-fill
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;" ::"r"(dst), "l"(src), "n"(BYTES), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one elected lane of a converged warp (warp-uniform control flow keeps the tcgen05 operands in uniform registers;
// a `tid == 0` branch makes the compiler wrap every MMA in a lane-serialising loop)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.b32 %0, 1, 0, P;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t bf16_bits(float v) { return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v)); }
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// optional phase clocks (compile with -DTMLA_PHASE_CLOCKS): thread 0 of every CTA accumulates the cycles between
// consecutive marks of the worker tile loop in shared memory; CTA 0 publishes them (profiles/phase_clocks.py)
#ifdef TMLA_PHASE_CLOCKS
__device__ unsigned long long g_phase_cycles[32];
__device__ unsigned int g_cta_loop[512];      // per CTA of the LAST launch: tile-loop cycles, SM id
#define TMLA_PH(i) do { if (tid == 0) { const long long c__ = clock64(); ph_acc[i] += (unsigned long long)(c__ - ph_clock); ph_clock = c__; } } while (0)
#else
#define TMLA_PH(i) do { } while (0)
#endif

struct TowerTrainArgs {
    // tower parameters (fp32 views into the flat vector; W2 from the bf16 pack)
    const float *W1, *B1;
    const __nv_bfloat16 *W2;       // the 128 KB operand image written by tmla_mlp_pack_bf16
    const float *B2, *Wh, *Bh;
    // minibatch
    const float *x;                 // obs [total][D]
    const int32_t *index;           // int32[M] row offsets into x / the [T*N] buffers (NULL = identity)
    int64_t M;
    const int32_t *actions;         // policy tower
    const float *adv, *old_logp;
    const float *returns;           // value tower
    const double *adv_sums;         // (sum, sum of squares, count) or NULL
    int normalize;
    float clip, ent_coef, vf_coef, inv_rows;
    // outputs
    __nv_bfloat16 *h1_out, *dz2_out;    // ceil(M/128) tile images of 64 KB each (shared-memory operand layout), for the dW2 GEMM
    float *out;                          // optional [M][NOUT] head outputs (logits / values)
    float *gW1, *gB1, *gB2, *gWh, *gBh;  // gradient slices (accumulated with atomics; caller zeroes)
    float *stats;                        // float[8] (tmla_ppo_loss layout), accumulated
};

// small [rows][16] bf16 operand tiles: chunk (r, cb) at (r/8)*256 + cb*128 + (r%8)*16
static constexpr uint32_t ksS = 128, ksG = 256;

template <int D, int NOUT>
struct TrainSmem {
    static constexpr uint32_t w = 0;                                   // W2 bf16 [256][256], K-major (kLBO/kSBO)
    static constexpr uint32_t tile = kWBytes;                          // [128][256] bf16, same layout: H1 -> H2 -> dZ2 -> dZ1
    static constexpr uint32_t wht = tile + 128 * 512;                  // [256 j][16] bf16: Wh^T hi | hi | lo  (K-major B of dH2 = DOUT . Wh; MN-major B of the head GEMM)
    static constexpr uint32_t dout = wht + 256 * 32;                   // [128 r][16] bf16: dout hi | lo | hi
    static constexpr uint32_t xb = dout + 128 * 32;                    // [128 r][16] bf16: x hi | x lo | 1
    static constexpr uint32_t w1t = xb + 128 * 32;                     // float [D][256]  (W1 transposed)
    static constexpr uint32_t b1 = w1t + D * H * 4;                    // float [256]
    static constexpr uint32_t b2 = b1 + H * 4;                         // float [256]
    static constexpr uint32_t xs = b2 + H * 4;                         // float [128][D]: next tile's observation rows (cp.async staging)
    static constexpr uint32_t ls = xs + 128 * D * 4;                   // [128][3] words: next tile's loss inputs (action|adv|old_logp or return)
    static constexpr uint32_t idx = ls + 128 * 12;                     // int32 [2][128]: buffer rows of the next two tiles (-1 = past the end)
    static constexpr uint32_t RS = (4 + NOUT) | 1;                     // odd row stride (bank-conflict free)
    static constexpr uint32_t racc = idx + 2 * 128 * 4;                // float [128][RS]: per-row running sums (4 loss statistics, NOUT head-bias gradients)
    static constexpr uint32_t bar = racc + 128 * RS * 4 + 16;          // + adv_mean, adv_inv_std
#ifdef TMLA_PHASE_CLOCKS
    static constexpr uint32_t total = bar + 64 + 256;
#else
    static constexpr uint32_t total = bar + 64;
#endif
};

// loss of the policy tower (the value tower's mean squared error is the same for both): PPO's clipped surrogate, or A2C's plain
// policy gradient -(adv * log_prob).mean() (SB3 2.9.0 a2c.py), which has no ratio, no clip and reads no old log-probabilities
enum { kLossPPO = 0, kLossA2C = 1 };

template <int D, int NOUT, int LOSS = kLossPPO>
__global__ void __launch_bounds__(kTrainThreads + 32, 1)
tc_tower_train_kernel(const __grid_constant__ TowerTrainArgs p) {
    using L = TrainSmem<D, NOUT>;
    constexpr bool PI = NOUT > 1;
    static_assert(3 * NOUT <= 16 && 2 * D + 1 <= 16, "operand tiles are 16 columns wide");
    // the next launch of the minibatch is a programmatic dependent (the value tower, which needs none of the policy tower's
    // results; then the weight-gradient kernel, which waits for the grids before its first image load): let its CTAs take
    // over every SM this kernel's CTA leaves (a no-op when the next launch is an ordinary one)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#ifdef TMLA_PHASE_CLOCKS
    const long long ph_t0 = clock64();
    unsigned long long ph_g0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ph_g0));
#endif
    // TMEM columns: ACC (Z2 / dH2 / dH1), H1 stash (bf16 pairs), persistent gradient accumulators
    constexpr uint32_t C_ACC = 0, C_H1 = 256, C_GWH = 384, C_GB2 = 416, C_GW1 = 448, C_HEAD = 480;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *Ws = smem + L::w, *Ts = smem + L::tile;
    float *w1t = reinterpret_cast<float *>(smem + L::w1t), *b1s = reinterpret_cast<float *>(smem + L::b1);
    float *b2s = reinterpret_cast<float *>(smem + L::b2);
    uint64_t *bar0 = reinterpret_cast<uint64_t *>(smem + L::bar), *bar1 = bar0 + 1;   // MMA groups done: M1/M3 and MH/M2/M4
    uint64_t *rdy = bar0 + 2, *bar_st = bar0 + 3;         // workers -> driver "operands staged"; driver -> workers "tile image read"
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + L::bar + 32);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);  // the same value, provably warp-uniform
    // Warps 0..15 are the workers (CUDA-core phases); warp 16 is the DRIVER: one elected lane issues every tcgen05.mma
    // and bulk-TMA store.  tcgen05.mma issue blocks while the tensor core's queue is full (measured: ~2400 cycles for
    // the 16 MMAs of M1), so a worker warp that also issues stalls the whole CTA at the next barrier.
    const bool is_driver = warp_u == kTrainThreads / 32;
    auto worker_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kTrainThreads) : "memory"); };
    const int64_t M = p.M;
    const int64_t ntiles = (M + 127) / 128;
    if ((int64_t)blockIdx.x >= ntiles) return;

    const int rt = (warp & 3) * 32 + lane, cq = warp >> 2;  // this thread's row of the tile and 64-column quarter
    uint8_t *trow = Ts + (rt >> 3) * kSBO + (rt & 7) * 16;  // + kb * kLBO: 16-byte chunk kb of row rt

    // Prefetch = cp.async straight into shared memory (no registers, nothing blocks; a prefetched value held in a
    // register gets spilled by ptxas, and the spill store waits for the load).  Per 128-row tile: the minibatch index,
    // then the observation rows it selects, then the loss inputs — thread (rt, cq) copies piece cq of row rt.
    float *xs = reinterpret_cast<float *>(smem + L::xs);
    uint32_t *lsb = reinterpret_cast<uint32_t *>(smem + L::ls);
    int32_t *idxs = reinterpret_cast<int32_t *>(smem + L::idx);
    auto fetch_index = [&](uint32_t parity, int64_t tile) {          // index of `tile` -> idxs[parity]
        if (cq == 3) {
            const int64_t row = tile * 128 + rt;
            if (tile < ntiles && row < M && p.index) cp_async_ca<4>(smem_u32(idxs + parity * 128 + rt), p.index + row, 4u);
            else idxs[parity * 128 + rt] = (tile < ntiles && row < M) ? (int32_t)row : -1;
        }
    };
    auto fetch_rows = [&](uint32_t parity) {                         // observation rows selected by idxs[parity] -> xs
        const int32_t sn = idxs[parity * 128 + rt];
        const bool ok = sn >= 0;
        const int64_t src = ok ? (int64_t)sn : 0;
        if (D == 7) {                                                // 28-byte rows: 4-byte pieces cq and cq + 4
            cp_async_ca<4>(smem_u32(xs + rt * D + cq), p.x + src * D + cq, ok ? 4u : 0u);
            if (cq + 4 < D) cp_async_ca<4>(smem_u32(xs + rt * D + cq + 4), p.x + src * D + cq + 4, ok ? 4u : 0u);
        } else if (D == 6) {
            if (cq < 3) cp_async_ca<8>(smem_u32(xs + rt * D + cq * 2), p.x + src * D + cq * 2, ok ? 8u : 0u);
        } else if (cq < 1) cp_async_ca<16>(smem_u32(xs + rt * D), p.x + src * D, ok ? 16u : 0u);
    };
    auto fetch_loss_inputs = [&](uint32_t parity) {                  // loss inputs of the rows selected by idxs[parity] -> ls
        if (cq == 3) {
            const int32_t sn = idxs[parity * 128 + rt];
            const bool ok = sn >= 0;
            const int64_t src = ok ? (int64_t)sn : 0;
            const uint32_t dst = smem_u32(lsb + rt * 3);
            if (PI) {
                cp_async_ca<4>(dst, p.actions + src, ok ? 4u : 0u);
                cp_async_ca<4>(dst + 4, p.adv + src, ok ? 4u : 0u);
                if (LOSS == kLossPPO) cp_async_ca<4>(dst + 8, p.old_logp + src, ok ? 4u : 0u);
            } else cp_async_ca<4>(dst, p.returns + src, ok ? 4u : 0u);
        }
    };
    // Prologue, ordered so that nothing waits alone: the index fetch of the first two tiles flies while the barriers are set up,
    // the W2 image load is issued and the constant tiles are built; the observation rows it selects fly while the transposed
    // layer-1 weights are staged.
    fetch_index(0u, blockIdx.x);
    fetch_index(1u, (int64_t)blockIdx.x + gridDim.x);
    cp_async_commit();

    if (warp == 0) tmem_alloc<512>(tmem_holder);
    if (tid == 32) { mbar_init(bar0, 1); mbar_init(bar1, 1); mbar_init(rdy, 1); mbar_init(bar_st, 1); fence_barrier_init(); }
    if (tid == 32) { mbar_expect_tx(bar0, kWBytes); bulk_load(smem_u32(Ws), p.W2, kWBytes, bar0); }   // W2 image: one bulk-TMA load
    // advantage normalisation constants (PPO.train: (adv - mean) / (std + 1e-8), std unbiased) and the per-row running
    // sums live in shared memory: registers are the scarce resource of this kernel
    float *racc = reinterpret_cast<float *>(smem + L::racc), *advc = racc + 128 * L::RS;
    if (tid == 64) {
        float adv_mean = 0.0f, adv_inv_std = 1.0f;
        if (PI && p.normalize) {
            const double cnt = p.adv_sums[2], mu = p.adv_sums[0] / cnt;
            double var = (p.adv_sums[1] - p.adv_sums[0] * mu) / (cnt - 1.0);
            var = var > 0.0 ? var : 0.0;
            adv_mean = (float)mu;
            adv_inv_std = 1.0f / ((float)sqrt(var) + 1e-8f);
            if (blockIdx.x == 0) { p.stats[6] = adv_mean; p.stats[7] = (float)sqrt(var); }
        }
        advc[0] = adv_mean; advc[1] = adv_inv_std;
    }
    for (int e = tid; e < 128 * (int)L::RS; e += blockDim.x) racc[e] = 0.0f;
    if (tid < H) { b1s[tid] = p.B1[tid]; b2s[tid] = p.B2[tid]; }
    if (tid >= 256 && tid < 256 + H) {                     // WHT[j][c]: c in [0,NOUT) hi, [NOUT,2NOUT) hi, [2NOUT,3NOUT) lo
        // one thread per hidden unit: its NOUT head weights are NOUT independent coalesced loads (one global latency for the
        // whole tile; the element-wise loop this replaces paid eight dependent ones), the row leaves as two 16-byte stores
        const int j = tid - 256;
        float w[NOUT], v[16];
#pragma unroll
        for (int a = 0; a < NOUT; ++a) w[a] = __ldg(p.Wh + a * H + j);
#pragma unroll
        for (int c = 0; c < 16; ++c) v[c] = 0.0f;
#pragma unroll
        for (int a = 0; a < NOUT; ++a) { v[a] = w[a]; v[NOUT + a] = w[a]; v[2 * NOUT + a] = w[a] - bf16_round(w[a]); }
        uint8_t *wr = smem + L::wht + (j >> 3) * ksG + (j & 7) * 16;
        *reinterpret_cast<uint4 *>(wr) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        *reinterpret_cast<uint4 *>(wr + ksS) = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
    }
    cp_async_wait_all();                                   // the index of the first two tiles
    __syncthreads();
    fetch_rows(0u);
    fetch_loss_inputs(0u);
    cp_async_commit();
    {                                                      // W1 transposed into shared memory: all loads of a thread in flight together
        constexpr int NW = (H * D + kTrainThreads + 31) / (kTrainThreads + 32);
        float wv[NW];
#pragma unroll
        for (int q = 0; q < NW; ++q) { const int e = tid + q * (kTrainThreads + 32); if (e < H * D) { const int k = e / H, j = e - k * H; wv[q] = __ldg(p.W1 + j * D + k); } }
#pragma unroll
        for (int q = 0; q < NW; ++q) { const int e = tid + q * (kTrainThreads + 32); if (e < H * D) w1t[e] = wv[q]; }
    }
    cp_async_wait_all();                                   // the first tile's rows
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
    const uint32_t lane_base = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t t_addr = smem_u32(Ts), w_addr = smem_u32(Ws);
    const uint32_t wht_addr = smem_u32(smem + L::wht), dout_addr = smem_u32(smem + L::dout), xb_addr = smem_u32(smem + L::xb);
    uint32_t ph0 = 0, ph1 = 0, phs = 0;                     // phs: parity of bar_st (workers) / rdy (driver)

    // layer 1, H1 = tanh(x W1^T + b1): this thread computes rows l1row + 8*i (i < 4) x 16 columns from l1col — every
    // weight load then serves four rows (broadcast LDS.128 costs four shared-memory cycles each, and one
    // row x 64 columns per thread needed 112 of them); observation rows come from the cp.async staging tile.
    const int l1row = (warp & 3) * 32 + (lane & 7), l1col = cq * 64 + (lane >> 3) * 16;
    uint32_t h1p[32];                                      // [4 rows][8 packed pairs]
    auto layer1 = [&]() {
        float xr[4][D];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < D; ++k) xr[i][k] = xs[(l1row + 8 * i) * D + k];
#pragma unroll
        for (int g = 0; g < 8; ++g) {                      // two hidden units per step (keeps the live weight registers at 14)
            const int col = l1col + g * 2;
            const float2 bb = *reinterpret_cast<const float2 *>(b1s + col);
            float2 ww[D];
#pragma unroll
            for (int k = 0; k < D; ++k) ww[k] = *reinterpret_cast<const float2 *>(w1t + k * H + col);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float2 v = bb;
#pragma unroll
                for (int k = 0; k < D; ++k) v = __ffma2_rn(make_float2(xr[i][k], xr[i][k]), ww[k], v);
                h1p[i * 8 + g] = pack_bf16(tanh_fast(v.x), tanh_fast(v.y));
            }
        }
    };
    if (!is_driver) layer1();
    mbar_wait(bar0, ph0);                                  // the W2 image has landed (its load overlapped everything above)
    ph0 ^= 1u;

    uint32_t it = 0;
#ifdef TMLA_PHASE_CLOCKS
    unsigned long long *ph_acc = reinterpret_cast<unsigned long long *>(smem + L::bar + 64);
    if (tid == 0) for (int i = 0; i < 32; ++i) ph_acc[i] = 0;
    long long ph_clock = clock64();
    const long long ph_t1 = ph_clock;
#endif
    if (is_driver) {
        // ================================ driver warp: tensor core + bulk TMA ================================
        if (elect_one()) {
            auto wait_ready = [&] { mbar_wait(rdy, phs); phs ^= 1u; tc_fence_after(); };
            for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
                // M1: Z2 = H1 . W2^T -> ACC, and the H1 tile image -> HBM.  The store is issued FIRST: tcgen05.mma issue
                // blocks while the tensor core's queue is full, the bulk copy then runs beside the MMAs
                wait_ready();
                if (p.h1_out) {                            // (NULL: the weight-gradient kernel recomputes H1, nothing to write)
                    bulk_store(p.h1_out + tile * (128 * H), t_addr, 128 * H * 2);
                    bulk_commit();
                }
#pragma unroll
                for (int kk = 0; kk < H / 16; ++kk)
                    umma_bf16(tmem_base + C_ACC, make_desc_raw(t_addr + kk * 2 * kLBO, kLBO, kSBO), make_desc_raw(w_addr + kk * 2 * kLBO, kLBO, kSBO),
                              make_idesc_major(128, 256, 0, 0), kk > 0 ? 1u : 0u);
                umma_commit(bar0);
                bulk_wait_read_all();                      // the store has read the tile: the workers may overwrite it with H2
                mbar_arrive(bar_st);
                // MH: head outputs = H2 . WHT -> HEAD (16 columns: hi | hi | lo parts of Wh; WHT read MN-major)
                wait_ready();
#pragma unroll
                for (int kk = 0; kk < H / 16; ++kk)
                    umma_bf16(tmem_base + C_HEAD, make_desc_raw(t_addr + kk * 2 * kLBO, kLBO, kSBO), make_desc_raw(wht_addr + kk * 2 * ksG, ksG, ksS),
                              make_idesc_major(128, 16, 0, 1), kk > 0 ? 1u : 0u);
                umma_commit(bar1);
                // M2: dH2 = DOUT . Wh -> ACC (one K=16 MMA);  dWh += H2^T . DOUT -> GWH (H2 tile and DOUT read MN-major)
                wait_ready();
                umma_bf16(tmem_base + C_ACC, make_desc_raw(dout_addr, ksS, ksG), make_desc_raw(wht_addr, ksS, ksG), make_idesc_major(128, 256, 0, 0), 0u);
#pragma unroll
                for (int mh = 0; mh < 2; ++mh)             // hidden units 0..127 / 128..255 = accumulator lanes
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk)         // K = 16 rows of the tile per step
                        umma_bf16(tmem_base + C_GWH + mh * 16, make_desc_raw(t_addr + mh * 16 * kLBO + kk * 2 * kSBO, kSBO, kLBO),
                                  make_desc_raw(dout_addr + kk * 2 * ksG, ksG, ksS), make_idesc_major(128, 16, 1, 1), (it > 0 || kk > 0) ? 1u : 0u);
                umma_commit(bar1);
                // M3: dH1 = dZ2 . W2 -> ACC (W2 tile read MN-major);  db2 += dZ2^T . XB -> GB2 (its ones column is db2);
                //     then the dZ2 tile image -> HBM
                wait_ready();
                bulk_store(p.dz2_out + tile * (128 * H), t_addr, 128 * H * 2);
                bulk_commit();
#pragma unroll
                for (int kk = 0; kk < H / 16; ++kk)        // K = layer-2 output index j: 16 rows of the W2 tile per step
                    umma_bf16(tmem_base + C_ACC, make_desc_raw(t_addr + kk * 2 * kLBO, kLBO, kSBO),
                              make_desc_raw(w_addr + kk * 2 * kSBO, /*LBO: K groups*/ kSBO, /*SBO: N groups*/ kLBO), make_idesc_major(128, 256, 0, 1), kk > 0 ? 1u : 0u);
#pragma unroll
                for (int mh = 0; mh < 2; ++mh)
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk)
                        umma_bf16(tmem_base + C_GB2 + mh * 16, make_desc_raw(t_addr + mh * 16 * kLBO + kk * 2 * kSBO, kSBO, kLBO),
                                  make_desc_raw(xb_addr + kk * 2 * ksG, ksG, ksS), make_idesc_major(128, 16, 1, 1), (it > 0 || kk > 0) ? 1u : 0u);
                umma_commit(bar0);
                bulk_wait_read_all();
                mbar_arrive(bar_st);
                // M4: dW1 | db1 += dZ1^T . [x_hi | x_lo | 1] -> GW1
                wait_ready();
#pragma unroll
                for (int mh = 0; mh < 2; ++mh)
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk)
                        umma_bf16(tmem_base + C_GW1 + mh * 16, make_desc_raw(t_addr + mh * 16 * kLBO + kk * 2 * kSBO, kSBO, kLBO),
                                  make_desc_raw(xb_addr + kk * 2 * ksG, ksG, ksS), make_idesc_major(128, 16, 1, 1), (it > 0 || kk > 0) ? 1u : 0u);
                umma_commit(bar1);
            }
            bulk_wait_all();                               // the last tile images have reached global memory
        }
        __syncwarp();
    } else
    // ======================================== worker warps: CUDA-core phases ========================================
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int64_t row0 = tile * 128;
        const bool has_next = tile + gridDim.x < ntiles;
        // ---- P1: H1 (computed during the previous tile's M3) -> tile + TMEM stash; XB = [x_hi | x_lo | 1]
        if (it > 0) { mbar_wait(bar1, ph1); ph1 ^= 1u; tc_fence_after(); }   // M4 of the previous tile has read the tile and XB
        TMLA_PH(0);
#pragma unroll
        for (int i = 0; i < 4; ++i) {                      // a quarter-warp writes 8 different rows of one chunk column: conflict-free
            uint8_t *dst = Ts + ((l1row + 8 * i) >> 3) * kSBO + (l1col >> 3) * kLBO + (lane & 7) * 16;
            *reinterpret_cast<uint4 *>(dst) = make_uint4(h1p[i * 8], h1p[i * 8 + 1], h1p[i * 8 + 2], h1p[i * 8 + 3]);
            *reinterpret_cast<uint4 *>(dst + kLBO) = make_uint4(h1p[i * 8 + 4], h1p[i * 8 + 5], h1p[i * 8 + 6], h1p[i * 8 + 7]);
        }
        if (cq == 0) {
            float v[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) v[c] = 0.0f;
#pragma unroll
            for (int k = 0; k < D; ++k) { const float xv = xs[rt * D + k]; v[k] = xv; v[D + k] = xv - bf16_round(xv); }
            v[2 * D] = 1.0f;
            uint8_t *xr = smem + L::xb + (rt >> 3) * ksG + (rt & 7) * 16;
            *reinterpret_cast<uint4 *>(xr) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
            *reinterpret_cast<uint4 *>(xr + ksS) = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
        }
        fence_proxy_async();
        tc_fence_before();
        worker_sync();
        TMLA_PH(1);
        // ---- M1: Z2 = H1 . W2^T -> ACC;  meanwhile the H1 image -> HBM, H1 rows -> TMEM stash, next-tile prefetch
        if (tid == 0) mbar_arrive(rdy);                    // -> driver: M1 (+ H1 image store)
        if (has_next) {                                    // xs is free (layer 1 and XB of this tile are done), so is this tile's index slot
            fetch_rows((it + 1) & 1u);
            fetch_index(it & 1u, tile + 2 * (int64_t)gridDim.x);
            cp_async_commit();
        }
        {                                                  // this thread's (row, 64 columns) of H1 -> TMEM stash for P7
            uint32_t hrow[32];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint4 v = *reinterpret_cast<const uint4 *>(trow + (cq * 8 + c) * kLBO);
                hrow[4 * c] = v.x; hrow[4 * c + 1] = v.y; hrow[4 * c + 2] = v.z; hrow[4 * c + 3] = v.w;
            }
            tmem_st16(lane_base + C_H1 + cq * 32, hrow);
            tmem_st16(lane_base + C_H1 + cq * 32 + 16, hrow + 16);
            tmem_wait_st();
        }
        mbar_wait(bar0, ph0);
        ph0 ^= 1u;
        TMLA_PH(2);
        tc_fence_after();
        mbar_wait(bar_st, phs);                            // the H1 image store has read the tile: it may be overwritten
        phs ^= 1u;
        worker_sync();
        TMLA_PH(3);
        // ---- P3: H2 = tanh(Z2 + b2) -> tile
        {
            const uint32_t taddr = lane_base + C_ACC + cq * 64;
            uint32_t acc[2][16];
            tmem_ld16_nowait(taddr, acc[0]);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                tmem_wait_ld();
                launder16(acc[c & 1]);
                if (c < 3) tmem_ld16_nowait(taddr + (c + 1) * 16, acc[(c + 1) & 1]);
                const int col = cq * 64 + c * 16;
                uint32_t o[8];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 bb = *reinterpret_cast<const float4 *>(b2s + col + 4 * q);
                    o[2 * q] = pack_bf16(tanh_fast(__uint_as_float(acc[c & 1][4 * q + 0]) + bb.x), tanh_fast(__uint_as_float(acc[c & 1][4 * q + 1]) + bb.y));
                    o[2 * q + 1] = pack_bf16(tanh_fast(__uint_as_float(acc[c & 1][4 * q + 2]) + bb.z), tanh_fast(__uint_as_float(acc[c & 1][4 * q + 3]) + bb.w));
                }
                const int kb = col >> 3;
                *reinterpret_cast<uint4 *>(trow + kb * kLBO) = make_uint4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<uint4 *>(trow + (kb + 1) * kLBO) = make_uint4(o[4], o[5], o[6], o[7]);
            }
        }
        fence_proxy_async();
        tc_fence_before();
        worker_sync();                                   // ACC drained, H2 tile complete
        TMLA_PH(4);
        // ---- MH: head outputs = H2 . WHT -> HEAD (16 columns: hi | hi | lo parts of Wh; WHT read MN-major)
        if (tid == 0) mbar_arrive(rdy);                    // -> driver: MH
        mbar_wait(bar1, ph1);
        ph1 ^= 1u;
        TMLA_PH(5);
        tc_fence_after();
        // ---- P4: loss of row rt (threads of column quarter 0), d(loss)/d(head output) -> DOUT tile (bf16 hi | lo | hi)
        if (cq == 0) {
            const bool valid = row0 + rt < M;
            float z[NOUT], dz[NOUT];
            const uint32_t *lin = lsb + rt * 3;             // action | adv | old_logp  or  return
            const int32_t a_cur = (int32_t)lin[0];
            const float f0_cur = __uint_as_float(PI ? lin[1] : lin[0]), f1_cur = __uint_as_float(lin[2]);
            {
                uint32_t hd[16];
                tmem_ld16(lane_base + C_HEAD, hd);
#pragma unroll
                for (int a = 0; a < NOUT; ++a) z[a] = (__uint_as_float(hd[a]) + __uint_as_float(hd[2 * NOUT + a])) + __ldg(p.Bh + a);
            }
            if (p.out && valid) {
#pragma unroll
                for (int a = 0; a < NOUT; ++a) p.out[(row0 + rt) * NOUT + a] = z[a];
            }
            if (PI) {
                float m = z[0];
#pragma unroll
                for (int j = 1; j < NOUT; ++j) m = fmaxf(m, z[j]);
                float pr[NOUT], lp[NOUT], S = 0.0f;
#pragma unroll
                for (int j = 0; j < NOUT; ++j) { pr[j] = __expf(z[j] - m); S += pr[j]; }
                const float logS = __logf(S), invS = __fdividef(1.0f, S);
                float ent = 0.0f;
#pragma unroll
                for (int j = 0; j < NOUT; ++j) { lp[j] = (z[j] - m) - logS; pr[j] *= invS; ent -= pr[j] * lp[j]; }
                float logp = lp[0];
#pragma unroll
                for (int j = 1; j < NOUT; ++j) logp = (a_cur == j) ? lp[j] : logp;
                float adv = f0_cur;
                if (p.normalize) adv = (adv - advc[0]) * advc[1];
                if constexpr (LOSS == kLossA2C) {
                    if (valid) {                          // (statistics first: log_prob dies here) approx_kl / clip_fraction stay 0
                        float *ra = racc + rt * L::RS;
                        ra[0] += -adv * logp; ra[1] += -ent;
                    }
                    const float dlogp = -adv * p.inv_rows;
#pragma unroll
                    for (int j = 0; j < NOUT; ++j)
                        dz[j] = valid ? dlogp * ((a_cur == j ? 1.0f : 0.0f) - pr[j]) + p.ent_coef * p.inv_rows * pr[j] * (lp[j] + ent) : 0.0f;
                } else {
                    const float lr = logp - f1_cur;
                    const float ratio = __expf(lr);
                    const float lo = 1.0f - p.clip, hi = 1.0f + p.clip;
                    const float s1 = adv * ratio, s2 = adv * fminf(fmaxf(ratio, lo), hi);
                    const bool inside = (ratio >= lo) && (ratio <= hi);
                    const bool active = inside || (s1 < s2);
                    const float dlogp = active ? (-adv * ratio * p.inv_rows) : 0.0f;
#pragma unroll
                    for (int j = 0; j < NOUT; ++j)
                        dz[j] = valid ? dlogp * ((a_cur == j ? 1.0f : 0.0f) - pr[j]) + p.ent_coef * p.inv_rows * pr[j] * (lp[j] + ent) : 0.0f;
                    if (valid) {
                        float *ra = racc + rt * L::RS;
                        ra[0] += -fminf(s1, s2); ra[1] += -ent; ra[2] += (ratio - 1.0f) - lr;
                        ra[3] += (fabsf(ratio - 1.0f) > p.clip) ? 1.0f : 0.0f;
                    }
                }
            } else {
                const float dv = z[0] - f0_cur;
                dz[0] = valid ? p.vf_coef * 2.0f * dv * p.inv_rows : 0.0f;
                if (valid) racc[rt * L::RS] += dv * dv;
            }
            float v[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) v[c] = 0.0f;
#pragma unroll
            for (int a = 0; a < NOUT; ++a) {
                racc[rt * L::RS + 4 + a] += dz[a];
                v[a] = dz[a]; v[NOUT + a] = dz[a] - bf16_round(dz[a]); v[2 * NOUT + a] = dz[a];
            }
            uint8_t *dr = smem + L::dout + (rt >> 3) * ksG + (rt & 7) * 16;
            *reinterpret_cast<uint4 *>(dr) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
            *reinterpret_cast<uint4 *>(dr + ksS) = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
        }
        fence_proxy_async();
        tc_fence_before();
        worker_sync();
        TMLA_PH(6);
        // ---- M2: dH2 = DOUT . Wh -> ACC (one K=16 MMA);  dWh += H2^T . DOUT -> GWH (H2 tile and DOUT read MN-major)
        if (tid == 0) mbar_arrive(rdy);                    // -> driver: M2
        mbar_wait(bar1, ph1);
        ph1 ^= 1u;
        TMLA_PH(7);
        tc_fence_after();
        // ---- P5: dZ2 = dH2 * (1 - H2^2) -> tile (this thread overwrites its own H2 chunks; M2 has finished reading them)
        {
            const uint32_t taddr = lane_base + C_ACC + cq * 64;
            uint32_t acc[2][16];
            tmem_ld16_nowait(taddr, acc[0]);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int kb = (cq * 64 + c * 16) >> 3;
                const uint4 ha = *reinterpret_cast<const uint4 *>(trow + kb * kLBO), hb = *reinterpret_cast<const uint4 *>(trow + (kb + 1) * kLBO);
                const uint32_t h2[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
                tmem_wait_ld();
                launder16(acc[c & 1]);
                if (c < 3) tmem_ld16_nowait(taddr + (c + 1) * 16, acc[(c + 1) & 1]);
                uint32_t o[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float h0 = bf16_lo(h2[j]), h1 = bf16_hi(h2[j]);
                    o[j] = pack_bf16(__uint_as_float(acc[c & 1][2 * j]) * (1.0f - h0 * h0), __uint_as_float(acc[c & 1][2 * j + 1]) * (1.0f - h1 * h1));
                }
                *reinterpret_cast<uint4 *>(trow + kb * kLBO) = make_uint4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<uint4 *>(trow + (kb + 1) * kLBO) = make_uint4(o[4], o[5], o[6], o[7]);
            }
        }
        cp_async_wait_all();                               // this thread's pieces of the next tile's rows have landed
        fence_proxy_async();
        tc_fence_before();
        worker_sync();
        TMLA_PH(8);
        // ---- M3: dH1 = dZ2 . W2 -> ACC (W2 tile read MN-major);  db2 += dZ2^T . XB -> GB2 (its ones column is db2)
        if (tid == 0) mbar_arrive(rdy);                    // -> driver: M3 (+ dZ2 image store)
        if (has_next) {
            fetch_loss_inputs((it + 1) & 1u);              // ls is free: P4 of this tile is done
            cp_async_commit();
            layer1();                                      // next tile's layer 1 on the CUDA cores while the tensor core runs M3
        }
        mbar_wait(bar0, ph0);
        ph0 ^= 1u;
        TMLA_PH(9);
        tc_fence_after();
        mbar_wait(bar_st, phs);                            // the dZ2 image store has read the tile
        phs ^= 1u;
        worker_sync();
        TMLA_PH(10);
        // ---- P7: dZ1 = dH1 * (1 - H1^2) -> tile (H1 from the TMEM stash, 8 packed pairs per 16 accumulator columns).
        // Not software-pipelined: the next tile's H1 (32 registers) is live here and this is the register-pressure peak.
        {
            const uint32_t taddr = lane_base + C_ACC + cq * 64, saddr = lane_base + C_H1 + cq * 32;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint32_t hst[8], acc[16];
                tmem_ld8_nowait(saddr + c * 8, hst);
                tmem_ld16_nowait(taddr + c * 16, acc);
                tmem_wait_ld();
                launder16(acc);
                launder8(hst);
                uint32_t o[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float h0 = bf16_lo(hst[j]), h1 = bf16_hi(hst[j]);
                    o[j] = pack_bf16(__uint_as_float(acc[2 * j]) * (1.0f - h0 * h0), __uint_as_float(acc[2 * j + 1]) * (1.0f - h1 * h1));
                }
                const int kb = (cq * 64 + c * 16) >> 3;
                *reinterpret_cast<uint4 *>(trow + kb * kLBO) = make_uint4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<uint4 *>(trow + (kb + 1) * kLBO) = make_uint4(o[4], o[5], o[6], o[7]);
            }
        }
        cp_async_wait_all();                               // next tile's loss inputs and the index after it have landed
        fence_proxy_async();
        tc_fence_before();
        worker_sync();
        TMLA_PH(11);
        // ---- M4: dW1 | db1 += dZ1^T . [x_hi | x_lo | 1] -> GW1
        if (tid == 0) mbar_arrive(rdy);                    // -> driver: M4
    }
    if (!is_driver) { mbar_wait(bar1, ph1); tc_fence_after(); }   // the last M4
#ifdef TMLA_PHASE_CLOCKS
    if (blockIdx.x == 0 && tid == 0) for (int i = 0; i < 16; ++i) g_phase_cycles[i] += ph_acc[i];
    const long long ph_t2 = clock64();
#endif

    // ---- flush: TMEM gradient accumulators (lane = hidden unit) -> one atomic per value; scalar sums
    // (rotating the order of the accumulator groups with the CTA index, so that 148 CTAs do not queue on one cache line, was
    // measured: no gain — 402.2 vs 401.3 us per minibatch — and, inlined, it raised the tile loop's spills: +15 us)
    if (warp < 4) {
#pragma unroll
        for (int mh = 0; mh < 2; ++mh) {
            const int j = mh * 128 + rt;
            uint32_t g[16];
            tmem_ld16(lane_base + C_GWH + mh * 16, g);
#pragma unroll
            for (int a = 0; a < NOUT; ++a) atomicAdd(p.gWh + a * H + j, __uint_as_float(g[a]) + __uint_as_float(g[NOUT + a]));
            tmem_ld16(lane_base + C_GB2 + mh * 16, g);
            atomicAdd(p.gB2 + j, __uint_as_float(g[2 * D]));
            tmem_ld16(lane_base + C_GW1 + mh * 16, g);
#pragma unroll
            for (int k = 0; k < D; ++k) atomicAdd(p.gW1 + j * D + k, __uint_as_float(g[k]) + __uint_as_float(g[D + k]));
            atomicAdd(p.gB1 + j, __uint_as_float(g[2 * D]));
        }
        // stats: pg_loss, value_loss, entropy_loss, approx_kl, clip_fraction, loss
        float st_acc[4], dbh_acc[NOUT];
#pragma unroll
        for (int q = 0; q < 4; ++q) st_acc[q] = warp_sum_f(racc[rt * L::RS + q]) * p.inv_rows;
#pragma unroll
        for (int a = 0; a < NOUT; ++a) dbh_acc[a] = warp_sum_f(racc[rt * L::RS + 4 + a]);
        if (lane == 0) {
#pragma unroll
            for (int a = 0; a < NOUT; ++a) atomicAdd(p.gBh + a, dbh_acc[a]);
            if (PI) {
                atomicAdd(p.stats + 0, st_acc[0]); atomicAdd(p.stats + 2, st_acc[1]);
                atomicAdd(p.stats + 3, st_acc[2]); atomicAdd(p.stats + 4, st_acc[3]);
                atomicAdd(p.stats + 5, st_acc[0] + p.ent_coef * st_acc[1]);
            } else {
                atomicAdd(p.stats + 1, st_acc[0]); atomicAdd(p.stats + 5, p.vf_coef * st_acc[0]);
            }
        }
    }
    // a programmatic dependent must not COMPLETE before its primary: the weight-gradient launch that follows waits for this
    // grid only, and needs the policy tower's images too (returns at once: the primary finished ~150 us ago; a no-op otherwise)
    if (!PI) asm volatile("griddepcontrol.wait;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
#ifdef TMLA_PHASE_CLOCKS
    if (tid == 0) {      // whole-kernel budget: prologue / tile loop / flush, CTA 0 summed and the maximum over CTAs
        const long long ph_t3 = clock64();
        if (blockIdx.x == 0) {
            unsigned long long ph_g1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ph_g1));
            g_phase_cycles[24] += ph_g1 - ph_g0; g_phase_cycles[25] += (unsigned long long)(ph_t3 - ph_t0);
            g_phase_cycles[16] += (unsigned long long)(ph_t1 - ph_t0); g_phase_cycles[17] += (unsigned long long)(ph_t2 - ph_t1);
            g_phase_cycles[18] += (unsigned long long)(ph_t3 - ph_t2);
        }
        unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        if (blockIdx.x < 256) { g_cta_loop[2 * blockIdx.x] = (unsigned)(ph_t2 - ph_t1); g_cta_loop[2 * blockIdx.x + 1] = smid; }
        atomicMax(&g_phase_cycles[20], (unsigned long long)(ph_t1 - ph_t0)); atomicMax(&g_phase_cycles[21], (unsigned long long)(ph_t2 - ph_t1));
        atomicMax(&g_phase_cycles[22], (unsigned long long)(ph_t3 - ph_t2)); atomicMax(&g_phase_cycles[23], (unsigned long long)(ph_t3 - ph_t0));
    }
#endif
}

// --------------------------------------------------------- G[256,256] += X^T . Y  over tile images
// X (dZ2) and Y (H1) arrive as the 64 KB tile images the training kernel wrote: 128 rows x 256 columns bf16 in the
// shared-memory operand layout (16-byte chunk (r, cb) at (r/8)*4096 + cb*128 + (r%8)*16).  A 64-row half image is
// 32 KB of contiguous global memory, so one chunk = two bulk-TMA loads (cp.async.bulk, mbarrier complete_tx) into
// a 3-stage ring — no per-thread loads, no transposes: the tensor core reads both operands through MN-major
// descriptors.  Warp-specialised: one producer thread, one MMA-issuing thread, full/empty mbarriers per stage;
// 256x256 fp32 accumulators in all 512 TMEM columns; split-K over CTAs finished with red.global.add.v4.f32.
// Two independent problems (the policy and the value tower of one minibatch) can share a launch: even CTAs take
// problem 0, odd CTAs problem 1 — one kernel boundary and half as many 256 KB atomic epilogues as two launches.
static constexpr uint32_t kwChunk = 64 * H * 2;               // 32768 B: 64 rows of one operand
static constexpr uint32_t kwStage = 2 * kwChunk;              // X and Y
static constexpr int kwStages = 3;
static constexpr uint32_t kWgradTiledSmem = kwStages * kwStage + 128;   // 196736 (>= the 128 KB epilogue stage)

__global__ void __launch_bounds__(256, 1)
tc_wgrad_tiled_kernel(const __nv_bfloat16 *__restrict__ Xt0, const __nv_bfloat16 *__restrict__ Yt0, float *__restrict__ G0,
                      const __nv_bfloat16 *__restrict__ Xt1, const __nv_bfloat16 *__restrict__ Yt1, float *__restrict__ G1, int64_t nchunks,
                      int reverse, int n1, int hint) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + kwStages * kwStage);   // full[3], empty[3], done
    uint64_t *empty = full + kwStages, *done = empty + kwStages;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + kwStages * kwStage + 64);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    // the optimizer step that follows is a programmatic dependent: its small CTAs may become resident now, fetch their slice of
    // the parameters and the Adam state, and wait for this grid before touching the gradient (a no-op after an ordinary launch)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // dual launch: n1 CTAs work on problem 1, the rest on problem 0.  n1 = grid/2 interleaves them (even / odd CTAs); a smaller
    // n1 hands problem 1 — whose image tail is still L2-resident when read back to front — fewer CTAs: its CTAs are
    // spread over the grid (every CTA with blockIdx % period == period - 1 ... see `second`)
    const bool dual = Xt1 != nullptr;
    const int n0 = (int)gridDim.x - n1;
    // problem-1 CTAs are spread evenly over the grid: CTA b belongs to problem 1 iff floor((b+1)*n1/grid) > floor(b*n1/grid)
    const int before1 = dual ? (int)(((int64_t)blockIdx.x * n1) / gridDim.x) : 0;          // problem-1 CTAs with a smaller index
    const bool second = dual && (int)(((int64_t)(blockIdx.x + 1) * n1) / gridDim.x) > before1;
    const __nv_bfloat16 *Xt = second ? Xt1 : Xt0, *Yt = second ? Yt1 : Yt0;
    float *G = second ? G1 : G0;
    const int64_t first = dual ? (second ? before1 : (int64_t)blockIdx.x - before1) : blockIdx.x, stride = dual ? (second ? n1 : n0) : gridDim.x;
    if (first >= nchunks) return;

    if (warp == 0) tmem_alloc<512>(tmem_holder);
    if (tid == 32) {
        for (int s = 0; s < kwStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
    const uint32_t s_addr = smem_u32(smem);
    const int64_t my_chunks = (nchunks - first + stride - 1) / stride;

    if (tid == 0) {                                        // producer: bulk-TMA loads, one stage ahead of the ring's tail
        uint32_t pe[kwStages] = {0u, 0u, 0u};
        const uint64_t pol = l2_policy_evict_first();
        // launched as a programmatic dependent of the tower kernels: everything above ran beside their last CTAs; the images
        // are complete (and visible) once the prerequisite grids have finished (returns at once after an ordinary launch)
        asm volatile("griddepcontrol.wait;" ::: "memory");
        for (int64_t j = 0; j < my_chunks; ++j) {
            const int s = (int)(j % kwStages);
            if (j >= kwStages) { mbar_wait(empty + s, pe[s]); pe[s] ^= 1u; }   // the MMAs of chunk j-3 have read this stage
            // reverse: walk the images from their END — the tower kernel wrote them front to back, so the tail is what the
            // 126 MB L2 still holds when this kernel starts
            const int64_t c = reverse ? nchunks - 1 - (first + j * stride) : first + j * stride;
            mbar_expect_tx(full + s, kwStage);
            if (hint) {       // read-once data: do not let it push the not-yet-read tail of the images out of L2
                bulk_load_hint(s_addr + s * kwStage, Xt + c * (64 * H), kwChunk, full + s, pol);
                bulk_load_hint(s_addr + s * kwStage + kwChunk, Yt + c * (64 * H), kwChunk, full + s, pol);
            } else {
                bulk_load(s_addr + s * kwStage, Xt + c * (64 * H), kwChunk, full + s);
                bulk_load(s_addr + s * kwStage + kwChunk, Yt + c * (64 * H), kwChunk, full + s);
            }
        }
    } else if (warp_u == 1 && elect_one()) {               // MMA issuer
        uint32_t pf[kwStages] = {0u, 0u, 0u};
        const uint32_t idesc = make_idesc_major(128, 256, 1, 1);
        for (int64_t j = 0; j < my_chunks; ++j) {
            const int s = (int)(j % kwStages);
            mbar_wait(full + s, pf[s]);
            pf[s] ^= 1u;
            tc_fence_after();
            const uint32_t x_addr = s_addr + s * kwStage, y_addr = x_addr + kwChunk;
#pragma unroll
            for (int mh = 0; mh < 2; ++mh)                 // X columns 0..127 / 128..255 -> TMEM columns 0..255 / 256..511
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)             // K = 16 rows = two 8-row groups
                    umma_bf16(tmem_base + mh * 256, make_desc_raw(x_addr + mh * 16 * kLBO + kk * 2 * kSBO, kSBO, kLBO),
                              make_desc_raw(y_addr + kk * 2 * kSBO, kSBO, kLBO), idesc, (j == 0 && kk == 0) ? 0u : 1u);
            umma_commit(empty + s);
        }
        umma_commit(done);
    }
    __syncwarp();
    mbar_wait(done, 0);
    tc_fence_after();
    // epilogue: TMEM -> registers -> smem stage (fp32 [128][256], 16-byte chunks XOR-swizzled by row) ->
    // coalesced red.global.add.v4.f32
#pragma unroll 1
    for (int mh = 0; mh < 2; ++mh) {
        __syncthreads();
        {
            const int rt = (warp & 3) * 32 + lane;
            const int colbase = (warp >> 2) * 128;
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mh * 256 + colbase);
            uint8_t *srow = smem + rt * 1024;
#pragma unroll 2
            for (int c0 = 0; c0 < 128; c0 += 16) {
                uint32_t acc[16];
                tmem_ld16(taddr + c0, acc);
                const int ch = (colbase + c0) >> 2;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    *reinterpret_cast<uint4 *>(srow + (((ch + q) ^ (rt & 7)) << 4)) = make_uint4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
            }
        }
        __syncthreads();
#pragma unroll 4
        for (int i = 0; i < 16; ++i) {
            const int r = warp + 8 * i;
            float *grow = G + (int64_t)(mh * 128 + r) * H;
#pragma unroll
            for (int hseg = 0; hseg < 2; ++hseg) {
                const int ch = hseg * 32 + lane;
                const float4 v = *reinterpret_cast<const float4 *>(smem + r * 1024 + ((ch ^ (r & 7)) << 4));
                asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(grow + ch * 4), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// --------------------------------------------------------- G[256,256] += dZ2^T . H1 with H1 RECOMPUTED, not read back
// The weight-gradient GEMM is HBM-bound on its operand images (1 KB per row).  H1 = tanh(x W1^T + b1) costs 24 B of x per row and
// ~1.5 K CUDA-core cycles per 64-row chunk to recompute — this kernel's CUDA cores are idle — so only dZ2 travels through HBM:
// the tower kernel no longer writes an H1 image, and the bytes this kernel reads halve (and what is left is the image whose
// tail is L2-resident).  Layer 1 is the tower kernel's, instruction for instruction (same FFMA2 order, tanh.approx, bf16 packing):
// the recomputed operand is bit-identical to the H1 the forward pass used.
//   warps 0..15 compute H1 of chunk j into the Y half of stage j % 3 (obs rows gathered through the minibatch index, two
//               chunks of register prefetch), warps 0..7 then run the epilogue;   warp 16: bulk-TMA producer of the dZ2 chunks;
//   warp 17: MMA issuer.  full[s] counts the producer's expect_tx arrive + one arrive per compute warp.
// An experiment kept behind TMLA_WGRAD_H1=recompute (bit-identical gradients, but slower than reading the image back: see
// tmla_ppo_minibatch_bf16).
struct WgradH1Problem { const __nv_bfloat16 *dz2; const float *W1, *B1; float *G; };
template <int D>
struct WgradH1Smem {
    static constexpr uint32_t bars = kwStages * kwStage;                 // full[3], empty[3], done, tmem holder
    static constexpr uint32_t w1t = bars + 128;                          // float [D][256]
    static constexpr uint32_t b1 = w1t + D * H * 4;
    static constexpr uint32_t xs = b1 + H * 4;                           // float [64][D]
    static constexpr uint32_t total = xs + 64 * D * 4 + 16;
};
static constexpr int kWgradH1Compute = 512;                // 16 compute warps: 2 rows x 16 columns of H1 per thread and chunk
static constexpr int kWgradH1Threads = kWgradH1Compute + 64;

template <int D>
__global__ void __launch_bounds__(kWgradH1Threads, 1)
tc_wgrad_h1_kernel(const __grid_constant__ WgradH1Problem p0, const __grid_constant__ WgradH1Problem p1, const float *__restrict__ x,
                   const int32_t *__restrict__ index, int64_t M, int64_t nchunks) {
    using L = WgradH1Smem<D>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + L::bars);
    uint64_t *empty = full + kwStages, *done = empty + kwStages;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + L::bars + 64);
    float *w1t = reinterpret_cast<float *>(smem + L::w1t), *b1s = reinterpret_cast<float *>(smem + L::b1);
    float *xs = reinterpret_cast<float *>(smem + L::xs);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const bool second = blockIdx.x & 1;
    const WgradH1Problem &P = second ? p1 : p0;
    const int64_t first = blockIdx.x >> 1, stride = gridDim.x >> 1;
    if (first >= nchunks) return;

    if (warp == 0) tmem_alloc<512>(tmem_holder);
    if (tid == 32) {
        for (int s = 0; s < kwStages; ++s) { mbar_init(full + s, 1 + kWgradH1Compute / 32); mbar_init(empty + s, 1); }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (tid < kWgradH1Compute) {
        for (int e = tid; e < H * D; e += kWgradH1Compute) { const int k = e / H, j = e - k * H; w1t[e] = P.W1[j * D + k]; }
        if (tid < H) b1s[tid] = P.B1[tid];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
    const uint32_t s_addr = smem_u32(smem);
    const int64_t my_chunks = (nchunks - first + stride - 1) / stride;
    auto chunk_of = [&](int64_t j) { return nchunks - 1 - (first + j * stride); };     // back to front: the image tail is in L2

    if (warp_u == kWgradH1Compute / 32) {
        if (lane == 0) {                                   // producer: dZ2 chunks
            uint32_t pe[kwStages] = {0u, 0u, 0u};
            const uint64_t pol = l2_policy_evict_first();
            for (int64_t j = 0; j < my_chunks; ++j) {
                const int s = (int)(j % kwStages);
                if (j >= kwStages) { mbar_wait(empty + s, pe[s]); pe[s] ^= 1u; }
                mbar_expect_tx(full + s, kwChunk);
                bulk_load_hint(s_addr + s * kwStage, P.dz2 + chunk_of(j) * (64 * H), kwChunk, full + s, pol);
            }
        }
        __syncwarp();
    } else if (warp_u == kWgradH1Compute / 32 + 1) {
        if (elect_one()) {                                 // MMA issuer
            uint32_t pf[kwStages] = {0u, 0u, 0u};
            const uint32_t idesc = make_idesc_major(128, 256, 1, 1);
            for (int64_t j = 0; j < my_chunks; ++j) {
                const int s = (int)(j % kwStages);
                mbar_wait(full + s, pf[s]);
                pf[s] ^= 1u;
                tc_fence_after();
                const uint32_t x_addr = s_addr + s * kwStage, y_addr = x_addr + kwChunk;
#pragma unroll
                for (int mh = 0; mh < 2; ++mh)
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16(tmem_base + mh * 256, make_desc_raw(x_addr + mh * 16 * kLBO + kk * 2 * kSBO, kSBO, kLBO),
                                  make_desc_raw(y_addr + kk * 2 * kSBO, kSBO, kLBO), idesc, (j == 0 && kk == 0) ? 0u : 1u);
                umma_commit(empty + s);
            }
            umma_commit(done);
        }
        __syncwarp();
    } else {
        // ---- compute warps 0..15: H1 of chunk j -> Y half of stage j % 3
        constexpr int PIECES = (D + 1) / 2;                // float2 pieces per observation row (D = 7: the last piece is one float)
        const int prow = tid & 63, ppiece = tid >> 6;      // prefetch role: row of the chunk, piece index (0..7, the first PIECES load)
        const int l1row = (warp & 3) * 16 + (lane & 7), l1col = (warp >> 2) * 64 + (lane >> 3) * 16;   // rows l1row, l1row + 8
        auto load_idx = [&](int64_t j) -> int32_t {        // buffer row of chunk j's row `prow` (-1 past the end)
            if (j >= my_chunks) return -1;
            const int64_t r = chunk_of(j) * 64 + prow;
            if (r >= M) return -1;
            return index ? __ldg(index + r) : (int32_t)r;
        };
        auto load_x = [&](int32_t src) -> float2 {
            float2 v = make_float2(0.0f, 0.0f);
            if (src >= 0 && ppiece < PIECES) {
                const float *q = x + (int64_t)src * D + 2 * ppiece;
                v.x = __ldg(q);
                if (2 * ppiece + 1 < D) v.y = __ldg(q + 1);
            }
            return v;
        };
        int32_t idx1 = load_idx(1);
        float2 xv = load_x(load_idx(0));
        uint32_t pe[kwStages] = {0u, 0u, 0u};
        for (int64_t j = 0; j < my_chunks; ++j) {
            const int s = (int)(j % kwStages);
            if (ppiece < PIECES) {
                xs[prow * D + 2 * ppiece] = xv.x;
                if (2 * ppiece + 1 < D) xs[prow * D + 2 * ppiece + 1] = xv.y;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kWgradH1Compute) : "memory");
            xv = load_x(idx1);                             // rows of chunk j+1, index of chunk j+2: in flight during layer 1
            idx1 = load_idx(j + 2);
            uint32_t h1p[16];
            {
                float xr[2][D];
#pragma unroll
                for (int i = 0; i < 2; ++i)
#pragma unroll
                    for (int k = 0; k < D; ++k) xr[i][k] = xs[(l1row + 8 * i) * D + k];
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    const int col = l1col + g * 2;
                    const float2 bb = *reinterpret_cast<const float2 *>(b1s + col);
                    float2 ww[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) ww[k] = *reinterpret_cast<const float2 *>(w1t + k * H + col);
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        float2 v = bb;
#pragma unroll
                        for (int k = 0; k < D; ++k) v = __ffma2_rn(make_float2(xr[i][k], xr[i][k]), ww[k], v);
                        h1p[i * 8 + g] = pack_bf16(tanh_fast(v.x), tanh_fast(v.y));
                    }
                }
            }
            if (j >= kwStages) { mbar_wait(empty + s, pe[s]); pe[s] ^= 1u; }      // the MMAs of chunk j-3 have read this stage
            uint8_t *Ys = smem + s * kwStage + kwChunk;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                uint8_t *dst = Ys + ((l1row + 8 * i) >> 3) * kSBO + (l1col >> 3) * kLBO + (lane & 7) * 16;
                *reinterpret_cast<uint4 *>(dst) = make_uint4(h1p[i * 8], h1p[i * 8 + 1], h1p[i * 8 + 2], h1p[i * 8 + 3]);
                *reinterpret_cast<uint4 *>(dst + kLBO) = make_uint4(h1p[i * 8 + 4], h1p[i * 8 + 5], h1p[i * 8 + 6], h1p[i * 8 + 7]);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(full + s);
            asm volatile("bar.sync 1, %0;" ::"n"(kWgradH1Compute) : "memory");   // xs is rewritten at the top of the next iteration
        }
    }
    mbar_wait(done, 0);
    tc_fence_after();
    // epilogue (warps 0..7): TMEM -> registers -> smem stage (fp32 [128][256], XOR-swizzled 16-byte chunks) -> red.global.add.v4.f32
#pragma unroll 1
    for (int mh = 0; mh < 2; ++mh) {
        __syncthreads();
        if (warp < 8) {
            const int rt = (warp & 3) * 32 + lane;
            const int colbase = (warp >> 2) * 128;
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mh * 256 + colbase);
            uint8_t *srow = smem + rt * 1024;
#pragma unroll 2
            for (int c0 = 0; c0 < 128; c0 += 16) {
                uint32_t acc[16];
                tmem_ld16(taddr + c0, acc);
                const int ch = (colbase + c0) >> 2;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    *reinterpret_cast<uint4 *>(srow + (((ch + q) ^ (rt & 7)) << 4)) = make_uint4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
            }
        }
        __syncthreads();
        if (warp < 8) {
#pragma unroll 4
            for (int i = 0; i < 16; ++i) {
                const int r = warp + 8 * i;
                float *grow = P.G + (int64_t)(mh * 128 + r) * H;
#pragma unroll
                for (int hseg = 0; hseg < 2; ++hseg) {
                    const int ch = hseg * 32 + lane;
                    const float4 v = *reinterpret_cast<const float4 *>(smem + r * 1024 + ((ch ^ (r & 7)) << 4));
                    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(grow + ch * 4), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------ descriptor probe (tests only)
// One CTA, A bf16 [128][256], B bf16 [256][256] staged exactly like the production tiles:
//   mode 0: out[128][256] = A . B^T   (both K-major)
//   mode 1: out[128][256] = A . B     (B tile read through the MN-major descriptor)
//   mode 2: out[256][256] = A^T . B[0:128]   (both MN-major; the wgrad shape)
__global__ void __launch_bounds__(256, 1)
tc_probe_kernel(const __nv_bfloat16 *__restrict__ A, const __nv_bfloat16 *__restrict__ B, float *__restrict__ out, int mode) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *Ws = smem, *As = smem + kWBytes;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kWBytes + kABytes);
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + kWBytes + kABytes + 16);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc<512>(tmem_holder);
    if (tid == 32) { mbar_init(bar, 1); fence_barrier_init(); }
    stage_rows<H>(Ws, B, 0, H);
    for (int i = 0; i < 16; ++i) {
        const int r = warp + 8 * i;
        *reinterpret_cast<uint4 *>(As + (r >> 3) * kaSBO + lane * kaLBO + (r & 7) * 16) = __ldg(reinterpret_cast<const uint4 *>(A + r * H) + lane);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    const uint32_t a_addr = smem_u32(As), w_addr = smem_u32(Ws);
    if (tid == 0) {
        if (mode == 0) {
            for (int kk = 0; kk < 16; ++kk)
                umma_bf16(tmem_base, make_desc_raw(a_addr + kk * 2 * kaLBO, kaLBO, kaSBO), make_desc_raw(w_addr + kk * 2 * kLBO, kLBO, kSBO),
                          make_idesc_major(128, 256, 0, 0), kk > 0);
        } else if (mode == 1) {
            for (int kk = 0; kk < 16; ++kk)
                umma_bf16(tmem_base, make_desc_raw(a_addr + kk * 2 * kaLBO, kaLBO, kaSBO), make_desc_raw(w_addr + kk * 2 * kSBO, kSBO, kLBO),
                          make_idesc_major(128, 256, 0, 1), kk > 0);
        } else {
            for (int mh = 0; mh < 2; ++mh)
                for (int kk = 0; kk < 8; ++kk)
                    umma_bf16(tmem_base + mh * 256, make_desc_raw(a_addr + mh * 16 * kaLBO + kk * 2 * kaSBO, kaSBO, kaLBO),
                              make_desc_raw(w_addr + kk * 2 * kSBO, kSBO, kLBO), make_idesc_major(128, 256, 1, 1), kk > 0);
        }
        umma_commit(bar);
    }
    mbar_wait(bar, 0);
    tc_fence_after();
    const int rt = (warp & 3) * 32 + lane, colbase = (warp >> 2) * 128;
    for (int mh = 0; mh < (mode == 2 ? 2 : 1); ++mh)
        for (int c = 0; c < 8; ++c) {
            uint32_t acc[16];
            tmem_ld16(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mh * 256 + colbase + c * 16), acc);
            for (int j = 0; j < 16; ++j) out[(int64_t)(mh * 128 + rt) * H + colbase + c * 16 + j] = __uint_as_float(acc[j]);
        }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}


// ------------------------------------------------------------------ tensor pipe / TMEM overlap probe (measurement hook)
// One CTA.  Warp 4 issues `n_mma` x (M128 N=`n` K16) MMAs into TMEM columns [0, n); warps 0..3 read `n_ld` x 16 columns of
// columns [256, 512) with tcgen05.ld.  clock64 around each role, alone and together:
//   out[0] MMAs alone (issue -> commit observed)   out[1] loads alone   out[2] MMAs with the loads running   out[3] loads while the
//   MMAs are in flight (started after the MMAs were issued)   out[4] cycles the issuing lane spent inside the tcgen05.mma instructions
// Answers whether a TMEM-reading CUDA-core phase can overlap MMAs that are already queued (DESIGN.md §5a).
__global__ void __launch_bounds__(160, 1)
tc_overlap_probe_kernel(unsigned long long *out, int n, int n_mma, int n_ld) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *Ws = smem, *As = smem + kWBytes;                       // operands: whatever the shared memory holds (timing only)
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kWBytes + 128 * 512);
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(bar + 4);
    volatile int *go = reinterpret_cast<volatile int *>(bar + 6);
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < (int)(kWBytes + 128 * 512) / 4; i += blockDim.x) reinterpret_cast<uint32_t *>(smem)[i] = 0x3c003c00u;
    if (warp == 0) tmem_alloc<512>(tmem_holder);
    if (tid == 32) { mbar_init(bar, 1); mbar_init(bar + 1, 1); fence_barrier_init(); *go = 0; }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    const uint32_t a_addr = smem_u32(As), w_addr = smem_u32(Ws);
    const uint32_t idesc = make_idesc_major(128, n, 0, 0);
    auto issue = [&](uint64_t *b) {
        long long inside = 0;
        for (int i = 0; i < n_mma; ++i) {
            const int kk = i & 15;
            const long long c0 = clock64();
            umma_bf16(tmem_base, make_desc_raw(a_addr + kk * 2 * kLBO, kLBO, kSBO), make_desc_raw(w_addr + kk * 2 * kLBO, kLBO, kSBO), idesc, i > 0 ? 1u : 0u);
            inside += clock64() - c0;
        }
        umma_commit(b);
        return inside;
    };
    auto loads = [&]() {
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + 256u;
        uint32_t acc[16], sink = 0;
        for (int i = 0; i < n_ld; ++i) {
            tmem_ld16(taddr + (i & 15) * 16, acc);
#pragma unroll
            for (int j = 0; j < 16; ++j) sink ^= acc[j];
        }
        return sink;
    };
    // (a) MMAs alone
    if (warp == 4 && elect_one()) {
        const long long t0 = clock64();
        const long long inside = issue(bar);
        mbar_wait(bar, 0);
        out[0] = (unsigned long long)(clock64() - t0);
        out[4] = (unsigned long long)inside;
    }
    __syncthreads();
    // (b) loads alone
    if (warp < 4) {
        const long long t0 = clock64();
        const uint32_t sink = loads();
        const long long t1 = clock64();
        if (tid == 0) out[1] = (unsigned long long)(t1 - t0);
        if (sink == 0x12345678u) out[7] = sink;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // (c) together: the loads start once the issuing lane has issued its first MMA
    if (warp == 4) {
        if (elect_one()) {
            const long long t0 = clock64();
            umma_bf16(tmem_base, make_desc_raw(a_addr, kLBO, kSBO), make_desc_raw(w_addr, kLBO, kSBO), idesc, 0u);
            *go = 1;
            issue(bar + 1);
            mbar_wait(bar + 1, 0);
            out[2] = (unsigned long long)(clock64() - t0);
        }
        __syncwarp();
    } else {
        while (*go == 0) { }
        const long long t0 = clock64();
        const uint32_t sink = loads();
        const long long t1 = clock64();
        if (tid == 0) out[3] = (unsigned long long)(t1 - t0);
        if (sink == 0x12345678u) out[7] = sink;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------ host side
static int sm_count_train() {
    static int n = 0;
    if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = 148; }
    return n;
}

// Xt, Yt: tile images covering `rows_padded` rows (a multiple of 128); Xt1/Yt1/G1 = an optional second problem of the same size
static int wgrad_reverse() {      // TMLA_WGRAD_REV=0 restores front-to-back reads (A/B)
    static const int r = [] { const char *e = getenv("TMLA_WGRAD_REV"); return (e && !strcmp(e, "0")) ? 0 : 1; }();
    return r;
}
static int tc_wgrad_tiled_launch(const void *Xt, const void *Yt, float *G, int64_t rows_padded, cudaStream_t st,
                                 const void *Xt1 = nullptr, const void *Yt1 = nullptr, float *G1 = nullptr, bool overlap_prev = false) {
    static int attr_done = 0;
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_wgrad_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWgradTiledSmem));
        attr_done = 1;
    }
    const int64_t nchunks = rows_padded / 64;
    unsigned grid = (unsigned)std::min<int64_t>(Xt1 ? 2 * nchunks : nchunks, sm_count_train());
    if (Xt1) grid &= ~1u;
    // share of the CTAs given to problem 1 (the tower that ran LAST: its image tail is L2-resident): TMLA_WGRAD_N1 per 148 CTAs
    static const int n1_of_148 = [] { const char *e = getenv("TMLA_WGRAD_N1"); return e ? atoi(e) : 74; }();
    static const int wgrad_hint = [] { const char *e = getenv("TMLA_WGRAD_HINT"); return e ? atoi(e) : 1; }();
    int n1 = Xt1 ? std::max(1, std::min((int)grid - 1, (int)((int64_t)grid * n1_of_148 / 148))) : 0;
    if (overlap_prev) {                                    // programmatic dependent of the tower kernel before it (see tower_train_launch_t)
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = kWgradTiledSmem; cfg.stream = st;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        TMLA_CUDA(cudaLaunchKernelEx(&cfg, tc_wgrad_tiled_kernel, (const __nv_bfloat16 *)Xt, (const __nv_bfloat16 *)Yt, G, (const __nv_bfloat16 *)Xt1,
                                     (const __nv_bfloat16 *)Yt1, G1, nchunks, wgrad_reverse(), n1, wgrad_hint));
    } else {
        tc_wgrad_tiled_kernel<<<grid, 256, kWgradTiledSmem, st>>>((const __nv_bfloat16 *)Xt, (const __nv_bfloat16 *)Yt, G,
                                                                  (const __nv_bfloat16 *)Xt1, (const __nv_bfloat16 *)Yt1, G1, nchunks, wgrad_reverse(), n1, wgrad_hint);
    }
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

template <int D>
static int wgrad_h1_launch_t(const WgradH1Problem &a, const WgradH1Problem &b, const float *x, const int32_t *index, int64_t M, int64_t rows_padded,
                             cudaStream_t st) {
    static int attr_done = 0;
    constexpr uint32_t smem = WgradH1Smem<D>::total;
    static_assert(smem <= 232448, "wgrad (recomputed H1) exceeds the 227 KB shared-memory limit");
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_wgrad_h1_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = 1;
    }
    const int64_t nchunks = rows_padded / 64;
    unsigned grid = (unsigned)std::min<int64_t>(2 * nchunks, sm_count_train()) & ~1u;
    tc_wgrad_h1_kernel<D><<<grid, kWgradH1Threads, smem, st>>>(a, b, x, index, M, nchunks);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

template <int D, int NOUT, int LOSS = kLossPPO>
static int tower_train_launch_t(const TowerTrainArgs &a, cudaStream_t st, bool overlap_prev) {
    static int attr_done = 0;
    constexpr uint32_t smem = TrainSmem<D, NOUT>::total;
    static_assert(smem <= 232448, "fused tower training kernel exceeds the 227 KB shared-memory limit");
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_tower_train_kernel<D, NOUT, LOSS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = 1;
    }
    const unsigned grid = (unsigned)std::min<int64_t>((a.M + 127) / 128, sm_count_train());
    if (overlap_prev) {
        // programmatic dependent launch: this kernel needs nothing the previous launch on the stream (the other tower of the
        // same minibatch, which triggers at its start) produces, so its CTAs may start on every SM the previous kernel's CTA has
        // left — the launch gap, the prologue and the previous kernel's last-round imbalance overlap instead of adding up
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kTrainThreads + 32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        TMLA_CUDA(cudaLaunchKernelEx(&cfg, tc_tower_train_kernel<D, NOUT, LOSS>, a));
    } else {
        tc_tower_train_kernel<D, NOUT, LOSS><<<grid, kTrainThreads + 32, smem, st>>>(a);
    }
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

extern "C" {

int tmla_ppo_minibatch_supported(int obs_dim, int hidden, int n_actions) {
    return (hidden == H && ((obs_dim == 6 && n_actions == 5) || (obs_dim == 4 && (n_actions == 4 || n_actions == 5)) ||
                            (obs_dim == 7 && n_actions == 3))) ? 1 : 0;
}

int64_t tmla_ppo_minibatch_scratch(int hidden, int64_t rows) { return 4 * ((rows + 127) / 128 * 128) * (int64_t)hidden; }

}  // extern "C"

template <int D, int A>
static int policy_tower_launch(const TowerTrainArgs &a, cudaStream_t st, int loss) {
    return loss == kLossA2C ? tower_train_launch_t<D, A, kLossA2C>(a, st, false) : tower_train_launch_t<D, A>(a, st, false);
}

// one fused batch of either loss: the policy tower with PPO's or A2C's loss, the shared value tower, the weight-gradient GEMMs
static int tower_batch_launch(int loss, const char *fn, const float *params, const void *wpack, int obs_dim, int hidden, int n_actions,
                              const float *obs, const int32_t *index, int64_t rows, int64_t global_rows, const int32_t *actions,
                              const float *advantages, const float *old_logp, const float *returns, const double *adv_sums,
                              int normalize_advantage, float clip_range, float ent_coef, float vf_coef, float *grads,
                              void *scratch, float *stats_out, float *logits_out, float *values_out, int flags, void *stream) {
    TMLA_REQUIRE(params && wpack && obs && actions && advantages && (old_logp || loss == kLossA2C) && returns && grads && scratch && stats_out,
                 "NULL buffer");
    TMLA_REQUIRE(rows > 0 && global_rows >= rows, "bad row counts");
    TMLA_REQUIRE(!normalize_advantage || adv_sums, "adv_sums required when normalising");
    if (!tmla_ppo_minibatch_supported(obs_dim, hidden, n_actions)) {
        tmla_set_error("%s: fused path covers hidden=256 with (obs_dim, actions) = (6,5), (4,5), (4,4), (7,3) (got %d/%d/%d)", fn, obs_dim, hidden, n_actions);
        return TMLA_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
    if (!(flags & TMLA_MB_GRADS_ZEROED)) TMLA_CUDA(cudaMemsetAsync(grads, 0, sizeof(float) * o.total, st));
    if (!(flags & TMLA_MB_ACCUMULATE_STATS)) TMLA_CUDA(cudaMemsetAsync(stats_out, 0, 8 * sizeof(float), st));
    const int64_t rows_padded = (rows + 127) / 128 * 128;  // whole tile images; rows past `rows` contribute exact zeros (dZ2 = 0)
    // scratch: H1 and dZ2 tile images of both towers (one weight-gradient launch covers the two towers)
    __nv_bfloat16 *img[2][2];
    for (int t = 0; t < 2; ++t) for (int q = 0; q < 2; ++q) img[t][q] = reinterpret_cast<__nv_bfloat16 *>(scratch) + (int64_t)(2 * t + q) * rows_padded * H;
    static const bool interleave = [] { const char *e = getenv("TMLA_WGRAD"); return e && !strcmp(e, "interleave"); }();   // A/B: wgrad right after each tower
    // TMLA_WGRAD_H1=recompute: the weight-gradient kernel recomputes H1 from the observations, so that no H1 image is written
    // or read (tc_wgrad_h1_kernel).  Measured on B200, one 262 144-row ball3d minibatch (2 towers + wgrad): 413.5 us with 8
    // compute warps, 431.6 us with 16, against 407-410 us for the default (both operands as tile images): the image read it
    // saves (134 MB per tower, mostly L2 hits on the tail) is cheaper than 2 x 262 144 x 256 tanh on this kernel's CUDA cores.
    static const bool h1_recompute = [] { const char *e = getenv("TMLA_WGRAD_H1"); return e && !strcmp(e, "recompute"); }();
    const bool recompute = h1_recompute && !interleave;
    static const bool pdl_on = [] { const char *e = getenv("TMLA_PDL"); return !(e && !strcmp(e, "0")); }();   // TMLA_PDL=0: ordinary launches (A/B)
    const bool pdl = pdl_on && !interleave;
    static const bool pdl_w = [] { const char *e = getenv("TMLA_PDL"); return !(e && !strcmp(e, "1")); }();   // TMLA_PDL=1: towers only
    const bool pdl_wgrad = pdl && pdl_w;
    for (int t = 0; t < 2; ++t) {
        __nv_bfloat16 *h1 = img[t][0], *dz2 = img[t][1];
        TowerTrainArgs a;
        a.W1 = params + o.w1[t]; a.B1 = params + o.b1[t];
        a.W2 = reinterpret_cast<const __nv_bfloat16 *>(wpack) + (int64_t)(4 + t) * H * H;
        a.B2 = params + o.b2[t]; a.Wh = params + o.wh[t]; a.Bh = params + o.bh[t];
        a.x = obs; a.index = index; a.M = rows;
        a.actions = actions; a.adv = advantages; a.old_logp = old_logp; a.returns = returns;
        a.adv_sums = adv_sums; a.normalize = normalize_advantage;
        a.clip = clip_range; a.ent_coef = ent_coef; a.vf_coef = vf_coef; a.inv_rows = (float)(1.0 / (double)global_rows);
        a.h1_out = recompute ? nullptr : h1; a.dz2_out = dz2; a.out = t == 0 ? logits_out : values_out;
        a.gW1 = grads + o.w1[t]; a.gB1 = grads + o.b1[t]; a.gB2 = grads + o.b2[t]; a.gWh = grads + o.wh[t]; a.gBh = grads + o.bh[t];
        a.stats = stats_out;
        int rc;
        if (obs_dim == 6) rc = t == 0 ? policy_tower_launch<6, 5>(a, st, loss) : tower_train_launch_t<6, 1>(a, st, pdl);
        else if (obs_dim == 7) rc = t == 0 ? policy_tower_launch<7, 3>(a, st, loss) : tower_train_launch_t<7, 1>(a, st, pdl);
        else if (n_actions == 5) rc = t == 0 ? policy_tower_launch<4, 5>(a, st, loss) : tower_train_launch_t<4, 1>(a, st, pdl);
        else rc = t == 0 ? policy_tower_launch<4, 4>(a, st, loss) : tower_train_launch_t<4, 1>(a, st, pdl);
        if (rc) return rc;
        if (interleave) { rc = tc_wgrad_tiled_launch(img[t][1], img[t][0], grads + o.w2[t], rows_padded, st); if (rc) return rc; }
    }
    if (interleave) return TMLA_OK;
    if (recompute) {
        const WgradH1Problem pa{img[0][1], params + o.w1[0], params + o.b1[0], grads + o.w2[0]}, pb{img[1][1], params + o.w1[1], params + o.b1[1], grads + o.w2[1]};
        if (obs_dim == 6) return wgrad_h1_launch_t<6>(pa, pb, obs, index, rows, rows_padded, st);
        if (obs_dim == 7) return wgrad_h1_launch_t<7>(pa, pb, obs, index, rows, rows_padded, st);
        return wgrad_h1_launch_t<4>(pa, pb, obs, index, rows, rows_padded, st);
    }
    return tc_wgrad_tiled_launch(img[0][1], img[0][0], grads + o.w2[0], rows_padded, st, img[1][1], img[1][0], grads + o.w2[1], pdl_wgrad);
}

extern "C" {

int tmla_ppo_minibatch_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *obs,
                            const int32_t *index, int64_t rows, int64_t global_rows, const int32_t *actions,
                            const float *advantages, const float *old_logp, const float *returns, const double *adv_sums,
                            int normalize_advantage, float clip_range, float ent_coef, float vf_coef, float *grads,
                            void *scratch, float *stats_out, float *logits_out, float *values_out, int flags, void *stream) {
    return tower_batch_launch(kLossPPO, "tmla_ppo_minibatch_bf16", params, wpack, obs_dim, hidden, n_actions, obs, index, rows, global_rows,
                              actions, advantages, old_logp, returns, adv_sums, normalize_advantage, clip_range, ent_coef, vf_coef, grads,
                              scratch, stats_out, logits_out, values_out, flags, stream);
}

int tmla_a2c_batch_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *obs,
                        const int32_t *index, int64_t rows, int64_t global_rows, const int32_t *actions, const float *advantages,
                        const float *returns, const double *adv_sums, int normalize_advantage, float ent_coef, float vf_coef,
                        float *grads, void *scratch, float *stats_out, float *logits_out, float *values_out, int flags, void *stream) {
    return tower_batch_launch(kLossA2C, "tmla_a2c_batch_bf16", params, wpack, obs_dim, hidden, n_actions, obs, index, rows, global_rows,
                              actions, advantages, nullptr, returns, adv_sums, normalize_advantage, 0.0f, ent_coef, vf_coef, grads,
                              scratch, stats_out, logits_out, values_out, flags, stream);
}

int tmla_tc_wgrad_tiled(const void *Xt, const void *Yt, float *G, int64_t rows_padded, void *stream) {
    TMLA_REQUIRE(Xt && Yt && G && rows_padded > 0 && rows_padded % 128 == 0, "bad arguments (rows_padded must be a positive multiple of 128)");
    return tc_wgrad_tiled_launch(Xt, Yt, G, rows_padded, (cudaStream_t)stream);
}

#ifdef TMLA_PHASE_CLOCKS
int tmla_debug_phase_cycles(unsigned long long *out32, int reset) {      // debug builds only; not part of include/tmla.h
    if (out32) TMLA_CUDA(cudaMemcpyFromSymbol(out32, g_phase_cycles, sizeof(g_phase_cycles)));
    if (out32 && reset == 2) { TMLA_CUDA(cudaMemcpyFromSymbol(out32, g_cta_loop, sizeof(g_cta_loop))); return TMLA_OK; }
    if (reset) { unsigned long long z[32] = {0}; TMLA_CUDA(cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z))); }
    return TMLA_OK;
}
#endif

int tmla_tc_overlap_probe(uint64_t *out8, int n, int n_mma, int n_ld, void *stream) {
    TMLA_REQUIRE(out8 && n >= 16 && n <= 256 && n % 16 == 0 && n_mma > 0 && n_ld > 0, "bad arguments");
    static int attr_done = 0;
    const int smem = (int)(kWBytes + 128 * 512 + 128);
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_overlap_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done = 1;
    }
    TMLA_CUDA(cudaMemsetAsync(out8, 0, 8 * sizeof(uint64_t), (cudaStream_t)stream));
    tc_overlap_probe_kernel<<<1, 160, smem, (cudaStream_t)stream>>>((unsigned long long *)out8, n, n_mma, n_ld);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int tmla_tc_probe(const void *A, const void *B, float *out, int mode, void *stream) {
    TMLA_REQUIRE(A && B && out && mode >= 0 && mode <= 2, "bad arguments");
    static int attr_done = 0;
    const int smem = (int)(kWBytes + kABytes + 64);
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done = 1;
    }
    tc_probe_kernel<<<1, 256, smem, (cudaStream_t)stream>>>((const __nv_bfloat16 *)A, (const __nv_bfloat16 *)B, out, mode);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

}  // extern "C"
