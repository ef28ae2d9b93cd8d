// ppo_kernels.cu — the non-GEMM half of SB3's PPO update, hand-written for sm_100a:
//   K6  gae_kernel            RolloutBuffer.compute_returns_and_advantage   (buffers.py, SB3 2.9.0)
//   -   permutation_kernel    RolloutBuffer.get  (np.random.permutation + swapaxes flatten)
//   K7  adv_stats_kernel      advantages.mean()/.std() of PPO.train (warp-shuffle reductions)
//   K8  ppo_loss_kernel       clipped surrogate + value MSE + entropy, forward AND backward (A2C.train: plain policy gradient)
//   K11 gradnorm/adam kernels clip_grad_norm_ + Adam.step
//   -   bootstrap_add_kernel  collect_rollouts' `rewards[i] += gamma * V(terminal_obs)`
// Reached in the reference from backend/mlagents/training.py:150,166 with the hyper-parameters of
// training.py:379-389.  SB3 is a pinned third-party dependency (backend/uv.lock:1686-1688), not in the
// reference tree: the algorithm is restated from its published source; oracle/ppo_oracle.py is the CPU twin.
// All of these are HBM-bound streaming kernels.
#include <algorithm>
#include <stdlib.h>
#include "common.cuh"
#include "philox.cuh"
#include "mlp_common.cuh"
#include <cuda_bf16.h>

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------------------ GAE
// One thread per env walks T backwards; rows of the [T,n] buffers are contiguous over envs, so every
// load/store is coalesced.  Operation order and roundings are NumPy's (SURVEY.md A.3):
//   delta = f32(f32(r + f32(f32(g*nv)*nnt)) - V) ;  last = f32(delta + f32(f32(gl*nnt)*last)),  gl = f32(gamma*lambda in double)
template <int UNROLL>
__global__ void __launch_bounds__(128)
gae_kernel(const float *__restrict__ rewards, const float *__restrict__ values, const uint8_t *__restrict__ dones,
           const float *__restrict__ last_values, float g, float gl, int T, int64_t n,
           float *__restrict__ adv, float *__restrict__ ret) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float last = 0.0f;
    float next_v = last_values[i];
    int t = T - 1;
    // Only the arithmetic is sequential; the loads are not.  Software pipeline: the UNROLL x 3 loads of the NEXT group are
    // issued before the current group is evaluated, so 2 x UNROLL rows per thread are in flight (65 536 threads alone
    // cannot cover the HBM latency otherwise: UNROLL 8 without the pipeline reached 61 % of the measured peak).
    float ra[UNROLL], va[UNROLL], rb[UNROLL], vb[UNROLL];   // two register buffers, indexed statically (ping-pong by code position)
    uint8_t da[UNROLL], db[UNROLL];
    auto load_group = [&](float (&r)[UNROLL], float (&v)[UNROLL], uint8_t (&d)[UNROLL], int t0) {
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int64_t off = (int64_t)(t0 - u) * n + i;
            r[u] = __ldcs(rewards + off);
            v[u] = __ldcs(values + off);
            d[u] = __ldcs(dones + off);
        }
    };
    auto eval_group = [&](const float (&r)[UNROLL], const float (&v)[UNROLL], const uint8_t (&d)[UNROLL], int t0) {
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const float nnt = __fsub_rn(1.0f, (float)d[u]);
            const float delta = __fsub_rn(__fadd_rn(r[u], __fmul_rn(__fmul_rn(g, next_v), nnt)), v[u]);
            last = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nnt), last));
            const int64_t off = (int64_t)(t0 - u) * n + i;
            __stcs(adv + off, last);
            __stcs(ret + off, __fadd_rn(last, v[u]));
            next_v = v[u];
        }
    };
    if (t >= UNROLL - 1) load_group(ra, va, da, t);
    while (t >= UNROLL - 1) {
        const bool more_b = t - UNROLL >= UNROLL - 1;
        if (more_b) load_group(rb, vb, db, t - UNROLL);
        eval_group(ra, va, da, t);
        t -= UNROLL;
        if (!more_b) break;
        const bool more_a = t - UNROLL >= UNROLL - 1;
        if (more_a) load_group(ra, va, da, t - UNROLL);
        eval_group(rb, vb, db, t);
        t -= UNROLL;
        if (!more_a) break;
    }
    for (; t >= 0; --t) {
        const int64_t off = (int64_t)t * n + i;
        const float rr = rewards[off], vv = values[off];
        const float nnt = __fsub_rn(1.0f, (float)dones[off]);
        const float delta = __fsub_rn(__fadd_rn(rr, __fmul_rn(__fmul_rn(g, next_v), nnt)), vv);
        last = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nnt), last));
        adv[off] = last;
        ret[off] = __fadd_rn(last, vv);
        next_v = vv;
    }
}

// --------------------------------------------------------------------------- minibatch permutation
__host__ __device__ __forceinline__ uint32_t perm_mix(uint32_t v) {
    v *= 0x9E3779B1u; v ^= v >> 15; v *= 0x85EBCA77u; v ^= v >> 13;
    return v;
}
// keyed 6-round Feistel network on 2*half bits + cycle walking = a bijection of [0,total)
__host__ __device__ __forceinline__ uint64_t perm_index(uint64_t x, uint64_t total, int half, uint4 key) {
    const uint32_t mask = (half >= 32) ? 0xFFFFFFFFu : ((1u << half) - 1u);
    const uint32_t k[4] = {key.x, key.y, key.z, key.w};
    do {
        uint32_t L = (uint32_t)(x >> half), R = (uint32_t)x & mask;
#pragma unroll
        for (int r = 0; r < 6; ++r) {                       // rounds 4, 5 reuse keys 0, 1 with a round constant
            const uint32_t F = perm_mix(R ^ k[r & 3] ^ (r >= 4 ? 0x9E3779B9u : 0u)) & mask;
            const uint32_t nl = R;
            R = L ^ F;
            L = nl;
        }
        x = ((uint64_t)L << half) | R;
    } while (x >= total);
    return x;
}
__global__ void permutation_kernel(uint4 key, int64_t total, int half, int T, int64_t n, int32_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint64_t s = perm_index((uint64_t)i, (uint64_t)total, half, key);   // SB3 flat index env*T + t
    const int64_t env = (int64_t)(s / (uint64_t)T), t = (int64_t)(s % (uint64_t)T);
    out[i] = (int32_t)(t * n + env);
}

// ------------------------------------------------------------------------------- advantage stats
__global__ void __launch_bounds__(256)
adv_stats_kernel(const float *__restrict__ adv, const int32_t *__restrict__ index, int64_t rows, double *sums) {
    __shared__ double sh[2][8];
    double s = 0.0, ss = 0.0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        const double a = (double)adv[index ? index[r] : r];
        s += a; ss += a * a;
    }
    s = warp_sum(s); ss = warp_sum(ss);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { sh[0][w] = s; sh[1][w] = ss; }
    __syncthreads();
    if (w == 0) {
        s = l < 8 ? sh[0][l] : 0.0; ss = l < 8 ? sh[1][l] : 0.0;
        s = warp_sum(s); ss = warp_sum(ss);
        if (l == 0) {
            atomicAdd(sums + 0, s); atomicAdd(sums + 1, ss);
            if (blockIdx.x == 0) atomicAdd(sums + 2, (double)rows);
        }
    }
}

// all minibatches of an epoch in one launch: blockIdx.y = minibatch, rows [mb*mb_rows, min(total, (mb+1)*mb_rows))
// DET: `sums` is double[n_mb][gridDim.x][2]: each block stores its (sum, sum of squares); adv_stats_det_reduce_kernel adds them
template <bool DET = false>
__global__ void __launch_bounds__(256)
adv_stats_batched_kernel(const float *__restrict__ adv, const int32_t *__restrict__ index, int64_t total, int64_t mb_rows, double *sums) {
    __shared__ double sh[2][8];
    const int64_t lo = (int64_t)blockIdx.y * mb_rows, hi = min(total, lo + mb_rows);
    double s = 0.0, ss = 0.0;
    for (int64_t r = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < hi; r += (int64_t)gridDim.x * blockDim.x) {
        const double a = (double)adv[index ? index[r] : r];
        s += a; ss += a * a;
    }
    s = warp_sum(s); ss = warp_sum(ss);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { sh[0][w] = s; sh[1][w] = ss; }
    __syncthreads();
    if (w == 0) {
        s = l < 8 ? sh[0][l] : 0.0; ss = l < 8 ? sh[1][l] : 0.0;
        s = warp_sum(s); ss = warp_sum(ss);
        if (l == 0) {
            if constexpr (DET) {
                double *o = sums + 2 * ((int64_t)blockIdx.y * gridDim.x + blockIdx.x);
                o[0] = s; o[1] = ss;
                return;
            }
            double *o = sums + 3 * blockIdx.y;
            atomicAdd(o + 0, s); atomicAdd(o + 1, ss);
            if (blockIdx.x == 0) atomicAdd(o + 2, (double)(hi - lo));
        }
    }
}
// one warp per minibatch: lane l adds the partials of blocks l, l+32, ... in order, then a fixed butterfly
__global__ void __launch_bounds__(32)
adv_stats_det_reduce_kernel(const double *__restrict__ part, int gx, int64_t total, int64_t mb_rows, double *__restrict__ sums) {
    const int l = threadIdx.x;
    const double *p = part + 2 * (int64_t)blockIdx.x * gx;
    double s = 0.0, ss = 0.0;
    for (int b = l; b < gx; b += 32) { s += p[2 * b]; ss += p[2 * b + 1]; }
    s = warp_sum(s); ss = warp_sum(ss);
    if (l == 0) {
        const int64_t lo = (int64_t)blockIdx.x * mb_rows, hi = min(total, lo + mb_rows);
        double *o = sums + 3 * blockIdx.x;
        o[0] = s; o[1] = ss; o[2] = (double)(hi - lo);
    }
}

// ------------------------------------------------------------------------------------ PPO loss
// One thread per sample of the minibatch.  Everything SB3's PPO.train does between evaluate_actions
// and loss.backward() for Categorical policies, with the analytic gradient of
//   loss = -mean(min(A r, A clip(r))) + ent_coef * -mean(H) + vf_coef * mean((R - V)^2)
// written straight into dlogits / dvalues (scaled by 1/global_rows).  A2C (SB3 2.9.0 a2c.py) replaces the surrogate by
//   -mean(A log pi(a|s))  (no ratio, no clip, no old_logp; approx_kl / clip_fraction stay 0)
// DET: `stats` is float[gridDim.x][8]: block b stores its six sums in row b (block 0 also mean / std in slots 6, 7), summed in
// block order by det_reduce_kernel
enum { kLossPPO = 0, kLossA2C = 1 };
template <int A, int LOSS = kLossPPO, bool DET = false>
__global__ void __launch_bounds__(256)
ppo_loss_kernel(const float *__restrict__ logits, const float *__restrict__ values, const int32_t *__restrict__ actions,
                const float *__restrict__ advantages, const float *__restrict__ old_logp, const float *__restrict__ returns,
                const int32_t *__restrict__ index, int64_t rows, double inv_rows, const double *__restrict__ adv_sums,
                int normalize, float clip, float ent_coef, float vf_coef, float *__restrict__ dlogits,
                float *__restrict__ dvalues, float *stats) {
    __shared__ float sh[5][8];
    float mean = 0.0f, inv_std = 1.0f;
    if (normalize) {   // (adv - mean) / (std + 1e-8), std unbiased (torch.Tensor.std)
        const double cnt = adv_sums[2], m = adv_sums[0] / cnt;
        double var = (adv_sums[1] - adv_sums[0] * m) / (cnt - 1.0);
        var = var > 0.0 ? var : 0.0;
        mean = (float)m;
        inv_std = 1.0f / ((float)sqrt(var) + 1e-8f);
        if (blockIdx.x == 0 && threadIdx.x == 0) { stats[6] = mean; stats[7] = (float)sqrt(var); }
    }
    const float invB = (float)inv_rows;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // pg, vl, ent, kl, clipfrac
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < rows) {
        const int64_t src = index ? index[r] : r;
        float z[A], lp[A], p[A];
#pragma unroll
        for (int j = 0; j < A; ++j) z[j] = logits[r * A + j];
        float m = z[0];
#pragma unroll
        for (int j = 1; j < A; ++j) m = fmaxf(m, z[j]);
        float S = 0.0f;
#pragma unroll
        for (int j = 0; j < A; ++j) { p[j] = expf(z[j] - m); S += p[j]; }
        const float logS = logf(S), invS = 1.0f / S;
        float ent = 0.0f;
#pragma unroll
        for (int j = 0; j < A; ++j) { lp[j] = (z[j] - m) - logS; p[j] *= invS; ent -= p[j] * lp[j]; }
        const int a = actions[src];
        float logp = lp[0];
#pragma unroll
        for (int j = 1; j < A; ++j) logp = (a == j) ? lp[j] : logp;
        float adv = advantages[src];
        if (normalize) adv = (adv - mean) * inv_std;
        if constexpr (LOSS == kLossA2C) {
            const float dlogp = -adv * invB;
            const float v = values[r], R = returns[src];
            const float dv = v - R;
            dvalues[r] = vf_coef * 2.0f * dv * invB;
#pragma unroll
            for (int j = 0; j < A; ++j)
                dlogits[r * A + j] = dlogp * ((a == j ? 1.0f : 0.0f) - p[j]) + ent_coef * invB * p[j] * (lp[j] + ent);
            acc[0] = -adv * logp;
            acc[1] = dv * dv;
            acc[2] = -ent;
        } else {
            const float lr = logp - old_logp[src];
            const float ratio = expf(lr);
            const float lo = 1.0f - clip, hi = 1.0f + clip;
            const float s1 = adv * ratio, s2 = adv * fminf(fmaxf(ratio, lo), hi);
            const bool inside = (ratio >= lo) && (ratio <= hi);
            const bool active = inside || (s1 < s2);
            const float dlogp = active ? (-adv * ratio * invB) : 0.0f;
            const float v = values[r], R = returns[src];
            const float dv = v - R;
            dvalues[r] = vf_coef * 2.0f * dv * invB;
#pragma unroll
            for (int j = 0; j < A; ++j)
                dlogits[r * A + j] = dlogp * ((a == j ? 1.0f : 0.0f) - p[j]) + ent_coef * invB * p[j] * (lp[j] + ent);
            acc[0] = -fminf(s1, s2);
            acc[1] = dv * dv;
            acc[2] = -ent;
            acc[3] = (ratio - 1.0f) - lr;
            acc[4] = (fabsf(ratio - 1.0f) > clip) ? 1.0f : 0.0f;
        }
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
    for (int q = 0; q < 5; ++q) { acc[q] = warp_sum(acc[q]); if (l == 0) sh[q][w] = acc[q]; }
    __syncthreads();
    if (w == 0) {
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            float x = l < 8 ? sh[q][l] : 0.0f;
            x = warp_sum(x);
            acc[q] = x * invB;
        }
        if (l == 0) {
            if constexpr (DET) {
                float *row = stats + 8 * (int64_t)blockIdx.x;
#pragma unroll
                for (int q = 0; q < 5; ++q) row[q] = acc[q];
                row[5] = acc[0] + ent_coef * acc[2] + vf_coef * acc[1];
                return;
            }
#pragma unroll
            for (int q = 0; q < 5; ++q) atomicAdd(stats + q, acc[q]);
            atomicAdd(stats + 5, acc[0] + ent_coef * acc[2] + vf_coef * acc[1]);
        }
    }
}

// ----------------------------------------------------------------- clip_grad_norm_ + Adam (fused)
// The squared norm is reduced in a FIXED order (per-block partials, then every block of the Adam kernel sums
// the partials identically), so data-parallel replicas that all-reduced the same gradient stay bit-identical.
static constexpr int kNormBlocks = TMLA_NORM_BLOCKS;     // mlp_common.cuh: comm.cu writes the same number of partials
__global__ void __launch_bounds__(256) gradnorm_kernel(const float *__restrict__ g, int64_t np, float scale, float *partial) {
    __shared__ float sh[8];
    float s = 0.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < np; i += (int64_t)gridDim.x * blockDim.x) {
        const float x = g[i] * scale;
        s += x * x;
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sh[w];
        partial[blockIdx.x] = t;
    }
}
__global__ void __launch_bounds__(256)
adam_kernel(float *__restrict__ p, const float *g, float *__restrict__ m, float *__restrict__ v, int64_t np,
            float scale, float max_norm, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt,
            const float *__restrict__ partial, float *norm_out, int zero_grads,
            __nv_bfloat16 *__restrict__ img0, __nv_bfloat16 *__restrict__ img1, int64_t w2_off0, int64_t w2_off1) {
    __shared__ float s_norm;
    if (threadIdx.x < 32) {                                // same summation order in every block and on every rank
        float t = 0.0f;
        for (int j = threadIdx.x; j < kNormBlocks; j += 32) t += partial[j];
        t = warp_sum(t);
        if (threadIdx.x == 0) s_norm = sqrtf(t);
    }
    __syncthreads();
    const float norm = s_norm;
    // torch.nn.utils.clip_grad_norm_: coef = max_norm / (norm + 1e-6), clamped to 1
    const float coef = max_norm > 0.0f ? fminf(max_norm / (norm + 1e-6f), 1.0f) : 1.0f;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && norm_out) *norm_out = norm;
    if (i >= np) return;
    const float gi = g[i] * scale * coef;
    if (zero_grads) const_cast<float *>(g)[i] = 0.0f;     // the next minibatch accumulates into a clean buffer (no memset launch)
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;      // torch.optim.Adam (no amsgrad, no weight decay)
    const float pn = p[i] - (lr / bc1) * (mi / denom);
    p[i] = pn;
    if (img0) {      // hidden-layer weight: refresh its bf16 entry of the tensor-core operand image (mlp_tc.cu:pack_w2_kernel layout)
        const int64_t e0 = i - w2_off0, e1 = i - w2_off1;
        const bool in0 = e0 >= 0 && e0 < 65536, in1 = e1 >= 0 && e1 < 65536;
        if (in0 || in1) {
            const int e = (int)(in0 ? e0 : e1), r = e >> 8, k = e & 255;
            (in0 ? img0 : img1)[(r >> 3) * 2048 + (k >> 3) * 64 + (r & 7) * 8 + (k & 7)] = __float2bfloat16_rn(pn);
        }
    }
}

__global__ void bootstrap_add_kernel(float *rew, const int32_t *count, const int32_t *idx, const float *vals, float g, int32_t cap) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = min(*count, cap);
    if (i < c) rew[idx[i]] = __fadd_rn(rew[idx[i]], __fmul_rn(g, vals[i]));
}

static unsigned adv_stats_batched_gx(int64_t mb_rows) { return (unsigned)std::min<int64_t>(ceil_div64(mb_rows, 256 * 8), 148 * 2); }

extern "C" {

int tmla_gae(const float *rewards, const float *values, const uint8_t *dones, const float *last_values, double gamma,
             double gae_lambda, int T, int64_t n, float *advantages, float *returns, void *stream) {
    TMLA_REQUIRE(rewards && values && dones && last_values && advantages && returns, "NULL buffer");
    TMLA_REQUIRE(T > 0 && n > 0, "T and n must be positive");
    const float g = (float)gamma, gl = (float)(gamma * gae_lambda);
    static int unroll = -1;                                // TMLA_GAE_UNROLL=8|16|32 (experiments); default 16
    if (unroll < 0) { const char *e = getenv("TMLA_GAE_UNROLL"); unroll = e ? atoi(e) : 16; }
    const unsigned grid = (unsigned)ceil_div64(n, 128);
    if (unroll >= 32) gae_kernel<32><<<grid, 128, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, g, gl, T, n, advantages, returns);
    else if (unroll >= 16) gae_kernel<16><<<grid, 128, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, g, gl, T, n, advantages, returns);
    else gae_kernel<8><<<grid, 128, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, g, gl, T, n, advantages, returns);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int tmla_permutation(uint64_t seed, uint64_t epoch, int64_t total, int T, int64_t n, int32_t *out, void *stream) {
    TMLA_REQUIRE(out && total > 0 && T > 0 && n > 0, "bad arguments");
    TMLA_REQUIRE(total == (int64_t)T * n && total < ((int64_t)1 << 31), "total must equal T*n and fit int32");
    int bits = 2;
    while (((int64_t)1 << bits) < total) ++bits;
    if (bits & 1) ++bits;
    uint4 c = make_uint4((uint32_t)epoch, (uint32_t)(epoch >> 32), 0u, TMLA_TAG_PERM);
    const uint4 key = philox4x32_10(c, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    permutation_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)stream>>>(key, total, bits / 2, T, n, out);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int tmla_adv_stats(const float *advantages, const int32_t *index, int64_t rows, double *adv_sums, void *stream) {
    TMLA_REQUIRE(advantages && adv_sums && rows > 0, "bad arguments");
    TMLA_CUDA(cudaMemsetAsync(adv_sums, 0, 3 * sizeof(double), (cudaStream_t)stream));
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div64(rows, 256 * 8), 148 * 8);
    adv_stats_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(advantages, index, rows, adv_sums);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int tmla_adv_stats_batched(const float *advantages, const int32_t *index, int64_t total, int64_t mb_rows, double *adv_sums,
                           void *stream) {
    TMLA_REQUIRE(advantages && adv_sums && total > 0 && mb_rows > 0, "bad arguments");
    const int64_t n_mb = ceil_div64(total, mb_rows);
    TMLA_REQUIRE(n_mb <= 65535, "too many minibatches");
    TMLA_CUDA(cudaMemsetAsync(adv_sums, 0, 3 * sizeof(double) * n_mb, (cudaStream_t)stream));
    const unsigned gx = adv_stats_batched_gx(mb_rows);
    adv_stats_batched_kernel<false><<<dim3(gx, (unsigned)n_mb), 256, 0, (cudaStream_t)stream>>>(advantages, index, total, mb_rows, adv_sums);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int64_t tmla_adv_stats_det_scratch_bytes(int64_t total, int64_t mb_rows) {
    if (total <= 0 || mb_rows <= 0) { tmla_set_error("total and mb_rows must be positive"); return TMLA_EINVAL; }
    return 16 * ceil_div64(total, mb_rows) * (int64_t)adv_stats_batched_gx(mb_rows);
}

int tmla_adv_stats_batched_det(const float *advantages, const int32_t *index, int64_t total, int64_t mb_rows, double *adv_sums,
                               void *partials, void *stream) {
    TMLA_REQUIRE(advantages && adv_sums && partials && total > 0 && mb_rows > 0, "bad arguments");
    const int64_t n_mb = ceil_div64(total, mb_rows);
    TMLA_REQUIRE(n_mb <= 65535, "too many minibatches");
    const unsigned gx = adv_stats_batched_gx(mb_rows);
    cudaStream_t st = (cudaStream_t)stream;
    adv_stats_batched_kernel<true><<<dim3(gx, (unsigned)n_mb), 256, 0, st>>>(advantages, index, total, mb_rows, (double *)partials);
    TMLA_LAUNCH_CHECK();
    adv_stats_det_reduce_kernel<<<(unsigned)n_mb, 32, 0, st>>>((const double *)partials, (int)gx, total, mb_rows, adv_sums);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

}  // extern "C"

int64_t loss_det_scratch_bytes(int64_t rows) { return 4 * 8 * ceil_div64(rows, 256); }

// det_part != NULL: the deterministic form (per-block statistics rows in det_part, then det_reduce)
template <int LOSS>
static int loss_launch(const char *fn, const float *logits, const float *values, const int32_t *actions, const float *advantages,
                       const float *old_logp, const float *returns, const int32_t *index, int64_t rows, int64_t global_rows,
                       int n_actions, const double *adv_sums, int normalize_advantage, float clip_range, float ent_coef,
                       float vf_coef, float *dlogits, float *dvalues, float *stats_out, void *stream, float *det_part = nullptr) {
    TMLA_REQUIRE(logits && values && actions && advantages && (old_logp || LOSS == kLossA2C) && returns && dlogits && dvalues && stats_out,
                 "NULL buffer");
    TMLA_REQUIRE(rows > 0 && global_rows >= rows, "bad row counts");
    TMLA_REQUIRE(!normalize_advantage || adv_sums, "adv_sums required when normalising");
    cudaStream_t st = (cudaStream_t)stream;
    TMLA_CUDA(cudaMemsetAsync(stats_out, 0, 8 * sizeof(float), st));
    const unsigned grid = (unsigned)ceil_div64(rows, 256);
    const double inv = 1.0 / (double)global_rows;
#define LOSS_LAUNCH(AA, DET, OUT)                                                                                              \
    ppo_loss_kernel<AA, LOSS, DET><<<grid, 256, 0, st>>>(logits, values, actions, advantages, old_logp, returns, index, rows, inv, \
                                                         adv_sums, normalize_advantage, clip_range, ent_coef, vf_coef, dlogits, dvalues, OUT)
    if (n_actions < 3 || n_actions > 5) { tmla_set_error("%s: n_actions must be 3, 4 or 5 (got %d)", fn, n_actions); return TMLA_EINVAL; }
    if (det_part) {
        if (n_actions == 3) LOSS_LAUNCH(3, true, det_part);
        else if (n_actions == 4) LOSS_LAUNCH(4, true, det_part);
        else LOSS_LAUNCH(5, true, det_part);
    } else {
        if (n_actions == 3) LOSS_LAUNCH(3, false, stats_out);
        else if (n_actions == 4) LOSS_LAUNCH(4, false, stats_out);
        else LOSS_LAUNCH(5, false, stats_out);
    }
#undef LOSS_LAUNCH
    TMLA_LAUNCH_CHECK();
    if (!det_part) return TMLA_OK;
    DetSeg sg[2] = {DetSeg{det_part, 8, (int)grid, 6, stats_out, nullptr, 0, 0, 0},
                    DetSeg{det_part + 6, 8, 1, 2, stats_out + 6, nullptr, 0, 0, 1}};     // block 0's mean / std
    return det_reduce_launch(sg, normalize_advantage ? 2 : 1, st);
}

extern "C" {

int tmla_ppo_loss(const float *logits, const float *values, const int32_t *actions, const float *advantages,
                  const float *old_logp, const float *returns, const int32_t *index, int64_t rows, int64_t global_rows,
                  int n_actions, const double *adv_sums, int normalize_advantage, float clip_range, float ent_coef,
                  float vf_coef, float *dlogits, float *dvalues, float *stats_out, void *stream) {
    return loss_launch<kLossPPO>("tmla_ppo_loss", logits, values, actions, advantages, old_logp, returns, index, rows, global_rows, n_actions,
                                 adv_sums, normalize_advantage, clip_range, ent_coef, vf_coef, dlogits, dvalues, stats_out, stream);
}

int tmla_a2c_loss(const float *logits, const float *values, const int32_t *actions, const float *advantages, const float *returns,
                  const int32_t *index, int64_t rows, int64_t global_rows, int n_actions, const double *adv_sums,
                  int normalize_advantage, float ent_coef, float vf_coef, float *dlogits, float *dvalues, float *stats_out,
                  void *stream) {
    return loss_launch<kLossA2C>("tmla_a2c_loss", logits, values, actions, advantages, nullptr, returns, index, rows, global_rows, n_actions,
                                 adv_sums, normalize_advantage, 0.0f, ent_coef, vf_coef, dlogits, dvalues, stats_out, stream);
}

int tmla_ppo_loss_det(const float *logits, const float *values, const int32_t *actions, const float *advantages,
                      const float *old_logp, const float *returns, const int32_t *index, int64_t rows, int64_t global_rows,
                      int n_actions, const double *adv_sums, int normalize_advantage, float clip_range, float ent_coef,
                      float vf_coef, float *dlogits, float *dvalues, float *stats_out, void *partials, void *stream) {
    TMLA_REQUIRE(partials, "NULL partials");
    return loss_launch<kLossPPO>("tmla_ppo_loss_det", logits, values, actions, advantages, old_logp, returns, index, rows, global_rows,
                                 n_actions, adv_sums, normalize_advantage, clip_range, ent_coef, vf_coef, dlogits, dvalues, stats_out, stream,
                                 (float *)partials);
}

int tmla_a2c_loss_det(const float *logits, const float *values, const int32_t *actions, const float *advantages, const float *returns,
                      const int32_t *index, int64_t rows, int64_t global_rows, int n_actions, const double *adv_sums,
                      int normalize_advantage, float ent_coef, float vf_coef, float *dlogits, float *dvalues, float *stats_out,
                      void *partials, void *stream) {
    TMLA_REQUIRE(partials, "NULL partials");
    return loss_launch<kLossA2C>("tmla_a2c_loss_det", logits, values, actions, advantages, nullptr, returns, index, rows, global_rows,
                                 n_actions, adv_sums, normalize_advantage, 0.0f, ent_coef, vf_coef, dlogits, dvalues, stats_out, stream,
                                 (float *)partials);
}

}  // extern "C"

// clip + Adam with the squared-norm partials either computed here (partials_ready = false) or already in norm_out[1..] (the
// fused all-reduce of comm.cu); shared by tmla_adam_clip_fused and tmla_adam_clip_allreduce
int adam_clip_launch(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                     float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, int zero_grads,
                     void *wpack, int obs_dim, int hidden, int n_actions, void *stream, bool partials_ready) {
    TMLA_REQUIRE(params && grads && m && v && norm_out, "NULL buffer (norm_out doubles as scratch)");
    TMLA_REQUIRE(num_params > 0 && step >= 1, "bad arguments");
    if (!partials_ready) {      // norm pass + clip + Adam in ONE cooperative launch when the shape fits (comm.cu:opt_step_kernel<1>)
        const int rc = opt_step_launch(nullptr, params, grads, m, v, num_params, grad_scale, max_grad_norm, lr, beta1, beta2, eps, step,
                                       norm_out, zero_grads, wpack, obs_dim, hidden, n_actions, stream);
        if (rc != TMLA_EINVAL) return rc;
    }
    __nv_bfloat16 *img0 = nullptr, *img1 = nullptr;
    int64_t off0 = 0, off1 = 0;
    if (wpack) {
        TMLA_REQUIRE(hidden == 256, "operand images exist for hidden = 256 only");
        const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
        TMLA_REQUIRE(o.total == num_params, "num_params does not match (obs_dim, n_actions)");
        img0 = reinterpret_cast<__nv_bfloat16 *>(wpack) + (int64_t)4 * 65536; img1 = img0 + 65536;
        off0 = o.w2[0]; off1 = o.w2[1];
    }
    cudaStream_t st = (cudaStream_t)stream;
    // norm_out[0] = norm, norm_out[1 .. 1+kNormBlocks) = per-block partial sums of squares
    if (!partials_ready) {                                 // (comm.cu's reduce_norm_kernel has written them already)
        gradnorm_kernel<<<kNormBlocks, 256, 0, st>>>(grads, num_params, grad_scale, norm_out + 1);
        TMLA_LAUNCH_CHECK();
    }
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    adam_kernel<<<(unsigned)ceil_div64(num_params, 256), 256, 0, st>>>(params, grads, m, v, num_params, grad_scale, max_grad_norm, lr,
                                                                      beta1, beta2, eps, (float)bc1, (float)sqrt(bc2), norm_out + 1, norm_out, zero_grads,
                                                                      img0, img1, off0, off1);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

extern "C" {

int tmla_adam_clip_fused(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                         float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, int zero_grads,
                         void *wpack, int obs_dim, int hidden, int n_actions, void *stream) {
    return adam_clip_launch(params, grads, m, v, num_params, grad_scale, max_grad_norm, lr, beta1, beta2, eps, step, norm_out, zero_grads,
                            wpack, obs_dim, hidden, n_actions, stream, false);
}
int tmla_adam_clip_zero(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                        float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, int zero_grads, void *stream) {
    return tmla_adam_clip_fused(params, grads, m, v, num_params, grad_scale, max_grad_norm, lr, beta1, beta2, eps, step, norm_out,
                                zero_grads, nullptr, 0, 0, 0, stream);
}
int tmla_adam_clip(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                   float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, void *stream) {
    return tmla_adam_clip_zero(params, grads, m, v, num_params, grad_scale, max_grad_norm, lr, beta1, beta2, eps, step, norm_out, 0, stream);
}

int tmla_bootstrap_add(float *rew_buf, const int32_t *trunc_count, const int32_t *trunc_index, const float *trunc_values,
                       double gamma, int32_t capacity, void *stream) {
    TMLA_REQUIRE(rew_buf && trunc_count && trunc_index && trunc_values && capacity > 0, "bad arguments");
    bootstrap_add_kernel<<<(unsigned)ceil_div64(capacity, 256), 256, 0, (cudaStream_t)stream>>>(rew_buf, trunc_count, trunc_index,
                                                                                               trunc_values, (float)gamma, capacity);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

}  // extern "C"
