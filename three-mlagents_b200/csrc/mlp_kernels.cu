// mlp_kernels.cu — MlpPolicy (SB3 ActorCriticPolicy, net_arch dict(pi=[256,256], vf=[256,256]), tanh)
// forward and backward in float32 on CUDA cores.
//
// Replaces ActorCriticPolicy.forward / evaluate_actions / predict_values and autograd's backward for
// them (SB3 2.9.0, built in the reference at backend/mlagents/training.py:150 with policy_kwargs from
// training.py:363-365).  This float32 path is the numerics reference on the device (it matches the
// reference's fp32 CPU arithmetic to ~1e-6); the bf16 tcgen05/TMEM path in mlp_tc.cu is the fast one.
//
// Layout: flat fp32 parameter vector in policy.parameters() order (include/tmla.h), PyTorch Linear
// weights [out,in].  Activations are [rows,256] row-major.
#include <algorithm>
#include <stdlib.h>
#include <string.h>
#include <cuda_bf16.h>
#include "common.cuh"

static constexpr int H = 256;   // hidden width (net_arch of training.py:363-365)

// activations are float (numerics-reference path) or bf16 (tensor-core path, mlp_tc.cu)
__device__ __forceinline__ float act_load(const float *p, int64_t i) { return p[i]; }
__device__ __forceinline__ float act_load(const __nv_bfloat16 *p, int64_t i) { return __bfloat162float(p[i]); }
__device__ __forceinline__ void act_store(float *p, int64_t i, float v) { p[i] = v; }
__device__ __forceinline__ void act_store(__nv_bfloat16 *p, int64_t i, float v) { p[i] = __float2bfloat16_rn(v); }

// launchers of the tcgen05 kernels (mlp_tc.cu)
int tc_linear_launch(int epi, const void *A, const void *W, const float *bias, const void *aux, void *out, int64_t M,
                     const int32_t *rows_dev, cudaStream_t st);
int tc_wgrad_launch(const void *X, const void *Y, float *G, int64_t rows, cudaStream_t st);
int64_t tc_wgrad_det_planes(int64_t rows);
int tc_wgrad_det_launch(const void *X, const void *Y, float *planes, int64_t rows, cudaStream_t st);
// deterministic-mode partials of the fused batch (mlp_train.cu) and of the loss statistics (ppo_kernels.cu), in bytes
int64_t fused_det_scratch_bytes(int obs_dim, int hidden, int n_actions, int64_t rows);
int64_t loss_det_scratch_bytes(int64_t rows);
int tc_pack_w2_launch(const float *w2, void *w, void *wt, void *img, cudaStream_t st);
int tc_tower_forward_dual_launch(int D, int n_actions, const float *const *W1, const float *const *B1, const void *const *W2,
                                 const float *const *B2, const float *const *Wh, const float *const *Bh, const float *x,
                                 const int32_t *index, int64_t M, const int32_t *rows_dev, float *const *out, void *const *h1,
                                 void *const *h2, cudaStream_t st);
int tc_tower_forward_pipe_dual_launch(int D, int n_actions, const float *const *W1, const float *const *B1, const void *const *W2,
                                      const float *const *B2, const float *const *Wh, const float *const *Bh, const float *x,
                                      const int32_t *index, int64_t M, const int32_t *rows_dev, float *const *out, cudaStream_t st);
int tc_tower_forward_launch(int D, int nout, const float *W1, const float *B1, const void *W2, const float *B2, const float *Wh,
                            const float *Bh, const float *x, const int32_t *index, int64_t M, const int32_t *rows_dev, float *out,
                            void *h1, void *h2, cudaStream_t st);
// hidden widths 64 and 128 (mlp_small.cu)
int small_mlp_forward(const float *params, int D, int hidden, int A, const float *x, const int32_t *index, int64_t rows,
                      const int32_t *rows_dev, float *logits, float *values, float *act_cache, cudaStream_t st);
int64_t small_mlp_backward_scratch(int D, int hidden, int A, int64_t rows);
int small_mlp_backward(const float *params, int D, int hidden, int A, const float *x, const int32_t *index, int64_t rows,
                       const float *act_cache, const float *dlogits, const float *dvalues, float *grads, float *scratch,
                       cudaStream_t st);

#include "mlp_common.cuh"

// rows per block of the backward's reduction kernels: ~4 blocks per SM, at least 64 rows
static int backward_rows_per_block(int64_t rows) { return (int)std::max<int64_t>(64, ceil_div64(ceil_div64(rows, 148 * 4), 64) * 64); }

__device__ __forceinline__ int64_t eff_rows(int64_t rows, const int32_t *rows_dev) {
    return rows_dev ? min(rows, (int64_t)*rows_dev) : rows;
}

// ----------------------------------------------------------------------------- layer 1 (K = D tiny)
// thread j owns hidden unit j: W1[j][:] in registers, x rows broadcast from shared memory.
template <int D, typename AT>
__global__ void __launch_bounds__(H)
l1_forward_kernel(const float *__restrict__ W1, const float *__restrict__ b1, const float *__restrict__ x,
                  const int32_t *__restrict__ index, int64_t rows, const int32_t *rows_dev, AT *__restrict__ h1) {
    constexpr int R = 32;
    __shared__ float sx[R][D];
    rows = eff_rows(rows, rows_dev);
    const int64_t r0 = (int64_t)blockIdx.x * R;
    if (r0 >= rows) return;
    const int nr = (int)min((int64_t)R, rows - r0);
    for (int e = threadIdx.x; e < nr * D; e += H) {
        const int r = e / D, k = e % D;
        const int64_t src = index ? index[r0 + r] : (r0 + r);
        sx[r][k] = x[src * D + k];
    }
    float w[D];
    const int j = threadIdx.x;
#pragma unroll
    for (int k = 0; k < D; ++k) w[k] = W1[j * D + k];
    const float b = b1[j];
    __syncthreads();
    for (int r = 0; r < nr; ++r) {
        float acc = b;
#pragma unroll
        for (int k = 0; k < D; ++k) acc = fmaf(sx[r][k], w[k], acc);
        act_store(h1, (r0 + r) * H + j, tanhf(acc));
    }
}

// dW1[j][k] = sum_r dZ1[r][j] x[r][k], db1[j] = sum_r dZ1[r][j]
// DET (deterministic mode, every kernel below): no atomics — block b stores its sums in row b of the partials (rows of
// H*D + H floats here: dW1 | db1; dW1 / db1 point into row 0), det_reduce_kernel adds the rows in order
template <int D, typename AT, bool DET = false>
__global__ void __launch_bounds__(H)
l1_backward_kernel(const AT *__restrict__ dz1, const float *__restrict__ x, const int32_t *__restrict__ index,
                   int64_t rows, int rows_per_block, float *__restrict__ dW1, float *__restrict__ db1) {
    constexpr int R = 32;
    __shared__ float sx[R][D];
    const int j = threadIdx.x;
    float acc[D], accb = 0.0f;
#pragma unroll
    for (int k = 0; k < D; ++k) acc[k] = 0.0f;
    const int64_t rb = (int64_t)blockIdx.x * rows_per_block, re = min(rows, rb + rows_per_block);
    for (int64_t r0 = rb; r0 < re; r0 += R) {
        const int nr = (int)min((int64_t)R, re - r0);
        __syncthreads();
        for (int e = threadIdx.x; e < nr * D; e += H) {
            const int r = e / D, k = e % D;
            const int64_t src = index ? index[r0 + r] : (r0 + r);
            sx[r][k] = x[src * D + k];
        }
        __syncthreads();
        for (int r = 0; r < nr; ++r) {
            const float g = act_load(dz1, (r0 + r) * H + j);
            accb += g;
#pragma unroll
            for (int k = 0; k < D; ++k) acc[k] = fmaf(g, sx[r][k], acc[k]);
        }
    }
    if constexpr (DET) {
        const int64_t row = (int64_t)blockIdx.x * (H * D + H);
#pragma unroll
        for (int k = 0; k < D; ++k) dW1[row + j * D + k] = acc[k];
        db1[row + j] = accb;
        return;
    }
#pragma unroll
    for (int k = 0; k < D; ++k) atomicAdd(dW1 + j * D + k, acc[k]);
    atomicAdd(db1 + j, accb);
}

// ------------------------------------------------------------------------------------ output heads
// one warp per row: lane holds 8 of the 256 hidden activations (two float4) and the matching weights.
template <int NOUT, typename AT>
__global__ void __launch_bounds__(256)
head_forward_kernel(const float *__restrict__ Wh, const float *__restrict__ bh, const AT *__restrict__ h2,
                    int64_t rows, const int32_t *rows_dev, float *__restrict__ out) {
    rows = eff_rows(rows, rows_dev);
    constexpr bool BF = sizeof(AT) == 2;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    // lane's 8 hidden units: bf16 -> one 16-byte load (elements 8*lane..); f32 -> two float4 (4*lane.., 128+4*lane..)
    float w[NOUT][8];      // scalar loads: the value head's weights are not 16-byte aligned in the flat vector
#pragma unroll
    for (int a = 0; a < NOUT; ++a)
#pragma unroll
        for (int q = 0; q < 8; ++q)
            w[a][q] = Wh[a * H + (BF ? lane * 8 + q : (q < 4 ? lane * 4 + q : 128 + lane * 4 + (q - 4)))];
    constexpr int RB = 4;                                  // rows in flight per warp
    for (int64_t r0 = warp * RB; r0 < rows; r0 += nwarps * RB) {
        float x[RB][8];
#pragma unroll
        for (int u = 0; u < RB; ++u) {
            const int64_t r = min(r0 + u, rows - 1);
            if constexpr (BF) {
                const uint4 v = __ldg(reinterpret_cast<const uint4 *>(h2 + r * H) + lane);
                const uint32_t w32[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) { x[u][2 * q] = __uint_as_float(w32[q] << 16); x[u][2 * q + 1] = __uint_as_float(w32[q] & 0xFFFF0000u); }
            } else {
                const float4 x0 = reinterpret_cast<const float4 *>(h2 + r * H)[lane];
                const float4 x1 = reinterpret_cast<const float4 *>(h2 + r * H)[32 + lane];
                x[u][0] = x0.x; x[u][1] = x0.y; x[u][2] = x0.z; x[u][3] = x0.w; x[u][4] = x1.x; x[u][5] = x1.y; x[u][6] = x1.z; x[u][7] = x1.w;
            }
        }
        float s[RB][NOUT];
#pragma unroll
        for (int u = 0; u < RB; ++u)
#pragma unroll
            for (int a = 0; a < NOUT; ++a) {
                float t = 0.0f;
#pragma unroll
                for (int q = 0; q < 8; ++q) t = fmaf(x[u][q], w[a][q], t);
                s[u][a] = t;
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)                   // RB*NOUT independent butterflies interleaved
#pragma unroll
            for (int u = 0; u < RB; ++u)
#pragma unroll
                for (int a = 0; a < NOUT; ++a) s[u][a] += __shfl_xor_sync(0xffffffffu, s[u][a], o);
        if (lane == 0) {
#pragma unroll
            for (int u = 0; u < RB; ++u)
                if (r0 + u < rows)
#pragma unroll
                    for (int a = 0; a < NOUT; ++a) out[(r0 + u) * NOUT + a] = s[u][a] + bh[a];
        }
    }
}

// thread j owns hidden column j over a chunk of rows:
//   dZ2[r][j] = (sum_a dOut[r][a] Wh[a][j]) * (1 - h2[r][j]^2)
//   dWh[a][j] += dOut[r][a] h2[r][j] ; db2[j] += dZ2[r][j] ; dbh[a] += dOut[r][a]
template <int NOUT, typename AT>
__global__ void __launch_bounds__(H)
head_backward_kernel(const float *__restrict__ Wh, const AT *__restrict__ h2, const float *__restrict__ dout,
                     int64_t rows, int rows_per_block, AT *__restrict__ dz2, float *__restrict__ dWh,
                     float *__restrict__ dbh, float *__restrict__ db2) {
    constexpr int R = 64;
    __shared__ float sd[R][NOUT];
    const int j = threadIdx.x;
    float w[NOUT], accw[NOUT], accb2 = 0.0f, accbh = 0.0f;
#pragma unroll
    for (int a = 0; a < NOUT; ++a) { w[a] = Wh[a * H + j]; accw[a] = 0.0f; }
    const int64_t rb = (int64_t)blockIdx.x * rows_per_block, re = min(rows, rb + rows_per_block);
    for (int64_t r0 = rb; r0 < re; r0 += R) {
        const int nr = (int)min((int64_t)R, re - r0);
        __syncthreads();
        for (int e = threadIdx.x; e < nr * NOUT; e += H) sd[e / NOUT][e % NOUT] = dout[r0 * NOUT + e];
        __syncthreads();
        for (int r = 0; r < nr; ++r) {
            const float h = act_load(h2, (r0 + r) * H + j);
            float g = 0.0f;
#pragma unroll
            for (int a = 0; a < NOUT; ++a) { g = fmaf(sd[r][a], w[a], g); accw[a] = fmaf(sd[r][a], h, accw[a]); }
            g *= (1.0f - h * h);
            act_store(dz2, (r0 + r) * H + j, g);
            accb2 += g;
        }
        if (j < NOUT) for (int r = 0; r < nr; ++r) accbh += sd[r][j];
    }
#pragma unroll
    for (int a = 0; a < NOUT; ++a) atomicAdd(dWh + a * H + j, accw[a]);
    atomicAdd(db2 + j, accb2);
    if (j < NOUT) atomicAdd(dbh + j, accbh);
}

// ------------------------------------------------------- bf16-path CUDA-core kernels (lane = 8 columns)
// Row-streaming versions of the first layer and the head backward for the tensor-core path: a warp owns a
// row, a lane owns 8 consecutive hidden units, so activations move as 16-byte loads/stores (512 contiguous
// bytes per warp) and the per-row inputs (obs row, dOut row) are warp-uniform broadcast loads.
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void unpack8(const uint4 &v, float *f) {
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) { f[2 * q] = __uint_as_float(u[q] << 16); f[2 * q + 1] = __uint_as_float(u[q] & 0xFFFF0000u); }
}
__device__ __forceinline__ uint4 pack8(const float *f) {
    uint32_t u[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        __nv_bfloat162 t = __floats2bfloat162_rn(f[2 * q], f[2 * q + 1]);
        u[q] = *reinterpret_cast<uint32_t *>(&t);
    }
    return make_uint4(u[0], u[1], u[2], u[3]);
}
// block-wide sum of one float per (warp, column): 8 warps x 256 columns -> 256 sums, then `emit(col, sum)`
template <class F>
__device__ __forceinline__ void reduce_planes(float (*sh)[H], const float *vals8, F emit) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 8; ++c) sh[warp][lane * 8 + c] = vals8[c];
    __syncthreads();
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sh[w][threadIdx.x];
    emit(threadIdx.x, s);
}

// ---- per-warp cp.async row pipeline: DEPTH rows of 512 B (+ up to 8 aux floats) in flight per warp at zero
// register cost.  Every iteration commits exactly one group (possibly empty), so wait_group<DEPTH-1> always
// means "the oldest row has landed".
template <int DEPTH>
struct WarpRowPipe {
    static constexpr int SLOT = 512 + 32;
    uint8_t *base;
    int lane;
    __device__ __forceinline__ WarpRowPipe(uint8_t *smem_block) : base(smem_block + (threadIdx.x >> 5) * DEPTH * SLOT), lane(threadIdx.x & 31) {}
    __device__ __forceinline__ void issue(int slot, const void *row512, const float *aux, int naux) {
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(base + slot * SLOT);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + lane * 16), "l"((const uint8_t *)row512 + lane * 16) : "memory");
        if (lane < naux) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 512 + lane * 4), "l"(aux + lane) : "memory");
    }
    __device__ __forceinline__ void commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
    __device__ __forceinline__ void wait_oldest() {
        asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH - 1) : "memory");
        __syncwarp();
    }
    __device__ __forceinline__ uint4 row(int slot) const { return *reinterpret_cast<const uint4 *>(base + slot * SLOT + lane * 16); }
    __device__ __forceinline__ float aux(int slot, int j) const { return *reinterpret_cast<const float *>(base + slot * SLOT + 512 + j * 4); }
};
static constexpr int kPipeDepth = 12;
static constexpr int kPipeSmem = 8 * kPipeDepth * (512 + 32);      // 52224 B per 256-thread block

// h1 = tanh(x W1^T + b1): W1 staged once per block through shared memory (coalesced), persistent grid,
// the obs gather is lane-parallel over windows of 32 rows (lane l fetches index and the D floats of row l,
// values are broadcast with shuffles) and the next window is prefetched while the current one is computed.
template <int D>
__global__ void __launch_bounds__(256)
l1_forward_bf16_kernel(const float *__restrict__ W1, const float *__restrict__ b1, const float *__restrict__ x,
                       const int32_t *__restrict__ index, int64_t rows, const int32_t *rows_dev, __nv_bfloat16 *__restrict__ h1) {
    __shared__ float sw[H * D + H];
    rows = eff_rows(rows, rows_dev);
    for (int e = threadIdx.x; e < H * D + H; e += 256) sw[e] = e < H * D ? W1[e] : b1[e - H * D];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    float w[8][D], b[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        b[c] = sw[H * D + lane * 8 + c];
#pragma unroll
        for (int k = 0; k < D; ++k) w[c][k] = sw[(lane * 8 + c) * D + k];
    }
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nwin = (rows + 31) / 32;
    auto fetch = [&](int64_t win, float *xv) {
        const int64_t r = win * 32 + lane;
        if (win < nwin && r < rows) {
            const int64_t src = index ? (int64_t)__ldg(index + r) : r;
#pragma unroll
            for (int k = 0; k < D; ++k) xv[k] = __ldg(x + src * D + k);
        } else {
#pragma unroll
            for (int k = 0; k < D; ++k) xv[k] = 0.0f;
        }
    };
    float cur[D], nxt[D];
    fetch(warp, cur);
    for (int64_t win = warp; win < nwin; win += nwarps) {
        fetch(win + nwarps, nxt);                          // in flight while this window is computed
        const int64_t r0 = win * 32;
        const int nr = (int)min((int64_t)32, rows - r0);
#pragma unroll 4
        for (int j = 0; j < nr; ++j) {
            float xr[D];
#pragma unroll
            for (int k = 0; k < D; ++k) xr[k] = __shfl_sync(0xffffffffu, cur[k], j);
            float o[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float acc = b[c];
#pragma unroll
                for (int k = 0; k < D; ++k) acc = fmaf(xr[k], w[c][k], acc);
                o[c] = tanh_approx(acc);
            }
            reinterpret_cast<uint4 *>(h1 + (r0 + j) * H)[lane] = pack8(o);
        }
#pragma unroll
        for (int k = 0; k < D; ++k) cur[k] = nxt[k];
    }
}

// dW1[j][k] += sum_r dZ1[r][j] x[r][k],  db1[j] += sum_r dZ1[r][j]
// dZ1 rows stream through the cp.async pipe; the gathered obs row rides along as the slot's aux floats.
template <int D, bool DET = false>
__global__ void __launch_bounds__(256)
l1_backward_bf16_kernel(const __nv_bfloat16 *__restrict__ dz1, const float *__restrict__ x, const int32_t *__restrict__ index,
                        int64_t rows, int rows_per_block, float *__restrict__ dW1, float *__restrict__ db1) {
    extern __shared__ __align__(16) uint8_t dyn[];
    float (*sh)[H] = reinterpret_cast<float (*)[H]>(dyn);            // reduce_planes scratch (8 KB), after the loop
    WarpRowPipe<kPipeDepth> pipe(dyn);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc[D + 1][8];
#pragma unroll
    for (int k = 0; k <= D; ++k)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[k][c] = 0.0f;
    const int64_t rb = (int64_t)blockIdx.x * rows_per_block, re = min(rows, rb + rows_per_block);
    const int n = re > rb + warp ? (int)((re - rb - warp + 7) / 8) : 0;      // rows of this warp: rb + warp + 8*i
    // indices of the warp's rows, 32 at a time, lane-parallel (window w covers i in [32w, 32w+32))
    auto load_idx = [&](int win) -> int64_t {
        const int i = win * 32 + lane;
        if (i >= n) return 0;
        const int64_t r = rb + warp + 8 * (int64_t)i;
        return index ? (int64_t)__ldg(index + r) : r;
    };
    int64_t idx_cur = load_idx(0), idx_nxt = load_idx(1);
    auto issue_row = [&](int i) {                          // i-th row of this warp into slot i % DEPTH
        if (i < n) {
            const int64_t r = rb + warp + 8 * (int64_t)i;
            const int64_t src = __shfl_sync(0xffffffffu, ((i >> 5) & 1) == 0 ? idx_cur : idx_nxt, i & 31);
            pipe.issue(i % kPipeDepth, dz1 + r * H, x + src * D, D);
        }
        pipe.commit();
    };
    // windows alternate between idx_cur (even) and idx_nxt (odd); refresh the one just finished
    for (int p = 0; p < kPipeDepth; ++p) issue_row(p);
    for (int i = 0; i < n; ++i) {
        pipe.wait_oldest();
        const int slot = i % kPipeDepth;
        float g[8], xr[D];
        unpack8(pipe.row(slot), g);
#pragma unroll
        for (int k = 0; k < D; ++k) xr[k] = pipe.aux(slot, k);
        __syncwarp();
        const int ni = i + kPipeDepth;
        if ((ni & 31) == 0) {                              // entering a new window at issue side: reload the stale register
            if (((ni >> 5) & 1) == 0) idx_cur = load_idx(ni >> 5); else idx_nxt = load_idx(ni >> 5);
        }
        issue_row(ni);
#pragma unroll
        for (int k = 0; k < D; ++k)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[k][c] = fmaf(g[c], xr[k], acc[k][c]);
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[D][c] += g[c];
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    if constexpr (DET) {                                   // rows of H*D + H floats: dW1 | db1
        const int64_t row = (int64_t)blockIdx.x * (H * D + H);
#pragma unroll
        for (int k = 0; k < D; ++k) reduce_planes(sh, acc[k], [&](int j, float s) { dW1[row + j * D + k] = s; });
        reduce_planes(sh, acc[D], [&](int j, float s) { db1[row + j] = s; });
        return;
    }
#pragma unroll
    for (int k = 0; k < D; ++k) reduce_planes(sh, acc[k], [&](int j, float s) { atomicAdd(dW1 + j * D + k, s); });
    reduce_planes(sh, acc[D], [&](int j, float s) { atomicAdd(db1 + j, s); });
}

//   dZ2[r][j] = (sum_a dOut[r][a] Wh[a][j]) * (1 - h2[r][j]^2) ; dWh[a][j] += dOut[r][a] h2[r][j] ; db2[j] += dZ2[r][j] ; dbh[a] += dOut[r][a]
// h2 rows (and the dOut row as aux) stream through the cp.async pipe.
template <int NOUT, bool DET = false>
__global__ void __launch_bounds__(256)
head_backward_bf16_kernel(const float *__restrict__ Wh, const __nv_bfloat16 *__restrict__ h2, const float *__restrict__ dout,
                          int64_t rows, int rows_per_block, __nv_bfloat16 *__restrict__ dz2, float *__restrict__ dWh,
                          float *__restrict__ dbh, float *__restrict__ db2) {
    extern __shared__ __align__(16) uint8_t dyn[];
    float (*sh)[H] = reinterpret_cast<float (*)[H]>(dyn);
    WarpRowPipe<kPipeDepth> pipe(dyn);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float w[NOUT][8], accw[NOUT][8], accb2[8], accbh[NOUT];
#pragma unroll
    for (int a = 0; a < NOUT; ++a) {
        accbh[a] = 0.0f;
#pragma unroll
        for (int c = 0; c < 8; ++c) { w[a][c] = Wh[a * H + lane * 8 + c]; accw[a][c] = 0.0f; }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) accb2[c] = 0.0f;
    const int64_t rb = (int64_t)blockIdx.x * rows_per_block, re = min(rows, rb + rows_per_block);
    const int n = re > rb + warp ? (int)((re - rb - warp + 7) / 8) : 0;
    auto issue_row = [&](int i) {
        if (i < n) {
            const int64_t r = rb + warp + 8 * (int64_t)i;
            pipe.issue(i % kPipeDepth, h2 + r * H, dout + r * NOUT, NOUT);
        }
        pipe.commit();
    };
    for (int p = 0; p < kPipeDepth; ++p) issue_row(p);
    for (int i = 0; i < n; ++i) {
        pipe.wait_oldest();
        const int slot = i % kPipeDepth;
        float h[8], d[NOUT], g[8];
        unpack8(pipe.row(slot), h);
#pragma unroll
        for (int a = 0; a < NOUT; ++a) d[a] = pipe.aux(slot, a);
        __syncwarp();
        issue_row(i + kPipeDepth);
#pragma unroll
        for (int a = 0; a < NOUT; ++a) accbh[a] += d[a];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            float t = 0.0f;
#pragma unroll
            for (int a = 0; a < NOUT; ++a) { t = fmaf(d[a], w[a][c], t); accw[a][c] = fmaf(d[a], h[c], accw[a][c]); }
            g[c] = t * (1.0f - h[c] * h[c]);
            accb2[c] += g[c];
        }
        reinterpret_cast<uint4 *>(dz2 + (rb + warp + 8 * (int64_t)i) * H)[lane] = pack8(g);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    if constexpr (DET) {                                   // rows of NOUT*H + NOUT + H floats: dWh | dbh | db2
        const int64_t row = (int64_t)blockIdx.x * (NOUT * H + NOUT + H);
#pragma unroll
        for (int a = 0; a < NOUT; ++a) reduce_planes(sh, accw[a], [&](int j, float s) { dWh[row + a * H + j] = s; });
        reduce_planes(sh, accb2, [&](int j, float s) { db2[row + j] = s; });
        __syncthreads();
        if (lane == 0)
#pragma unroll
            for (int a = 0; a < NOUT; ++a) sh[warp][a] = accbh[a];
        __syncthreads();
        if (threadIdx.x < NOUT) {
            float t = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; ++w) t += sh[w][threadIdx.x];
            dbh[row + threadIdx.x] = t;
        }
        return;
    }
#pragma unroll
    for (int a = 0; a < NOUT; ++a) reduce_planes(sh, accw[a], [&](int j, float s) { atomicAdd(dWh + a * H + j, s); });
    reduce_planes(sh, accb2, [&](int j, float s) { atomicAdd(db2 + j, s); });
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < NOUT; ++a) atomicAdd(dbh + a, accbh[a]);
    }
}

// out[r][a] = h2[r] . Wh[a] + bh[a] for the tensor-core path: h2 rows stream through the cp.async pipe,
// weights come from shared memory (staged once per block), NOUT butterflies are interleaved.
template <int NOUT>
__global__ void __launch_bounds__(256)
head_forward_bf16_kernel(const float *__restrict__ Wh, const float *__restrict__ bh, const __nv_bfloat16 *__restrict__ h2,
                         int64_t rows, const int32_t *rows_dev, float *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t dyn[];
    __shared__ float sw[NOUT * H];
    rows = eff_rows(rows, rows_dev);
    for (int e = threadIdx.x; e < NOUT * H; e += 256) sw[e] = Wh[e];
    __syncthreads();
    WarpRowPipe<kPipeDepth> pipe(dyn);
    const int lane = threadIdx.x & 31;
    float w[NOUT][8];
#pragma unroll
    for (int a = 0; a < NOUT; ++a)
#pragma unroll
        for (int q = 0; q < 8; ++q) w[a][q] = sw[a * H + lane * 8 + q];
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int n = rows > warp ? (int)((rows - warp + nwarps - 1) / nwarps) : 0;   // rows warp + nwarps*i
    auto issue_row = [&](int i) {
        if (i < n) pipe.issue(i % kPipeDepth, h2 + (warp + nwarps * (int64_t)i) * H, nullptr, 0);
        pipe.commit();
    };
    for (int p = 0; p < kPipeDepth; ++p) issue_row(p);
    for (int i = 0; i < n; ++i) {
        pipe.wait_oldest();
        float x[8];
        unpack8(pipe.row(i % kPipeDepth), x);
        __syncwarp();
        issue_row(i + kPipeDepth);
        float s[NOUT];
#pragma unroll
        for (int a = 0; a < NOUT; ++a) {
            float t = 0.0f;
#pragma unroll
            for (int q = 0; q < 8; ++q) t = fmaf(x[q], w[a][q], t);
            s[a] = t;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int a = 0; a < NOUT; ++a) s[a] += __shfl_xor_sync(0xffffffffu, s[a], o);
        if (lane < NOUT) {
            float v = s[0];
#pragma unroll
            for (int a = 1; a < NOUT; ++a) v = lane == a ? s[a] : v;
            out[(warp + nwarps * (int64_t)i) * NOUT + lane] = v + bh[lane];
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// --------------------------------------------------------------------------- 128x128x8 SIMT SGEMM
// C[M,N] = epi( sum_k A(m,k) B(k,n) ).  256 threads, 8x8 micro-tile per thread split as 2x2 blocks of
// 4x4 (conflict-free float4 shared-memory reads), register prefetch of the next k-chunk.
//   A_KMAJOR : A is stored [M][K] (k contiguous) else [K][M]
//   B_KMAJOR : B is stored [N][K] (k contiguous) else [K][N]
enum { EPI_BIAS_TANH = 0, EPI_DTANH = 1, EPI_ATOMIC = 2 };

template <bool KMAJOR>
__device__ __forceinline__ void load_tile(const float *__restrict__ P, int ld, int64_t mn0, int64_t MN, int64_t k0, int64_t Kend, float4 &v) {
    // fetch this thread's float4 of a 128(mn) x 8(k) tile
    const int tid = threadIdx.x;
    v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (KMAJOR) {           // [MN][K]: 2 threads per row, float4 along k
        const int64_t row = mn0 + (tid >> 1), k = k0 + (tid & 1) * 4;
        if (row < MN) {
            if (k + 3 < Kend) v = *reinterpret_cast<const float4 *>(P + row * ld + k);
            else {
                if (k + 0 < Kend) v.x = P[row * ld + k + 0];
                if (k + 1 < Kend) v.y = P[row * ld + k + 1];
                if (k + 2 < Kend) v.z = P[row * ld + k + 2];
            }
        }
    } else {                // [K][MN]: 32 threads per k row, float4 along mn
        const int64_t k = k0 + (tid >> 5), mn = mn0 + (tid & 31) * 4;
        if (k < Kend) {
            if (mn + 3 < MN) v = *reinterpret_cast<const float4 *>(P + k * ld + mn);
            else {
                if (mn + 0 < MN) v.x = P[k * ld + mn + 0];
                if (mn + 1 < MN) v.y = P[k * ld + mn + 1];
                if (mn + 2 < MN) v.z = P[k * ld + mn + 2];
            }
        }
    }
}
template <bool KMAJOR>
__device__ __forceinline__ void store_tile(float (*S)[128], const float4 &v) {
    const int tid = threadIdx.x;
    if (KMAJOR) {
        const int mn = tid >> 1, k = (tid & 1) * 4;
        S[k + 0][mn] = v.x; S[k + 1][mn] = v.y; S[k + 2][mn] = v.z; S[k + 3][mn] = v.w;
    } else {
        *reinterpret_cast<float4 *>(&S[tid >> 5][(tid & 31) * 4]) = v;
    }
}

template <bool A_KMAJOR, bool B_KMAJOR, int EPI>
__global__ void __launch_bounds__(256)
sgemm_kernel(const float *__restrict__ A, const float *__restrict__ B, float *__restrict__ C, int64_t M, int N, int64_t K,
             int lda, int ldb, int ldc, int64_t k_per_split, const float *__restrict__ aux, const int32_t *rows_dev) {
    __shared__ __align__(16) float As[8][128];
    __shared__ __align__(16) float Bs[8][128];
    if (rows_dev && EPI != EPI_ATOMIC) M = min(M, (int64_t)*rows_dev);
    const int64_t m0 = (int64_t)blockIdx.x * 128;
    const int n0 = blockIdx.y * 128;
    if (m0 >= M) return;
    const int64_t kb = (int64_t)blockIdx.z * k_per_split, ke = min(K, kb + k_per_split);
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

    float4 ra, rb;
    load_tile<A_KMAJOR>(A, lda, m0, M, kb, ke, ra);
    load_tile<B_KMAJOR>(B, ldb, n0, N, kb, ke, rb);
    for (int64_t k0 = kb; k0 < ke; k0 += 8) {
        __syncthreads();
        store_tile<A_KMAJOR>(As, ra);
        store_tile<B_KMAJOR>(Bs, rb);
        __syncthreads();
        if (k0 + 8 < ke) {
            load_tile<A_KMAJOR>(A, lda, m0, M, k0 + 8, ke, ra);
            load_tile<B_KMAJOR>(B, ldb, n0, N, k0 + 8, ke, rb);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
    }
    // epilogue
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (m >= M) continue;
#pragma unroll
        for (int jh = 0; jh < 2; ++jh) {
            const int n = n0 + (jh ? 64 : 0) + tx * 4;
            float4 v = make_float4(acc[i][jh * 4 + 0], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]);
            if (EPI == EPI_BIAS_TANH) {          // aux = bias[N]
                const float4 b = *reinterpret_cast<const float4 *>(aux + n);
                v.x = tanhf(v.x + b.x); v.y = tanhf(v.y + b.y); v.z = tanhf(v.z + b.z); v.w = tanhf(v.w + b.w);
                *reinterpret_cast<float4 *>(C + m * ldc + n) = v;
            } else if (EPI == EPI_DTANH) {       // aux = activation [M][N]: multiply by 1 - h^2
                const float4 h = *reinterpret_cast<const float4 *>(aux + m * ldc + n);
                v.x *= 1.0f - h.x * h.x; v.y *= 1.0f - h.y * h.y; v.z *= 1.0f - h.z * h.z; v.w *= 1.0f - h.w * h.w;
                *reinterpret_cast<float4 *>(C + m * ldc + n) = v;
            } else {                             // split-K accumulation
                atomicAdd(C + m * ldc + n + 0, v.x); atomicAdd(C + m * ldc + n + 1, v.y);
                atomicAdd(C + m * ldc + n + 2, v.z); atomicAdd(C + m * ldc + n + 3, v.w);
            }
        }
    }
}

// --------------------------------------------------------------------------------------- host API
static int ensure_pipe_attrs() {
    static int done = 0;
    if (done) return TMLA_OK;
#define PIPE_ATTR(K) TMLA_CUDA(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, kPipeSmem))
    PIPE_ATTR(head_forward_bf16_kernel<1>); PIPE_ATTR(head_forward_bf16_kernel<3>); PIPE_ATTR(head_forward_bf16_kernel<4>);
    PIPE_ATTR(head_forward_bf16_kernel<5>);
    PIPE_ATTR(head_backward_bf16_kernel<1>); PIPE_ATTR(head_backward_bf16_kernel<3>); PIPE_ATTR(head_backward_bf16_kernel<4>);
    PIPE_ATTR(head_backward_bf16_kernel<5>);
    PIPE_ATTR(l1_backward_bf16_kernel<4>); PIPE_ATTR(l1_backward_bf16_kernel<6>);
    PIPE_ATTR((head_backward_bf16_kernel<1, true>)); PIPE_ATTR((head_backward_bf16_kernel<3, true>));   // deterministic forms
    PIPE_ATTR((head_backward_bf16_kernel<4, true>)); PIPE_ATTR((head_backward_bf16_kernel<5, true>));
    PIPE_ATTR((l1_backward_bf16_kernel<4, true>)); PIPE_ATTR((l1_backward_bf16_kernel<6, true>));
#undef PIPE_ATTR
    done = 1;
    return TMLA_OK;
}

// shared body of the fp32 (AT=float, SIMT SGEMM) and bf16 (AT=__nv_bfloat16, tcgen05) paths
template <typename AT>
static int mlp_forward_impl(const float *params, const void *wpack, int obs_dim, int n_actions, const float *x, const int32_t *index,
                            int64_t rows, const int32_t *rows_dev, float *logits, float *values, AT *act_cache, cudaStream_t st,
                            bool keep_act = true) {
    constexpr bool BF = sizeof(AT) == 2;
    if (BF) { int rc = ensure_pipe_attrs(); if (rc) return rc; }
    const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
    if constexpr (BF) {
        if (obs_dim <= 6 && logits && values) {      // both towers, one launch (even / odd CTAs)
            const float *W1[2], *B1[2], *B2[2], *Wh[2], *Bh[2];
            const void *W2[2];
            float *out[2] = {logits, values};
            void *h1[2], *h2[2];
            for (int t = 0; t < 2; ++t) {
                W1[t] = params + o.w1[t]; B1[t] = params + o.b1[t]; B2[t] = params + o.b2[t]; Wh[t] = params + o.wh[t]; Bh[t] = params + o.bh[t];
                W2[t] = reinterpret_cast<const __nv_bfloat16 *>(wpack) + (int64_t)(4 + t) * H * H;      // operand images
                h1[t] = keep_act ? (void *)(act_cache + (int64_t)(2 * t) * rows * H) : nullptr;
                h2[t] = keep_act ? (void *)(act_cache + (int64_t)(2 * t + 1) * rows * H) : nullptr;
            }
            if (!keep_act) {      // inference (rollout step): the pipelined kernel — double-buffered TMEM accumulator, driver warp
                static const bool classic = [] { const char *e = getenv("TMLA_FWD"); return e && !strcmp(e, "classic"); }();
                if (!classic) {
                    const int rcp = tc_tower_forward_pipe_dual_launch(obs_dim, n_actions, W1, B1, W2, B2, Wh, Bh, x, index, rows, rows_dev, out, st);
                    if (rcp != TMLA_EINVAL) return rcp;
                }
            }
            const int rc = tc_tower_forward_dual_launch(obs_dim, n_actions, W1, B1, W2, B2, Wh, Bh, x, index, rows, rows_dev, out, h1, h2, st);
            if (rc != TMLA_EINVAL) return rc;
        }
    }
    for (int t = 0; t < 2; ++t) {
        float *out = t == 0 ? logits : values;
        if (!out) continue;
        AT *h1 = act_cache + (int64_t)(2 * t) * rows * H, *h2 = act_cache + (int64_t)(2 * t + 1) * rows * H;
        if constexpr (BF) {
            if (obs_dim <= 6) {      // fused tower: gather + layer 1 + tcgen05 layer 2 + head in one persistent kernel
                // W2 as its 128 KB operand IMAGE (wpack matrices 4, 5): one bulk-TMA load per CTA instead of a per-thread staging loop
                const __nv_bfloat16 *w2 = reinterpret_cast<const __nv_bfloat16 *>(wpack) + (int64_t)(4 + t) * H * H;
                int rc = tc_tower_forward_launch(obs_dim, o.nout[t], params + o.w1[t], params + o.b1[t], w2, params + o.b2[t],
                                                 params + o.wh[t], params + o.bh[t], x, index, rows, rows_dev, out,
                                                 keep_act ? (void *)h1 : nullptr, keep_act ? (void *)h2 : nullptr, st);
                if (rc) return rc;
                continue;
            }
        }
        const unsigned g1 = (unsigned)ceil_div64(rows, 32);
#define L1F(DD) l1_forward_kernel<DD, AT><<<g1, H, 0, st>>>(params + o.w1[t], params + o.b1[t], x, index, rows, rows_dev, h1)
        const unsigned gs = (unsigned)std::min<int64_t>(ceil_div64(rows, 256), 148 * 2);    // persistent: 32-row windows per warp
        if constexpr (BF) {
            if (obs_dim == 4) l1_forward_bf16_kernel<4><<<gs, 256, 0, st>>>(params + o.w1[t], params + o.b1[t], x, index, rows, rows_dev, h1);
            else if (obs_dim == 6) l1_forward_bf16_kernel<6><<<gs, 256, 0, st>>>(params + o.w1[t], params + o.b1[t], x, index, rows, rows_dev, h1);
            else if (obs_dim == 45) L1F(45); else if (obs_dim == 7) L1F(7); else if (obs_dim == 16) L1F(16); else L1F(21);
        } else {
            if (obs_dim == 4) L1F(4); else if (obs_dim == 6) L1F(6); else if (obs_dim == 45) L1F(45); else if (obs_dim == 7) L1F(7); else if (obs_dim == 16) L1F(16); else L1F(21);
        }
#undef L1F
        TMLA_LAUNCH_CHECK();
        if constexpr (BF) {
            const __nv_bfloat16 *w2 = reinterpret_cast<const __nv_bfloat16 *>(wpack) + (int64_t)(2 * t) * H * H;
            int rc = tc_linear_launch(0, h1, w2, params + o.b2[t], nullptr, h2, rows, rows_dev, st);
            if (rc) return rc;
        } else {
            dim3 grid((unsigned)ceil_div64(rows, 128), H / 128, 1);
            sgemm_kernel<true, true, EPI_BIAS_TANH><<<grid, 256, 0, st>>>((const float *)h1, params + o.w2[t], (float *)h2, rows, H, H, H, H,
                                                                          H, H, params + o.b2[t], rows_dev);
            TMLA_LAUNCH_CHECK();
        }
        if constexpr (BF) {
            const unsigned gh = (unsigned)std::min<int64_t>(ceil_div64(rows, 8 * kPipeDepth), 148 * 4);
            if (t == 1) head_forward_bf16_kernel<1><<<gh, 256, kPipeSmem, st>>>(params + o.wh[1], params + o.bh[1], h2, rows, rows_dev, out);
            else if (n_actions == 3) head_forward_bf16_kernel<3><<<gh, 256, kPipeSmem, st>>>(params + o.wh[0], params + o.bh[0], h2, rows, rows_dev, out);
            else if (n_actions == 4) head_forward_bf16_kernel<4><<<gh, 256, kPipeSmem, st>>>(params + o.wh[0], params + o.bh[0], h2, rows, rows_dev, out);
            else head_forward_bf16_kernel<5><<<gh, 256, kPipeSmem, st>>>(params + o.wh[0], params + o.bh[0], h2, rows, rows_dev, out);
        } else {
            const unsigned gh = (unsigned)std::min<int64_t>(ceil_div64(rows, 8), 148 * 8);
            if (t == 1) head_forward_kernel<1, AT><<<gh, 256, 0, st>>>(params + o.wh[1], params + o.bh[1], h2, rows, rows_dev, out);
            else if (n_actions == 3) head_forward_kernel<3, AT><<<gh, 256, 0, st>>>(params + o.wh[0], params + o.bh[0], h2, rows, rows_dev, out);
            else if (n_actions == 4) head_forward_kernel<4, AT><<<gh, 256, 0, st>>>(params + o.wh[0], params + o.bh[0], h2, rows, rows_dev, out);
            else head_forward_kernel<5, AT><<<gh, 256, 0, st>>>(params + o.wh[0], params + o.bh[0], h2, rows, rows_dev, out);
        }
        TMLA_LAUNCH_CHECK();
    }
    return TMLA_OK;
}

template <typename AT>
static int mlp_backward_impl(const float *params, const void *wpack, int obs_dim, int n_actions, const float *x, const int32_t *index,
                             int64_t rows, const AT *act_cache, const float *dlogits, const float *dvalues, float *grads,
                             AT *scratch, cudaStream_t st) {
    constexpr bool BF = sizeof(AT) == 2;
    if (BF) { int rc = ensure_pipe_attrs(); if (rc) return rc; }
    const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
    TMLA_CUDA(cudaMemsetAsync(grads, 0, sizeof(float) * o.total, st));
    AT *dz2 = scratch, *dz1 = scratch + rows * H;
    // chunk rows so that ~4 blocks per SM share the reduction kernels
    const int rpb = backward_rows_per_block(rows);
    const unsigned gr = (unsigned)ceil_div64(rows, rpb);
    for (int t = 0; t < 2; ++t) {
        const AT *h1 = act_cache + (int64_t)(2 * t) * rows * H, *h2 = act_cache + (int64_t)(2 * t + 1) * rows * H;
        const float *dout = t == 0 ? dlogits : dvalues;
        if constexpr (BF) {
            if (t == 1) head_backward_bf16_kernel<1><<<gr, 256, kPipeSmem, st>>>(params + o.wh[1], h2, dout, rows, rpb, dz2, grads + o.wh[1], grads + o.bh[1], grads + o.b2[1]);
            else if (n_actions == 3) head_backward_bf16_kernel<3><<<gr, 256, kPipeSmem, st>>>(params + o.wh[0], h2, dout, rows, rpb, dz2, grads + o.wh[0], grads + o.bh[0], grads + o.b2[0]);
            else if (n_actions == 4) head_backward_bf16_kernel<4><<<gr, 256, kPipeSmem, st>>>(params + o.wh[0], h2, dout, rows, rpb, dz2, grads + o.wh[0], grads + o.bh[0], grads + o.b2[0]);
            else head_backward_bf16_kernel<5><<<gr, 256, kPipeSmem, st>>>(params + o.wh[0], h2, dout, rows, rpb, dz2, grads + o.wh[0], grads + o.bh[0], grads + o.b2[0]);
        } else {
            if (t == 1) head_backward_kernel<1, AT><<<gr, H, 0, st>>>(params + o.wh[1], h2, dout, rows, rpb, dz2, grads + o.wh[1], grads + o.bh[1], grads + o.b2[1]);
            else if (n_actions == 3) head_backward_kernel<3, AT><<<gr, H, 0, st>>>(params + o.wh[0], h2, dout, rows, rpb, dz2, grads + o.wh[0], grads + o.bh[0], grads + o.b2[0]);
            else if (n_actions == 4) head_backward_kernel<4, AT><<<gr, H, 0, st>>>(params + o.wh[0], h2, dout, rows, rpb, dz2, grads + o.wh[0], grads + o.bh[0], grads + o.b2[0]);
            else head_backward_kernel<5, AT><<<gr, H, 0, st>>>(params + o.wh[0], h2, dout, rows, rpb, dz2, grads + o.wh[0], grads + o.bh[0], grads + o.b2[0]);
        }
        TMLA_LAUNCH_CHECK();
        if constexpr (BF) {
            // dZ1 = (dZ2 . W2) * (1 - h1^2) with W2^T as the K-major weight;  dW2 += dZ2^T . h1  (tcgen05)
            const __nv_bfloat16 *w2t = reinterpret_cast<const __nv_bfloat16 *>(wpack) + (int64_t)(2 * t + 1) * H * H;
            int rc = tc_linear_launch(1, dz2, w2t, nullptr, h1, dz1, rows, nullptr, st);
            if (rc) return rc;
            rc = tc_wgrad_launch(dz2, h1, grads + o.w2[t], rows, st);
            if (rc) return rc;
        } else {
            // dZ1 = (dZ2 . W2) * (1 - h1^2)      A = dZ2 [rows][H] (k-major), B = W2 [K=out][N=in]
            dim3 gd((unsigned)ceil_div64(rows, 128), H / 128, 1);
            sgemm_kernel<true, false, EPI_DTANH><<<gd, 256, 0, st>>>((const float *)dz2, params + o.w2[t], (float *)dz1, rows, H, H, H, H, H, H,
                                                                     (const float *)h1, nullptr);
            TMLA_LAUNCH_CHECK();
            // dW2[j][i] = sum_r dZ2[r][j] h1[r][i]   A = dZ2 as [K=rows][M=H], B = h1 as [K=rows][N=H]; split-K + atomics
            int64_t splits = std::min<int64_t>(std::max<int64_t>(1, ceil_div64(rows, 1024)), 148);
            const int64_t kps = ceil_div64(ceil_div64(rows, splits), 8) * 8;
            splits = ceil_div64(rows, kps);
            dim3 gw(H / 128, H / 128, (unsigned)splits);
            sgemm_kernel<false, false, EPI_ATOMIC><<<gw, 256, 0, st>>>((const float *)dz2, (const float *)h1, grads + o.w2[t], H, H, rows, H, H, H,
                                                                      kps, nullptr, nullptr);
            TMLA_LAUNCH_CHECK();
        }
#define L1B(DD) l1_backward_kernel<DD, AT><<<gr, H, 0, st>>>(dz1, x, index, rows, rpb, grads + o.w1[t], grads + o.b1[t])
        if constexpr (BF) {
            if (obs_dim == 4) l1_backward_bf16_kernel<4><<<gr, 256, kPipeSmem, st>>>(dz1, x, index, rows, rpb, grads + o.w1[t], grads + o.b1[t]);
            else if (obs_dim == 6) l1_backward_bf16_kernel<6><<<gr, 256, kPipeSmem, st>>>(dz1, x, index, rows, rpb, grads + o.w1[t], grads + o.b1[t]);
            else if (obs_dim == 45) L1B(45); else if (obs_dim == 7) L1B(7); else if (obs_dim == 16) L1B(16); else L1B(21);
        } else {
            if (obs_dim == 4) L1B(4); else if (obs_dim == 6) L1B(6); else if (obs_dim == 45) L1B(45); else if (obs_dim == 7) L1B(7); else if (obs_dim == 16) L1B(16); else L1B(21);
        }
#undef L1B
        TMLA_LAUNCH_CHECK();
    }
    return TMLA_OK;
}

// Deterministic form of the bf16 backward: the same kernels and block split, every atomic replaced by a partial row per block
// (a 256x256 plane per weight-gradient CTA), then one det_reduce launch.  Partials (floats), per tower t:
//   W2 planes [2][P] | head rows [2][gr][A_t*H + A_t + H] | layer-1 rows [2][gr][H*D + H]     (P = tc_wgrad_det_planes(rows))
struct BackwardDetLayout {
    int64_t planes, gr, head[2], l1, w2_off[2], head_off[2], l1_off[2], total;
};
static BackwardDetLayout backward_det_layout(int D, int A, int64_t planes, int64_t gr) {
    BackwardDetLayout L;
    L.planes = planes; L.gr = gr;
    L.head[0] = (int64_t)A * H + A + H; L.head[1] = H + 1 + H; L.l1 = (int64_t)H * D + H;
    int64_t p = 0;
    for (int t = 0; t < 2; ++t) { L.w2_off[t] = p; p += planes * H * H; }
    for (int t = 0; t < 2; ++t) { L.head_off[t] = p; p += gr * L.head[t]; }
    for (int t = 0; t < 2; ++t) { L.l1_off[t] = p; p += gr * L.l1; }
    L.total = p;
    return L;
}
static int64_t backward_det_bytes(int D, int A, int64_t rows) {     // monotone in rows: upper bounds of the block counts
    const int64_t gr_max = std::min<int64_t>(ceil_div64(rows, 64), 148 * 4);
    return 4 * backward_det_layout(D, A, tc_wgrad_det_planes(rows), gr_max).total;
}

static int mlp_backward_bf16_det(const float *params, const void *wpack, int obs_dim, int n_actions, const float *x, const int32_t *index,
                                 int64_t rows, const __nv_bfloat16 *act_cache, const float *dlogits, const float *dvalues, float *grads,
                                 __nv_bfloat16 *scratch, float *part, cudaStream_t st) {
    int rc = ensure_pipe_attrs();
    if (rc) return rc;
    const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
    TMLA_CUDA(cudaMemsetAsync(grads, 0, sizeof(float) * o.total, st));
    __nv_bfloat16 *dz2 = scratch, *dz1 = scratch + rows * H;
    const int rpb = backward_rows_per_block(rows);
    const unsigned gr = (unsigned)ceil_div64(rows, rpb);
    const BackwardDetLayout L = backward_det_layout(obs_dim, n_actions, tc_wgrad_det_planes(rows), gr);
    for (int t = 0; t < 2; ++t) {
        const __nv_bfloat16 *h1 = act_cache + (int64_t)(2 * t) * rows * H, *h2 = act_cache + (int64_t)(2 * t + 1) * rows * H;
        const float *dout = t == 0 ? dlogits : dvalues;
        const int nout = o.nout[t];
        float *hw = part + L.head_off[t], *hb = hw + nout * H, *hb2 = hb + nout;        // row 0: dWh | dbh | db2
        const float *wh = params + o.wh[t];
        if (t == 1) head_backward_bf16_kernel<1, true><<<gr, 256, kPipeSmem, st>>>(wh, h2, dout, rows, rpb, dz2, hw, hb, hb2);
        else if (n_actions == 3) head_backward_bf16_kernel<3, true><<<gr, 256, kPipeSmem, st>>>(wh, h2, dout, rows, rpb, dz2, hw, hb, hb2);
        else if (n_actions == 4) head_backward_bf16_kernel<4, true><<<gr, 256, kPipeSmem, st>>>(wh, h2, dout, rows, rpb, dz2, hw, hb, hb2);
        else head_backward_bf16_kernel<5, true><<<gr, 256, kPipeSmem, st>>>(wh, h2, dout, rows, rpb, dz2, hw, hb, hb2);
        TMLA_LAUNCH_CHECK();
        const __nv_bfloat16 *w2t = reinterpret_cast<const __nv_bfloat16 *>(wpack) + (int64_t)(2 * t + 1) * H * H;
        rc = tc_linear_launch(1, dz2, w2t, nullptr, h1, dz1, rows, nullptr, st);
        if (rc) return rc;
        rc = tc_wgrad_det_launch(dz2, h1, part + L.w2_off[t], rows, st);
        if (rc) return rc;
        float *lw = part + L.l1_off[t], *lb = lw + H * obs_dim;                       // row 0: dW1 | db1
#define L1B(DD) l1_backward_kernel<DD, __nv_bfloat16, true><<<gr, H, 0, st>>>(dz1, x, index, rows, rpb, lw, lb)
        if (obs_dim == 4) l1_backward_bf16_kernel<4, true><<<gr, 256, kPipeSmem, st>>>(dz1, x, index, rows, rpb, lw, lb);
        else if (obs_dim == 6) l1_backward_bf16_kernel<6, true><<<gr, 256, kPipeSmem, st>>>(dz1, x, index, rows, rpb, lw, lb);
        else if (obs_dim == 45) L1B(45); else if (obs_dim == 7) L1B(7); else if (obs_dim == 16) L1B(16); else L1B(21);
#undef L1B
        TMLA_LAUNCH_CHECK();
    }
    DetSeg sg[kDetMaxSegs];
    int n = 0;
    const int g = (int)gr;
    for (int t = 0; t < 2; ++t) {
        const int nout = o.nout[t];
        sg[n++] = DetSeg{part + L.w2_off[t], H * H, (int)L.planes, H * H, grads + o.w2[t], nullptr, 0, 0, 0};
        sg[n++] = DetSeg{part + L.head_off[t], L.head[t], g, nout * H + nout, grads + o.wh[t], nullptr, 0, 0, 0};     // Wh | bh
        sg[n++] = DetSeg{part + L.head_off[t] + nout * H + nout, L.head[t], g, H, grads + o.b2[t], nullptr, 0, 0, 0};
        sg[n++] = DetSeg{part + L.l1_off[t], L.l1, g, (int)L.l1, grads + o.w1[t], nullptr, 0, 0, 0};             // W1 | b1
    }
    return det_reduce_launch(sg, n, st);
}

extern "C" {

static bool small_width(int hidden) { return hidden == 64 || hidden == 128; }

int64_t tmla_mlp_num_params(int obs_dim, int hidden, int n_actions) {
    if (!(hidden == H || small_width(hidden))) { tmla_set_error("hidden must be 64, 128 or 256, got %d", hidden); return TMLA_EINVAL; }
    if (obs_dim <= 0 || n_actions <= 0) return TMLA_EINVAL;
    return mlp_offsets(obs_dim, n_actions, hidden).total;
}

// fp32: the float32 entry points (hidden 64, 128 or 256); otherwise the bf16 tensor-core ones (256 only)
static int check_shape(int D, int hidden, int A, bool fp32 = false) {
    if (fp32 && !(hidden == H || small_width(hidden))) {
        tmla_set_error("hidden must be 64, 128 or 256, got %d", hidden);
        return TMLA_EINVAL;
    }
    if (!fp32 && hidden != H) {
        tmla_set_error("the bf16 tensor-core path covers hidden = 256 only (got %d); widths 64 and 128 run on tmla_mlp_forward / "
                       "tmla_mlp_backward in float32", hidden);
        return TMLA_EINVAL;
    }
    if (!(D == 4 || D == 6 || D == 7 || D == 16 || D == 21 || D == 45)) { tmla_set_error("obs_dim must be 4, 6, 7, 16, 21 or 45, got %d", D); return TMLA_EINVAL; }
    if (!(A >= 3 && A <= 5)) { tmla_set_error("n_actions must be 3, 4 or 5, got %d", A); return TMLA_EINVAL; }
    return TMLA_OK;
}

int tmla_mlp_forward(const float *params, int obs_dim, int hidden, int n_actions, const float *x, const int32_t *index,
                     int64_t rows, const int32_t *rows_dev, float *logits, float *values, float *act_cache, void *stream) {
    TMLA_REQUIRE(params && x, "params/x must be non-NULL");
    TMLA_REQUIRE(act_cache || small_width(hidden), "act_cache (the activation workspace) may be NULL only for hidden 64 and 128");
    TMLA_REQUIRE(rows > 0, "rows must be positive");
    TMLA_REQUIRE(logits || values, "nothing to compute");
    int rc = check_shape(obs_dim, hidden, n_actions, true);
    if (rc) return rc;
    if (hidden != H)
        return small_mlp_forward(params, obs_dim, hidden, n_actions, x, index, rows, rows_dev, logits, values, act_cache, (cudaStream_t)stream);
    return mlp_forward_impl<float>(params, nullptr, obs_dim, n_actions, x, index, rows, rows_dev, logits, values, act_cache, (cudaStream_t)stream);
}

int tmla_mlp_forward_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *x,
                          const int32_t *index, int64_t rows, const int32_t *rows_dev, float *logits, float *values,
                          void *act_cache, void *stream) {
    TMLA_REQUIRE(params && wpack && x, "params/wpack/x must be non-NULL");
    TMLA_REQUIRE(act_cache || obs_dim <= 6, "act_cache may be NULL (inference, activations not kept) only for the fused path (obs_dim <= 6)");
    TMLA_REQUIRE(rows > 0, "rows must be positive");
    TMLA_REQUIRE(logits || values, "nothing to compute");
    int rc = check_shape(obs_dim, hidden, n_actions);
    if (rc) return rc;
    return mlp_forward_impl<__nv_bfloat16>(params, wpack, obs_dim, n_actions, x, index, rows, rows_dev, logits, values,
                                           (__nv_bfloat16 *)act_cache, (cudaStream_t)stream, act_cache != nullptr);
}

int64_t tmla_mlp_backward_scratch(int obs_dim, int hidden, int n_actions, int64_t rows) {
    if (small_width(hidden)) return small_mlp_backward_scratch(obs_dim, hidden, n_actions, rows);    // per-chunk partial gradients
    return 2 * rows * (int64_t)hidden;
}

int tmla_mlp_backward(const float *params, int obs_dim, int hidden, int n_actions, const float *x, const int32_t *index,
                      int64_t rows, const float *act_cache, const float *dlogits, const float *dvalues, float *grads,
                      float *scratch, void *stream) {
    TMLA_REQUIRE(params && x && act_cache && dlogits && dvalues && grads && scratch, "NULL buffer");
    TMLA_REQUIRE(rows > 0, "rows must be positive");
    int rc = check_shape(obs_dim, hidden, n_actions, true);
    if (rc) return rc;
    if (hidden != H)
        return small_mlp_backward(params, obs_dim, hidden, n_actions, x, index, rows, act_cache, dlogits, dvalues, grads, scratch,
                                  (cudaStream_t)stream);
    return mlp_backward_impl<float>(params, nullptr, obs_dim, n_actions, x, index, rows, act_cache, dlogits, dvalues, grads, scratch,
                                    (cudaStream_t)stream);
}

int tmla_mlp_backward_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *x,
                           const int32_t *index, int64_t rows, const void *act_cache, const float *dlogits,
                           const float *dvalues, float *grads, void *scratch, void *stream) {
    TMLA_REQUIRE(params && wpack && x && act_cache && dlogits && dvalues && grads && scratch, "NULL buffer");
    TMLA_REQUIRE(rows > 0, "rows must be positive");
    int rc = check_shape(obs_dim, hidden, n_actions);
    if (rc) return rc;
    return mlp_backward_impl<__nv_bfloat16>(params, wpack, obs_dim, n_actions, x, index, rows, (const __nv_bfloat16 *)act_cache,
                                            dlogits, dvalues, grads, (__nv_bfloat16 *)scratch, (cudaStream_t)stream);
}

int tmla_mlp_backward_bf16_det(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *x,
                               const int32_t *index, int64_t rows, const void *act_cache, const float *dlogits,
                               const float *dvalues, float *grads, void *scratch, void *partials, void *stream) {
    TMLA_REQUIRE(params && wpack && x && act_cache && dlogits && dvalues && grads && scratch && partials, "NULL buffer");
    TMLA_REQUIRE(rows > 0, "rows must be positive");
    int rc = check_shape(obs_dim, hidden, n_actions);
    if (rc) return rc;
    return mlp_backward_bf16_det(params, wpack, obs_dim, n_actions, x, index, rows, (const __nv_bfloat16 *)act_cache, dlogits, dvalues,
                                 grads, (__nv_bfloat16 *)scratch, (float *)partials, (cudaStream_t)stream);
}

int64_t tmla_det_scratch_bytes(int obs_dim, int hidden, int n_actions, int64_t rows) {
    if (rows <= 0) { tmla_set_error("rows must be positive"); return TMLA_EINVAL; }
    int64_t b = loss_det_scratch_bytes(rows);
    if (hidden == H && check_shape(obs_dim, hidden, n_actions) == TMLA_OK) b = std::max(b, backward_det_bytes(obs_dim, n_actions, rows));
    return std::max(b, fused_det_scratch_bytes(obs_dim, hidden, n_actions, rows));
}

// bf16 copies of the two hidden-layer weights per tower: wpack = [pi.W2, pi.W2^T, vf.W2, vf.W2^T, pi.W2 image, vf.W2 image],
// each 256*256 bf16 (the images are the shared-memory operand layout of csrc/mlp_train.cu)
int tmla_mlp_pack_bf16(const float *params, int obs_dim, int hidden, int n_actions, void *wpack, void *stream) {
    TMLA_REQUIRE(params && wpack, "NULL buffer");
    int rc = check_shape(obs_dim, hidden, n_actions);
    if (rc) return rc;
    const MlpOffsets o = mlp_offsets(obs_dim, n_actions);
    for (int t = 0; t < 2; ++t) {
        __nv_bfloat16 *w = reinterpret_cast<__nv_bfloat16 *>(wpack) + (int64_t)(2 * t) * H * H;
        rc = tc_pack_w2_launch(params + o.w2[t], w, w + H * H, reinterpret_cast<__nv_bfloat16 *>(wpack) + (int64_t)(4 + t) * H * H, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return TMLA_OK;
}

}  // extern "C"
