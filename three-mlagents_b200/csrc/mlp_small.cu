// mlp_small.cu — MlpPolicy with hidden width H = 64 or 128 (net_arch [H, H]; SB3's own default is [64, 64]): forward and
// backward in float32 on CUDA cores.
//
// At these widths one tower's weights fit in shared memory (H = 128: W2 is 64 KB, W1 at most 45 x 128 x 4 = 23 KB), so each
// CTA stages the weights of ONE tower once (blockIdx.y picks the tower) and then streams 32-row tiles through them:
//   forward   gather x -> tanh(x W1^T + b1) -> tanh(h1 W2^T + b2) -> head, all in shared memory, one launch for both towers;
//   backward  per 32-row tile: dZ2 = (dOut Wh) * (1 - h2^2), dW2 += dZ2^T h1 (register micro-tile), dZ1 = (dZ2 W2) * (1 - h1^2),
//             dW1 += dZ1^T x; every CTA owns a fixed contiguous chunk of rows and writes its partial gradient to scratch, a
//             second kernel sums the partials in CTA order.  No atomics: two calls on the same inputs give the same bits.
// The 256-wide network keeps its own kernels (mlp_kernels.cu fp32, mlp_tc.cu / mlp_train.cu bf16); this file serves only
// H in {64, 128}, dispatched from tmla_mlp_forward / tmla_mlp_backward.
#include <algorithm>
#include <string.h>
#include "common.cuh"
#include "mlp_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kTile = 32;          // rows per CTA tile
constexpr int kMaxOut = 5;         // widest head (n_actions <= 5; the value head is 1)
constexpr int kBwdChunks = 148;    // row chunks of the backward pass: a constant, so the summation order depends on `rows` only

template <int H>
struct Cfg {
    static constexpr int LD = H + 4;            // padded row stride (floats) of W2 and of the activation tiles
    static constexpr int TX = H / 4;            // dense passes: thread (tx, ty) owns columns tx + TX*c (c < 4) ...
    static constexpr int TY = kThreads / TX;
    static constexpr int RT = kTile / TY;       // ... of rows ty*RT + i (i < RT)
    static constexpr int G = kThreads / H;      // elementwise passes: thread (hj, hg) owns hidden unit hj, rows hg + G*i
    static constexpr int MQ = H / 64;           // dW2 micro-tile: MQ float4 quads per side (rows tj*4+64p.., cols tk*4+64q..)
};

struct SmallTower {
    const float *w1, *b1, *w2, *b2, *wh, *bh;   // this tower's parameters inside the flat vector
    float *out;                                 // forward: [rows, nout]
    float *h1, *h2;                             // act_cache planes [rows, H] (forward writes, backward reads); may be NULL in forward
    const float *dout;                          // backward: dlogits [rows, A] or dvalues [rows]
    int64_t o_w1, o_b1, o_w2, o_b2, o_wh, o_bh; // backward: offsets of the gradient slices
    int nout;
};

struct SmallArgs {
    SmallTower t[2];
    const float *x;
    const int32_t *index;
    const int32_t *rows_dev;
    int64_t rows, chunk, P;                     // P = number of parameters (row length of the partial-gradient scratch)
    float *part;
    int t0;                                     // tower of blockIdx.y == 0
};

__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }

template <int D>
__device__ __forceinline__ void load_x_tile(float *sx, const SmallArgs &a, int64_t r0, int nr) {
    for (int e = threadIdx.x; e < kTile * D; e += kThreads) {
        const int r = e / D, d = e - r * D;
        float v = 0.0f;
        if (r < nr) {
            const int64_t src = a.index ? (int64_t)a.index[r0 + r] : r0 + r;
            v = a.x[src * D + d];
        }
        sx[e] = v;
    }
}

// ------------------------------------------------------------------------------------------------ forward
template <int H, int D>
constexpr int fwd_smem_floats() {
    return H * Cfg<H>::LD + kTile * Cfg<H>::LD + H * (D | 1) + 2 * H + kMaxOut * H + 8 + kTile * D;
}

template <int H, int D>
__global__ void __launch_bounds__(kThreads, 2)
small_mlp_forward_kernel(const SmallArgs a) {
    using C = Cfg<H>;
    constexpr int LD = C::LD, LD1 = D | 1;      // odd W1 row stride: a warp's 32 hidden units read 32 different banks
    extern __shared__ __align__(16) float smem[];
    float *sW2 = smem;                          // [H][LD]   W2[j][k]
    float *sh = sW2 + H * LD;                   // [kTile][LD] h1, then h2
    float *sW1 = sh + kTile * LD;               // [H][LD1]  W1[j][d]
    float *sb1 = sW1 + H * LD1, *sb2 = sb1 + H, *sWh = sb2 + H, *sbh = sWh + kMaxOut * H, *sx = sbh + 8;
    const SmallTower tw = a.t0 + blockIdx.y == 0 ? a.t[0] : a.t[1];
    const int nout = tw.nout, tid = threadIdx.x;
    for (int e = tid; e < H * H; e += kThreads) sW2[(e / H) * LD + e % H] = tw.w2[e];
    for (int e = tid; e < H * D; e += kThreads) sW1[(e / D) * LD1 + e % D] = tw.w1[e];
    for (int e = tid; e < H; e += kThreads) { sb1[e] = tw.b1[e]; sb2[e] = tw.b2[e]; }
    for (int e = tid; e < kMaxOut * H; e += kThreads) sWh[e] = e < nout * H ? tw.wh[e] : 0.0f;
    if (tid < kMaxOut) sbh[tid] = tid < nout ? tw.bh[tid] : 0.0f;
    const int64_t rows = a.rows_dev ? min(a.rows, (int64_t)*a.rows_dev) : a.rows;
    const int tx = tid % C::TX, ty = tid / C::TX;
    const int warp = tid >> 5, lane = tid & 31;
    for (int64_t r0 = (int64_t)blockIdx.x * kTile; r0 < rows; r0 += (int64_t)gridDim.x * kTile) {
        const int nr = (int)min((int64_t)kTile, rows - r0);
        __syncthreads();                        // weights staged / previous tile's head done with sh, sx
        load_x_tile<D>(sx, a, r0, nr);
        __syncthreads();
        // layer 1
#pragma unroll
        for (int i = 0; i < C::RT; ++i) {
            const int r = ty * C::RT + i;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = tx + C::TX * c;
                float acc = sb1[j];
#pragma unroll
                for (int d = 0; d < D; ++d) acc = fmaf(sx[r * D + d], sW1[j * LD1 + d], acc);
                const float v = tanhf(acc);
                sh[r * LD + j] = v;
                if (tw.h1 && r < nr) tw.h1[(r0 + r) * H + j] = v;
            }
        }
        __syncthreads();
        // layer 2: acc[i][c] = h1[row i] . W2[col c]
        float acc[C::RT][4];
#pragma unroll
        for (int i = 0; i < C::RT; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[i][c] = 0.0f;
#pragma unroll 4
        for (int k = 0; k < H; k += 4) {
            float4 hv[C::RT], wv[4];
#pragma unroll
            for (int i = 0; i < C::RT; ++i) hv[i] = ld4(sh + (ty * C::RT + i) * LD + k);
#pragma unroll
            for (int c = 0; c < 4; ++c) wv[c] = ld4(sW2 + (tx + C::TX * c) * LD + k);
#pragma unroll
            for (int i = 0; i < C::RT; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    acc[i][c] = fmaf(hv[i].x, wv[c].x, acc[i][c]);
                    acc[i][c] = fmaf(hv[i].y, wv[c].y, acc[i][c]);
                    acc[i][c] = fmaf(hv[i].z, wv[c].z, acc[i][c]);
                    acc[i][c] = fmaf(hv[i].w, wv[c].w, acc[i][c]);
                }
        }
        __syncthreads();                        // every thread is done reading h1
#pragma unroll
        for (int i = 0; i < C::RT; ++i) {
            const int r = ty * C::RT + i;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = tx + C::TX * c;
                const float v = tanhf(acc[i][c] + sb2[j]);
                sh[r * LD + j] = v;
                if (tw.h2 && r < nr) tw.h2[(r0 + r) * H + j] = v;
            }
        }
        __syncthreads();
        // head: warp w owns rows 4w..4w+3, lanes split the hidden units, butterfly sums
        if (tw.out) {
            float s[4][kMaxOut];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int o = 0; o < kMaxOut; ++o) s[u][o] = 0.0f;
#pragma unroll
            for (int q = 0; q < H / 32; ++q) {
                const int j = lane + 32 * q;
                float hv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) hv[u] = sh[(warp * 4 + u) * LD + j];
#pragma unroll
                for (int o = 0; o < kMaxOut; ++o) {
                    if (o < nout) {
                        const float w = sWh[o * H + j];
#pragma unroll
                        for (int u = 0; u < 4; ++u) s[u][o] = fmaf(hv[u], w, s[u][o]);
                    }
                }
            }
#pragma unroll
            for (int m = 16; m > 0; m >>= 1)
#pragma unroll
                for (int u = 0; u < 4; ++u)
#pragma unroll
                    for (int o = 0; o < kMaxOut; ++o)
                        if (o < nout) s[u][o] += __shfl_xor_sync(0xffffffffu, s[u][o], m);
            if (lane == 0) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int r = warp * 4 + u;
                    if (r < nr)
#pragma unroll
                        for (int o = 0; o < kMaxOut; ++o)
                            if (o < nout) tw.out[(r0 + r) * nout + o] = s[u][o] + sbh[o];
                }
            }
        }
    }
}

// ----------------------------------------------------------------------------------------------- backward
template <int H, int D>
constexpr int bwd_smem_floats() {
    return H * Cfg<H>::LD + 2 * kTile * Cfg<H>::LD + kMaxOut * H + kTile * D + kTile * kMaxOut;
}

template <int H, int D>
__global__ void __launch_bounds__(kThreads, 2)
small_mlp_backward_kernel(const SmallArgs a) {
    using C = Cfg<H>;
    constexpr int LD = C::LD, G = C::G, MQ = C::MQ, ND = (D + G - 1) / G;
    extern __shared__ __align__(16) float smem[];
    float *sW2 = smem;                          // [H][LD]     W2[j][k]
    float *sh1 = sW2 + H * LD;                  // [kTile][LD] h1, then dZ1
    float *sh2 = sh1 + kTile * LD;              // [kTile][LD] h2, then dZ2
    float *sWh = sh2 + kTile * LD;              // [kMaxOut][H]
    float *sx = sWh + kMaxOut * H;              // [kTile][D]
    float *sd = sx + kTile * D;                 // [kTile][kMaxOut]
    const SmallTower tw = blockIdx.y == 0 ? a.t[0] : a.t[1];
    const int nout = tw.nout, tid = threadIdx.x;
    for (int e = tid; e < H * H; e += kThreads) sW2[(e / H) * LD + e % H] = tw.w2[e];
    for (int e = tid; e < kMaxOut * H; e += kThreads) sWh[e] = e < nout * H ? tw.wh[e] : 0.0f;
    const int tx = tid % C::TX, ty = tid / C::TX;           // dZ1 pass
    const int tj = tid >> 4, tk = tid & 15;                 // dW2 micro-tile
    const int hj = tid % H, hg = tid / H;                   // elementwise passes
    float gw2[4 * MQ][4 * MQ], gw1[ND], gwh[kMaxOut], gb2 = 0.0f, gbh = 0.0f, gb1 = 0.0f;
#pragma unroll
    for (int i = 0; i < 4 * MQ; ++i)
#pragma unroll
        for (int k = 0; k < 4 * MQ; ++k) gw2[i][k] = 0.0f;
#pragma unroll
    for (int i = 0; i < ND; ++i) gw1[i] = 0.0f;
#pragma unroll
    for (int o = 0; o < kMaxOut; ++o) gwh[o] = 0.0f;
    float wh[kMaxOut];
    const int64_t rb = (int64_t)blockIdx.x * a.chunk, re = min(a.rows, rb + a.chunk);
    __syncthreads();
#pragma unroll
    for (int o = 0; o < kMaxOut; ++o) wh[o] = sWh[o * H + hj];
    for (int64_t r0 = rb; r0 < re; r0 += kTile) {
        const int nr = (int)min((int64_t)kTile, re - r0);
        __syncthreads();                        // previous tile's dW1 pass done with sh1, sx
        load_x_tile<D>(sx, a, r0, nr);
        for (int e = tid; e < kTile * (H / 4); e += kThreads) {
            const int r = e / (H / 4), q = (e % (H / 4)) * 4;
            float4 v1 = make_float4(0.f, 0.f, 0.f, 0.f), v2 = v1;
            if (r < nr) { v1 = ld4(tw.h1 + (r0 + r) * H + q); v2 = ld4(tw.h2 + (r0 + r) * H + q); }
            *reinterpret_cast<float4 *>(sh1 + r * LD + q) = v1;
            *reinterpret_cast<float4 *>(sh2 + r * LD + q) = v2;
        }
        for (int e = tid; e < kTile * kMaxOut; e += kThreads) {
            const int r = e / kMaxOut, o = e % kMaxOut;
            sd[e] = (r < nr && o < nout) ? tw.dout[(r0 + r) * nout + o] : 0.0f;
        }
        __syncthreads();
        // dZ2 = (dOut . Wh) * (1 - h2^2), in place of h2;  dWh += dOut^T h2, db2 += dZ2, dbh += dOut
#pragma unroll
        for (int i = 0; i < kTile / G; ++i) {
            const int r = hg + G * i;
            const float h = sh2[r * LD + hj];
            float g = 0.0f;
#pragma unroll
            for (int o = 0; o < kMaxOut; ++o) {
                const float d = sd[r * kMaxOut + o];          // 0 beyond nout
                g = fmaf(d, wh[o], g);
                gwh[o] = fmaf(d, h, gwh[o]);
            }
            g *= 1.0f - h * h;
            sh2[r * LD + hj] = g;
            gb2 += g;
            if (hj < kMaxOut) gbh += sd[r * kMaxOut + hj];
        }
        __syncthreads();
        // dW2[j][k] += dZ2[r][j] h1[r][k]
        for (int r = 0; r < nr; ++r) {
            float z[4 * MQ], h[4 * MQ];
#pragma unroll
            for (int p = 0; p < MQ; ++p) {
                const float4 v = ld4(sh2 + r * LD + tj * 4 + 64 * p);
                z[4 * p] = v.x; z[4 * p + 1] = v.y; z[4 * p + 2] = v.z; z[4 * p + 3] = v.w;
                const float4 u = ld4(sh1 + r * LD + tk * 4 + 64 * p);
                h[4 * p] = u.x; h[4 * p + 1] = u.y; h[4 * p + 2] = u.z; h[4 * p + 3] = u.w;
            }
#pragma unroll
            for (int i = 0; i < 4 * MQ; ++i)
#pragma unroll
                for (int k = 0; k < 4 * MQ; ++k) gw2[i][k] = fmaf(z[i], h[k], gw2[i][k]);
        }
        // dH1[r][k] = sum_j dZ2[r][j] W2[j][k]
        float dh[C::RT][4];
#pragma unroll
        for (int i = 0; i < C::RT; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) dh[i][c] = 0.0f;
#pragma unroll 2
        for (int j = 0; j < H; j += 4) {
            float4 zv[C::RT];
#pragma unroll
            for (int i = 0; i < C::RT; ++i) zv[i] = ld4(sh2 + (ty * C::RT + i) * LD + j);
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float w = sW2[(j + jj) * LD + tx + C::TX * c];
#pragma unroll
                    for (int i = 0; i < C::RT; ++i) {
                        const float zz = jj == 0 ? zv[i].x : jj == 1 ? zv[i].y : jj == 2 ? zv[i].z : zv[i].w;
                        dh[i][c] = fmaf(zz, w, dh[i][c]);
                    }
                }
            }
        }
        __syncthreads();                        // every thread is done reading h1 (dW2) and dZ2
#pragma unroll
        for (int i = 0; i < C::RT; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float *p = sh1 + (ty * C::RT + i) * LD + tx + C::TX * c;
                const float h = *p;
                *p = dh[i][c] * (1.0f - h * h);
            }
        __syncthreads();
        // dW1[k][d] += dZ1[r][k] x[r][d], db1 += dZ1
        for (int r = 0; r < nr; ++r) {
            const float z = sh1[r * LD + hj];
            if (hg == 0) gb1 += z;
#pragma unroll
            for (int i = 0; i < ND; ++i) {
                const int d = hg + G * i;
                if (d < D) gw1[i] = fmaf(z, sx[r * D + d], gw1[i]);
            }
        }
    }
    // this chunk's partial gradient -> its row of the scratch (every entry of the tower's slices is written exactly once)
    float *part = a.part + (int64_t)blockIdx.x * a.P;
#pragma unroll
    for (int p = 0; p < MQ; ++p)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = tj * 4 + 64 * p + e;
#pragma unroll
            for (int q = 0; q < MQ; ++q)
#pragma unroll
                for (int f = 0; f < 4; ++f) part[tw.o_w2 + (int64_t)j * H + tk * 4 + 64 * q + f] = gw2[4 * p + e][4 * q + f];
        }
#pragma unroll
    for (int i = 0; i < ND; ++i) {
        const int d = hg + G * i;
        if (d < D) part[tw.o_w1 + (int64_t)hj * D + d] = gw1[i];
    }
    if (hg == 0) part[tw.o_b1 + hj] = gb1;
    // per-group partials of dWh, db2, dbh: combined in group order through shared memory
    __syncthreads();
    float *red = sh2;                           // [G][kMaxOut + 2][H]  (fits: G * 7 * H = 1792 floats)
#pragma unroll
    for (int o = 0; o < kMaxOut; ++o) red[(hg * (kMaxOut + 2) + o) * H + hj] = gwh[o];
    red[(hg * (kMaxOut + 2) + kMaxOut) * H + hj] = gb2;
    red[(hg * (kMaxOut + 2) + kMaxOut + 1) * H + hj] = gbh;
    __syncthreads();
    if (hg == 0) {
#pragma unroll
        for (int q = 0; q < kMaxOut + 2; ++q) {
            float s = red[q * H + hj];
#pragma unroll
            for (int g = 1; g < G; ++g) s += red[(g * (kMaxOut + 2) + q) * H + hj];
            if (q < nout) part[tw.o_wh + (int64_t)q * H + hj] = s;
            else if (q == kMaxOut) part[tw.o_b2 + hj] = s;
            else if (q == kMaxOut + 1 && hj < nout) part[tw.o_bh + hj] = s;
        }
    }
}

// grads[i] = sum over chunks c = 0, 1, ... of part[c][i]
__global__ void __launch_bounds__(256)
small_mlp_reduce_kernel(const float *__restrict__ part, int64_t P, int nchunks, float *__restrict__ grads) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.0f;
        for (int c = 0; c < nchunks; ++c) s += part[(int64_t)c * P + i];
        grads[i] = s;
    }
}

// ------------------------------------------------------------------------------------------------- host side
template <int H, int D>
struct Kernels {
    // dynamic shared memory beyond 48 KB is opt-in; blocks per SM of the forward sizes its persistent grid
    static int setup(int *fwd_blocks_per_sm) {
        static int rc = -1, nb = 1;
        if (rc < 0) {
            const size_t fs = sizeof(float) * fwd_smem_floats<H, D>(), bs = sizeof(float) * bwd_smem_floats<H, D>();
            cudaError_t e = cudaFuncSetAttribute(small_mlp_forward_kernel<H, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fs);
            if (e == cudaSuccess)
                e = cudaFuncSetAttribute(small_mlp_backward_kernel<H, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bs);
            if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, small_mlp_forward_kernel<H, D>, kThreads, fs);
            if (e != cudaSuccess) {
                tmla_set_error("mlp_small setup (H=%d, D=%d): %s", H, D, cudaGetErrorString(e));
                return TMLA_ECUDA;
            }
            rc = TMLA_OK;
            nb = std::max(nb, 1);
        }
        *fwd_blocks_per_sm = nb;
        return rc;
    }
    static int forward(const SmallArgs &a, int ntowers, cudaStream_t st) {
        int nb = 1;
        int rc = setup(&nb);
        if (rc) return rc;
        int dev = 0, sms = 148;
        TMLA_CUDA(cudaGetDevice(&dev));
        TMLA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        const int64_t tiles = ceil_div64(a.rows, kTile);
        const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)sms * nb / ntowers));
        small_mlp_forward_kernel<H, D><<<dim3(gx, ntowers), kThreads, sizeof(float) * fwd_smem_floats<H, D>(), st>>>(a);
        TMLA_LAUNCH_CHECK();
        return TMLA_OK;
    }
    static int backward(const SmallArgs &a, int nchunks, float *grads, cudaStream_t st) {
        int nb = 1;
        int rc = setup(&nb);
        if (rc) return rc;
        small_mlp_backward_kernel<H, D><<<dim3(nchunks, 2), kThreads, sizeof(float) * bwd_smem_floats<H, D>(), st>>>(a);
        TMLA_LAUNCH_CHECK();
        small_mlp_reduce_kernel<<<(unsigned)ceil_div64(a.P, 256), 256, 0, st>>>(a.part, a.P, nchunks, grads);
        TMLA_LAUNCH_CHECK();
        return TMLA_OK;
    }
};

template <int H>
int dispatch_d(bool fwd, int D, const SmallArgs &a, int n, float *grads, cudaStream_t st) {
#define SMALL_D(DD) case DD: return fwd ? Kernels<H, DD>::forward(a, n, st) : Kernels<H, DD>::backward(a, n, grads, st);
    switch (D) {
        SMALL_D(4) SMALL_D(6) SMALL_D(7) SMALL_D(16) SMALL_D(21) SMALL_D(45)
        default: break;
    }
#undef SMALL_D
    tmla_set_error("obs_dim must be 4, 6, 7, 16, 21 or 45, got %d", D);
    return TMLA_EINVAL;
}

SmallArgs make_args(const float *params, int D, int hidden, int A, const float *x, const int32_t *index, int64_t rows,
                    const float *act_cache) {
    SmallArgs a;
    memset(&a, 0, sizeof(a));
    const MlpOffsets o = mlp_offsets(D, A, hidden);
    for (int t = 0; t < 2; ++t) {
        SmallTower &tw = a.t[t];
        tw.w1 = params + o.w1[t]; tw.b1 = params + o.b1[t]; tw.w2 = params + o.w2[t]; tw.b2 = params + o.b2[t];
        tw.wh = params + o.wh[t]; tw.bh = params + o.bh[t];
        tw.o_w1 = o.w1[t]; tw.o_b1 = o.b1[t]; tw.o_w2 = o.w2[t]; tw.o_b2 = o.b2[t]; tw.o_wh = o.wh[t]; tw.o_bh = o.bh[t];
        tw.nout = o.nout[t];
        if (act_cache) {
            tw.h1 = const_cast<float *>(act_cache) + (int64_t)(2 * t) * rows * hidden;
            tw.h2 = const_cast<float *>(act_cache) + (int64_t)(2 * t + 1) * rows * hidden;
        }
    }
    a.x = x; a.index = index; a.rows = rows; a.P = o.total;
    return a;
}

// Chunk budget of the backward: min(kBwdChunks, tiles).  It never decreases with `rows`, so scratch sized for a minibatch of B
// rows also serves every shorter one (the last minibatch of an epoch); the chunks actually used, ceil(rows / chunk), never
// exceed it.  rows > 0.
int64_t bwd_chunk_budget(int64_t rows) { return std::min<int64_t>(kBwdChunks, ceil_div64(rows, kTile)); }

// rows per backward chunk (a multiple of the tile) and the number of chunks
void bwd_chunks(int64_t rows, int64_t *chunk, int *nchunks) {
    *chunk = ceil_div64(ceil_div64(rows, bwd_chunk_budget(rows)), kTile) * kTile;
    *nchunks = (int)ceil_div64(rows, *chunk);
}

}  // namespace

int small_mlp_forward(const float *params, int D, int hidden, int A, const float *x, const int32_t *index, int64_t rows,
                      const int32_t *rows_dev, float *logits, float *values, float *act_cache, cudaStream_t st) {
    SmallArgs a = make_args(params, D, hidden, A, x, index, rows, act_cache);
    a.rows_dev = rows_dev;
    a.t[0].out = logits;
    a.t[1].out = values;
    a.t0 = logits ? 0 : 1;
    const int n = (logits && values) ? 2 : 1;
    return hidden == 64 ? dispatch_d<64>(true, D, a, n, nullptr, st) : dispatch_d<128>(true, D, a, n, nullptr, st);
}

int64_t small_mlp_backward_scratch(int D, int hidden, int A, int64_t rows) {
    if (rows <= 0 || D <= 0 || A <= 0) {
        tmla_set_error("tmla_mlp_backward_scratch: rows, obs_dim and n_actions must be positive (got %lld, %d, %d)", (long long)rows, D, A);
        return TMLA_EINVAL;
    }
    return bwd_chunk_budget(rows) * mlp_offsets(D, A, hidden).total;
}

int small_mlp_backward(const float *params, int D, int hidden, int A, const float *x, const int32_t *index, int64_t rows,
                       const float *act_cache, const float *dlogits, const float *dvalues, float *grads, float *scratch,
                       cudaStream_t st) {
    SmallArgs a = make_args(params, D, hidden, A, x, index, rows, act_cache);
    a.t[0].dout = dlogits;
    a.t[1].dout = dvalues;
    a.part = scratch;
    int n;
    bwd_chunks(rows, &a.chunk, &n);
    return hidden == 64 ? dispatch_d<64>(false, D, a, n, grads, st) : dispatch_d<128>(false, D, a, n, grads, st);
}
