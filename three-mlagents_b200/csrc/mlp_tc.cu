// mlp_tc.cu — the 256x256 hidden-layer GEMMs of the policy/value MLP on the 5th-generation tensor cores
// (tcgen05.mma, accumulators in TMEM), bf16 operands, fp32 accumulation.  sm_100a only.
//
// Replaces the three [rows x 256 x 256] matrix products per tower that SB3's ActorCriticPolicy / autograd
// execute as torch CPU GEMMs (policy built at backend/mlagents/training.py:150, net_arch training.py:363-365):
//     forward   H2  = tanh(H1 . W2^T + b2)                 tc_linear_kernel<EPI_BIAS_TANH>
//     dgrad     dZ1 = (dZ2 . W2) * (1 - H1^2)              tc_linear_kernel<EPI_DTANH>   (with W2^T as weight)
//     wgrad     dW2 = dZ2^T . H1   (reduction over rows)   tc_wgrad_kernel
// The K=obs_dim first layer and the N<=5 heads stay on CUDA cores (mlp_kernels.cu, bf16 activation variants).
//
// Design (no TMA, no swizzle — operands are staged by the CTA's own threads):
//   * Operand tiles live in shared memory in the canonical K-major SWIZZLE_NONE layout of the UMMA shared
//     memory descriptor: 8-row x 16-byte "core matrices" stored as 128 contiguous bytes; LBO = byte stride
//     between core matrices adjacent in K, SBO = byte stride between 8-row groups
//     (element (r,k) at (r/8)*SBO + (k/8)*LBO + (r%8)*16 + (k%8)*2).
//   * One thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=256, K=16 per instruction) and
//     tcgen05.commit -> mbarrier; everybody waits on the mbarrier, then the 8 warps drain TMEM with
//     tcgen05.ld.32x32b.x16 (thread = accumulator row) and apply the fused epilogue.
//   * The 256x256 weight stays resident in shared memory for the whole persistent CTA (one CTA per SM).
//   * wgrad transposes its operands while staging them (8x8 bf16 blocks through PRMT) so that the same
//     K-major descriptors apply, accumulates 256x256 fp32 in all 512 TMEM columns across the CTA's row
//     chunks, and finishes with red.global.add.f32 into the flat gradient (split-K over CTAs).
#include <algorithm>
#include <cuda_bf16.h>
#include "common.cuh"
#include "tc_common.cuh"

__device__ int g_desc_swap = 0;      // debug: exchange the LBO/SBO fields (tmla_tc_debug)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    if (g_desc_swap) { const uint32_t t = lbo; lbo = sbo; sbo = t; }
    return make_desc_raw(saddr, lbo, sbo);
}

// -------------------------------------------------------------------- out = epi(A[M,256] . W[256,256]^T)
enum { EPI_BIAS_TANH = 0, EPI_DTANH = 1 };

static constexpr uint32_t kLinearSmem = kWBytes + kABytes + 64;

__device__ __forceinline__ uint4 mul_dtanh(const uint4 &v, const uint4 &h) {   // v * (1 - h^2), 8 bf16 lanes
    const uint32_t vv[4] = {v.x, v.y, v.z, v.w}, hh[4] = {h.x, h.y, h.z, h.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float a = bf16_lo(hh[j]), b = bf16_hi(hh[j]);
        o[j] = pack_bf16(bf16_lo(vv[j]) * (1.0f - a * a), bf16_hi(vv[j]) * (1.0f - b * b));
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// Per 128-row tile:  registers(prefetched A) -> smem (K-major) -> 16 x tcgen05.mma -> TMEM -> registers ->
// smem stage (XOR-swizzled rows) -> coalesced 512-byte row stores.  The A tile of the NEXT row block (and the
// dgrad epilogue's 1-h^2 operand) are prefetched into registers right after the MMAs have been issued, so
// global-load latency overlaps the tensor-core work and the epilogue.  All global traffic is issued as full
// 512-byte rows per warp (4 L1 wavefronts per request).
template <int EPI>
__global__ void __launch_bounds__(256, 1)
tc_linear_kernel(const __nv_bfloat16 *__restrict__ A, const __nv_bfloat16 *__restrict__ W, const float *__restrict__ bias,
                 const __nv_bfloat16 *__restrict__ aux, __nv_bfloat16 *__restrict__ out, int64_t M, const int32_t *rows_dev) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *Ws = smem, *As = smem + kWBytes;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kWBytes + kABytes);
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + kWBytes + kABytes + 16);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (rows_dev) M = min(M, (int64_t)*rows_dev);
    const int64_t ntiles = (M + 127) / 128;
    if ((int64_t)blockIdx.x >= ntiles) return;            // whole CTA exits before any allocation

    // this thread's 16 chunks of a tile: row r = warp + 8*i, 16-byte chunk `lane` of that row
    uint4 pre[16];
    auto prefetch = [&](int64_t tile) {
        const int64_t row0 = tile * 128, nvalid = M - row0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int r = warp + 8 * i;
            pre[i] = (r < nvalid) ? __ldg(reinterpret_cast<const uint4 *>(A + (row0 + r) * H) + lane) : make_uint4(0u, 0u, 0u, 0u);
        }
    };
    prefetch(blockIdx.x);

    if (warp == 0) tmem_alloc<256>(tmem_holder);
    if (tid == 32) { mbar_init(bar, 1); fence_barrier_init(); }
    stage_rows<H>(Ws, W, 0, H);                           // resident weight: W[n][k], K-major
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    const uint32_t idesc = make_idesc(128, 256);
    const uint32_t a_addr = smem_u32(As), w_addr = smem_u32(Ws);
    uint32_t phase = 0;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * 128;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int r = warp + 8 * i;
            *reinterpret_cast<uint4 *>(As + (r >> 3) * kaSBO + lane * kaLBO + (r & 7) * 16) = pre[i];
        }
        fence_proxy_async();                              // generic-proxy smem writes -> visible to the tensor core
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
#pragma unroll
            for (int kk = 0; kk < H / 16; ++kk)           // 16 MMAs of K=16: two core matrices along K each
                umma_bf16(tmem_base, make_desc(a_addr + kk * 2 * kaLBO, kaLBO, kaSBO), make_desc(w_addr + kk * 2 * kLBO, kLBO, kSBO),
                          idesc, kk > 0 ? 1u : 0u);
            umma_commit(bar);                             // arrives on `bar` when all MMAs above have finished
        }
        if (tile + gridDim.x < ntiles) prefetch(tile + gridDim.x);   // in flight during the MMAs and the epilogue
        uint4 hx[EPI == EPI_DTANH ? 16 : 1];
        if (EPI == EPI_DTANH) {                           // same (row, chunk) mapping as the copy-out below
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int64_t r = row0 + warp + 8 * i;
                hx[i] = (r < M) ? __ldg(reinterpret_cast<const uint4 *>(aux + r * H) + lane) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
        mbar_wait(bar, phase);
        phase ^= 1u;
        tc_fence_after();
        // TMEM -> registers -> stage.  warp w drains lanes 32*(w%4).. of columns (w/4)*128..+127; thread = one row.
        // stage layout: row-major 512 B rows, 16-byte chunk c of row r stored at chunk (c ^ (r & 7)).
        {
            const int rt = (warp & 3) * 32 + lane;        // row inside the tile
            const int colbase = (warp >> 2) * 128;
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)colbase;
            uint8_t *srow = As + rt * 512;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint32_t acc[16];
                tmem_ld16(taddr + c * 16, acc);
                const int col = colbase + c * 16;
                uint32_t o[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float v0 = __uint_as_float(acc[2 * j]), v1 = __uint_as_float(acc[2 * j + 1]);
                    if (EPI == EPI_BIAS_TANH) {
                        v0 = tanh_fast(v0 + __ldg(bias + col + 2 * j));
                        v1 = tanh_fast(v1 + __ldg(bias + col + 2 * j + 1));
                    }
                    o[j] = pack_bf16(v0, v1);
                }
                const int ch = col >> 3;                  // first of two 16-byte chunks
                *reinterpret_cast<uint4 *>(srow + ((ch ^ (rt & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<uint4 *>(srow + (((ch + 1) ^ (rt & 7)) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
            }
        }
        tc_fence_before();
        __syncthreads();                                  // stage complete, TMEM drained
#pragma unroll
        for (int i = 0; i < 16; ++i) {                    // coalesced copy-out: a warp writes one full 512-byte row
            const int r = warp + 8 * i;
            uint4 v = *reinterpret_cast<const uint4 *>(As + r * 512 + ((lane ^ (r & 7)) << 4));
            if (EPI == EPI_DTANH) v = mul_dtanh(v, hx[i]);
            if (row0 + r < M) reinterpret_cast<uint4 *>(out + (row0 + r) * H)[lane] = v;
        }
        __syncthreads();                                  // As free for the next tile
    }
    if (warp == 0) tmem_dealloc<256>(tmem_base);
}

// --------------------------------------------------------- G[256,256] += X[rows,256]^T . Y[rows,256]
// 64-row chunks, two shared-memory stages and two chunks of register prefetch: while the tensor core works on
// stage s the threads transpose and stage the next chunk into stage s^1, and the loads of the chunk after that
// are already in flight (per-stage mbarriers signal "MMAs done reading").
static constexpr int kgRows = 64;                        // rows (= K) per chunk
static constexpr uint32_t kgLBO = 128;
static constexpr uint32_t kgSBO = (kgRows / 8) * kgLBO + 16;   // 1040: 8 k-blocks per 8-row group + 16 B pad (bank spread)
static constexpr uint32_t kgTile = 32 * kgSBO;           // 33280 B: 256 rows x K=64
static constexpr uint32_t kgStage = 2 * kgTile;          // X and Y tiles
static constexpr uint32_t kWgradSmem = 2 * kgStage + 64; // 133184 (>= 128 KB epilogue stage)

// thread = one 8x8 block of the chunk (k-block = warp, m-group = lane): 8 LDG.128 (a warp reads 512 contiguous
// bytes per row), 32 PRMT, 8 STS.128 into the K-major tile [256 (m) x 64 (k)]
__device__ __forceinline__ void load_block(uint4 (&in)[8], const __nv_bfloat16 *__restrict__ src, int64_t row0, int64_t nvalid) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int r = warp * 8 + i;
        in[i] = (r < nvalid) ? __ldg(reinterpret_cast<const uint4 *>(src + (row0 + r) * H + lane * 8)) : make_uint4(0u, 0u, 0u, 0u);
    }
}
__device__ __forceinline__ void store_block_transposed(uint8_t *dst, const uint4 (&in)[8]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *base = dst + lane * kgSBO + warp * kgLBO;
#pragma unroll
    for (int c = 0; c < 8; ++c) {                         // output row c = column lane*8+c over the 8 source rows
        const uint32_t sel = (c & 1) ? 0x7632u : 0x5410u;
        uint32_t w[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const uint32_t a = (c >> 1) == 0 ? in[2 * p].x : ((c >> 1) == 1 ? in[2 * p].y : ((c >> 1) == 2 ? in[2 * p].z : in[2 * p].w));
            const uint32_t b = (c >> 1) == 0 ? in[2 * p + 1].x : ((c >> 1) == 1 ? in[2 * p + 1].y : ((c >> 1) == 2 ? in[2 * p + 1].z : in[2 * p + 1].w));
            w[p] = __byte_perm(a, b, sel);
        }
        *reinterpret_cast<uint4 *>(base + c * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// DET: G is an array of 256x256 partial planes, CTA b stores its split-K share in plane b (summed in order by det_reduce_kernel)
template <bool DET = false>
__global__ void __launch_bounds__(256, 1)
tc_wgrad_kernel(const __nv_bfloat16 *__restrict__ X, const __nv_bfloat16 *__restrict__ Y, float *__restrict__ G, int64_t rows) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + 2 * kgStage);        // bar[0], bar[1]
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + 2 * kgStage + 32);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t nchunks = (rows + kgRows - 1) / kgRows;
    if ((int64_t)blockIdx.x >= nchunks) return;

    if (warp == 0) tmem_alloc<512>(tmem_holder);
    if (tid == 32) { mbar_init(bar, 1); mbar_init(bar + 1, 1); fence_barrier_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    const uint32_t idesc = make_idesc(128, 256);
    uint32_t ph[2] = {0u, 0u};
    // software pipeline: (xa,ya) = chunk being staged now, (xb,yb) = the one after (loads in flight)
    uint4 xa[8], ya[8], xb[8], yb[8];
    const int64_t stride = gridDim.x;
    int64_t chunk = blockIdx.x;
    load_block(xa, X, chunk * kgRows, rows - chunk * kgRows);
    load_block(ya, Y, chunk * kgRows, rows - chunk * kgRows);
    if (chunk + stride < nchunks) {
        load_block(xb, X, (chunk + stride) * kgRows, rows - (chunk + stride) * kgRows);
        load_block(yb, Y, (chunk + stride) * kgRows, rows - (chunk + stride) * kgRows);
    }
    int it = 0;
    for (; chunk < nchunks; chunk += stride, ++it) {
        const int s = it & 1;
        if (it >= 2) { mbar_wait(bar + s, ph[s]); ph[s] ^= 1u; }   // MMAs of chunk it-2 have finished reading stage s
        uint8_t *Xs = smem + s * kgStage, *Ys = Xs + kgTile;
        store_block_transposed(Xs, xa);
        store_block_transposed(Ys, ya);
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const uint32_t x_addr = smem_u32(Xs), y_addr = smem_u32(Ys);
#pragma unroll
            for (int mh = 0; mh < 2; ++mh)                // output rows 0..127 / 128..255 -> TMEM columns 0..255 / 256..511
#pragma unroll
                for (int kk = 0; kk < kgRows / 16; ++kk)
                    umma_bf16(tmem_base + mh * 256, make_desc(x_addr + mh * 16 * kgSBO + kk * 2 * kgLBO, kgLBO, kgSBO),
                              make_desc(y_addr + kk * 2 * kgLBO, kgLBO, kgSBO), idesc, (it == 0 && kk == 0) ? 0u : 1u);
            umma_commit(bar + s);
        }
        // rotate the register pipeline and launch the loads two chunks ahead
#pragma unroll
        for (int i = 0; i < 8; ++i) { xa[i] = xb[i]; ya[i] = yb[i]; }
        const int64_t nxt = chunk + 2 * stride;
        if (nxt < nchunks) {
            load_block(xb, X, nxt * kgRows, rows - nxt * kgRows);
            load_block(yb, Y, nxt * kgRows, rows - nxt * kgRows);
        }
    }
    const int last = (it - 1) & 1;                        // every commit on bar[last] but the newest has been waited for
    mbar_wait(bar + last, ph[last]);
    tc_fence_after();
    // epilogue: TMEM -> registers -> smem stage (fp32 [128][256], 16-byte chunks XOR-swizzled by row) ->
    // coalesced red.global.add.v4.f32 (split-K reduction over CTAs): a warp adds one 1 KB row in two requests
#pragma unroll 1
    for (int mh = 0; mh < 2; ++mh) {
        __syncthreads();                                  // previous half fully flushed / MMAs done with smem
        {
            const int rt = (warp & 3) * 32 + lane;
            const int colbase = (warp >> 2) * 128;
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mh * 256 + colbase);
            uint8_t *srow = smem + rt * 1024;
#pragma unroll 2
            for (int c0 = 0; c0 < 128; c0 += 16) {
                uint32_t acc[16];
                tmem_ld16(taddr + c0, acc);
                const int ch = (colbase + c0) >> 2;       // first of four 16-byte chunks (4 floats each)
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
            if constexpr (DET) grow += (int64_t)blockIdx.x * (H * H);
#pragma unroll
            for (int hseg = 0; hseg < 2; ++hseg) {
                const int ch = hseg * 32 + lane;
                const float4 v = *reinterpret_cast<const float4 *>(smem + r * 1024 + ((ch ^ (r & 7)) << 4));
                if constexpr (DET) *reinterpret_cast<float4 *>(grow + ch * 4) = v;
                else asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(grow + ch * 4), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------- fused forward of one tower
//   out[r] = head( tanh( tanh(x[r] W1^T + b1) W2^T + b2 ) )          (ActorCriticPolicy.forward, one tower)
// Per 128-row tile: gather obs rows -> layer 1 on CUDA cores straight into the K-major shared-memory operand
// (H1 never round-trips HBM for the GEMM) -> 16 x tcgen05.mma against the resident W2 -> TMEM -> epilogue
// (bias, tanh, head dot products from registers) -> logits/values; H1/H2 are written out (coalesced) only
// when the caller keeps them for the backward pass.  The next tile's obs rows are prefetched into registers
// while the MMAs run.
static constexpr int kTowerThreads = 512;                 // 16 warps: 4 per SM sub-partition (latency hiding)
template <int D, int NOUT>
struct TowerSmem {
    static constexpr uint32_t w = 0;                                   // W2 bf16, K-major (kLBO/kSBO)
    static constexpr uint32_t a = kWBytes;                             // H1 tile, K-major padded (kaLBO/kaSBO); H2 stage
    static constexpr uint32_t w1 = a + kABytes;                        // float [256][D]
    static constexpr uint32_t b1 = w1 + H * D * 4;                     // float [256]
    static constexpr uint32_t b2 = b1 + H * 4;                         // float [256]
    static constexpr uint32_t wh = b2 + H * 4;                         // float [NOUT][256]
    static constexpr uint32_t xs = wh + NOUT * H * 4;                  // float [128][D]
    static constexpr uint32_t part = xs + 128 * D * 4;                 // float [3][128][NOUT] partial head sums of column quarters 1..3
    static constexpr uint32_t bar = (part + 3 * 128 * NOUT * 4 + 15) & ~15u;
    static constexpr uint32_t total = bar + 64;
};

// bid / nblk: this CTA's index and the number of CTAs working on THIS tower (the dual launch gives even CTAs to the policy
// tower and odd CTAs to the value tower)
template <int D, int NOUT>
__device__ __forceinline__ void
tower_forward_body(const float *__restrict__ W1, const float *__restrict__ B1, const __nv_bfloat16 *__restrict__ W2,
                   const float *__restrict__ B2, const float *__restrict__ Wh, const float *__restrict__ Bh,
                   const float *__restrict__ x, const int32_t *__restrict__ index, int64_t M, const int32_t *rows_dev,
                   float *__restrict__ out, __nv_bfloat16 *__restrict__ h1_out, __nv_bfloat16 *__restrict__ h2_out,
                   const int64_t bid, const int64_t nblk) {
    using L = TowerSmem<D, NOUT>;
    constexpr int NT = kTowerThreads, NW = NT / 32;        // 16 warps
    constexpr int RPW = 128 / NW;                          // rows per warp in the row-parallel phases (8)
    constexpr int XPT = (128 * D + NT - 1) / NT;           // gathered obs elements per thread per tile
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *Ws = smem + L::w, *As = smem + L::a;
    float *w1s = reinterpret_cast<float *>(smem + L::w1), *b1s = reinterpret_cast<float *>(smem + L::b1);
    float *b2s = reinterpret_cast<float *>(smem + L::b2), *whs = reinterpret_cast<float *>(smem + L::wh);
    float *xs = reinterpret_cast<float *>(smem + L::xs), *part = reinterpret_cast<float *>(smem + L::part);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::bar);
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(smem + L::bar + 16);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (rows_dev) M = min(M, (int64_t)*rows_dev);
    const int64_t ntiles = (M + 127) / 128;
    if (bid >= ntiles) return;

    float xpre[XPT];
    auto prefetch_x = [&](int64_t tile) {                  // element e = tid + NT*i of the [128][D] obs tile
        const int64_t row0 = tile * 128;
#pragma unroll
        for (int i = 0; i < XPT; ++i) {
            const int e = tid + NT * i, r = e / D, k = e - r * D;
            float v = 0.0f;
            if (e < 128 * D && row0 + r < M) {
                const int64_t src = index ? (int64_t)__ldg(index + row0 + r) : row0 + r;
                v = __ldg(x + src * D + k);
            }
            xpre[i] = v;
        }
    };
    prefetch_x(bid);

    if (warp == 0) tmem_alloc<256>(tmem_holder);
    uint64_t *barw = bar + 1;                              // W2 (given as its operand image, mlp_tc.cu:pack_w2_kernel) landing
    if (tid == 32) {
        mbar_init(bar, 1); mbar_init(barw, 1); fence_barrier_init();
        mbar_expect_tx(barw, kWBytes); bulk_load(smem_u32(Ws), W2, kWBytes, barw);   // one bulk-TMA load, overlaps the rest of the prologue
    }
    bool w2_pending = true;
    for (int e = tid; e < H * D; e += NT) w1s[e] = W1[e];
    for (int e = tid; e < NOUT * H; e += NT) whs[e] = Wh[e];
    if (tid < H) { b1s[tid] = B1[tid]; b2s[tid] = B2[tid]; }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    const uint32_t idesc = make_idesc(128, 256);
    const uint32_t a_addr = smem_u32(As), w_addr = smem_u32(Ws);
    uint32_t phase = 0;
    // layer-1 weights of this thread's 8 hidden units (k-block `lane`)
    float w1r[8][D], b1r[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        b1r[c] = b1s[lane * 8 + c];
#pragma unroll
        for (int k = 0; k < D; ++k) w1r[c][k] = w1s[(lane * 8 + c) * D + k];
    }

    for (int64_t tile = bid; tile < ntiles; tile += nblk) {
        const int64_t row0 = tile * 128;
#pragma unroll
        for (int i = 0; i < XPT; ++i) { const int e = tid + NT * i; if (e < 128 * D) xs[e] = xpre[i]; }
        __syncthreads();                                   // obs tile staged; previous tile's stage fully copied out
        // ---- layer 1: rows warp+NW*i, hidden units 8*lane..8*lane+7 -> bf16 chunk (r, kb=lane) of the K-major tile
#pragma unroll 2
        for (int i = 0; i < RPW; ++i) {
            const int r = warp + NW * i;
            float xr[D];
#pragma unroll
            for (int k = 0; k < D; ++k) xr[k] = xs[r * D + k];
            uint32_t o[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float v0 = b1r[2 * c], v1 = b1r[2 * c + 1];
#pragma unroll
                for (int k = 0; k < D; ++k) { v0 = fmaf(xr[k], w1r[2 * c][k], v0); v1 = fmaf(xr[k], w1r[2 * c + 1][k], v1); }
                o[c] = pack_bf16(tanh_fast(v0), tanh_fast(v1));
            }
            *reinterpret_cast<uint4 *>(As + (r >> 3) * kaSBO + lane * kaLBO + (r & 7) * 16) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            if (w2_pending) { mbar_wait(barw, 0); w2_pending = false; }
            tc_fence_after();
#pragma unroll
            for (int kk = 0; kk < H / 16; ++kk)
                umma_bf16(tmem_base, make_desc(a_addr + kk * 2 * kaLBO, kaLBO, kaSBO), make_desc(w_addr + kk * 2 * kLBO, kLBO, kSBO),
                          idesc, kk > 0 ? 1u : 0u);
            umma_commit(bar);
        }
        if (h1_out) {                                      // keep H1 for the backward pass: coalesced rows, overlaps the MMAs
#pragma unroll 2
            for (int i = 0; i < RPW; ++i) {
                const int r = warp + NW * i;
                const uint4 v = *reinterpret_cast<const uint4 *>(As + (r >> 3) * kaSBO + lane * kaLBO + (r & 7) * 16);
                if (row0 + r < M) reinterpret_cast<uint4 *>(h1_out + (row0 + r) * H)[lane] = v;
            }
        }
        if (tile + nblk < ntiles) prefetch_x(tile + nblk);   // dependent index->obs loads, hidden behind the MMAs
        mbar_wait(bar, phase);
        phase ^= 1u;
        tc_fence_after();
        // ---- epilogue: thread = row rt, column quarter (warp>>2): bias + tanh, head partial dots, H2 stage
        const int rt = (warp & 3) * 32 + lane;
        const int cq = warp >> 2;
        const int colbase = cq * 64;
        float hsum[NOUT];
#pragma unroll
        for (int a = 0; a < NOUT; ++a) hsum[a] = 0.0f;
        {
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)colbase;
            uint8_t *srow = As + rt * 512;
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
                uint32_t acc[16];
                tmem_ld16(taddr + c * 16, acc);
                const int col = colbase + c * 16;
                float hv[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 bb = *reinterpret_cast<const float4 *>(b2s + col + 4 * q);
                    hv[4 * q + 0] = tanh_fast(__uint_as_float(acc[4 * q + 0]) + bb.x);
                    hv[4 * q + 1] = tanh_fast(__uint_as_float(acc[4 * q + 1]) + bb.y);
                    hv[4 * q + 2] = tanh_fast(__uint_as_float(acc[4 * q + 2]) + bb.z);
                    hv[4 * q + 3] = tanh_fast(__uint_as_float(acc[4 * q + 3]) + bb.w);
                }
#pragma unroll
                for (int a = 0; a < NOUT; ++a)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 ww = *reinterpret_cast<const float4 *>(whs + a * H + col + 4 * q);
                        hsum[a] = fmaf(hv[4 * q + 0], ww.x, hsum[a]); hsum[a] = fmaf(hv[4 * q + 1], ww.y, hsum[a]);
                        hsum[a] = fmaf(hv[4 * q + 2], ww.z, hsum[a]); hsum[a] = fmaf(hv[4 * q + 3], ww.w, hsum[a]);
                    }
                if (h2_out) {
                    uint32_t o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = pack_bf16(hv[2 * j], hv[2 * j + 1]);
                    const int ch = col >> 3;
                    *reinterpret_cast<uint4 *>(srow + ((ch ^ (rt & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
                    *reinterpret_cast<uint4 *>(srow + (((ch + 1) ^ (rt & 7)) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
                }
            }
        }
        if (cq > 0) {
#pragma unroll
            for (int a = 0; a < NOUT; ++a) part[((cq - 1) * 128 + rt) * NOUT + a] = hsum[a];
        }
        tc_fence_before();
        __syncthreads();                                   // stage + partial sums complete, TMEM drained
        if (cq == 0 && row0 + rt < M) {
#pragma unroll
            for (int a = 0; a < NOUT; ++a)
                out[(row0 + rt) * NOUT + a] = ((hsum[a] + part[rt * NOUT + a]) + (part[(128 + rt) * NOUT + a] + part[(256 + rt) * NOUT + a])) + __ldg(Bh + a);
        }
        if (h2_out) {
#pragma unroll 2
            for (int i = 0; i < RPW; ++i) {
                const int r = warp + NW * i;
                const uint4 v = *reinterpret_cast<const uint4 *>(As + r * 512 + ((lane ^ (r & 7)) << 4));
                if (row0 + r < M) reinterpret_cast<uint4 *>(h2_out + (row0 + r) * H)[lane] = v;
            }
        }
        // the __syncthreads at the top of the next iteration orders these stage reads before the next H1 stores
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc<256>(tmem_base);
}

template <int D, int NOUT>
__global__ void __launch_bounds__(kTowerThreads, 1)
tc_tower_forward_kernel(const float *__restrict__ W1, const float *__restrict__ B1, const __nv_bfloat16 *__restrict__ W2,
                        const float *__restrict__ B2, const float *__restrict__ Wh, const float *__restrict__ Bh,
                        const float *__restrict__ x, const int32_t *__restrict__ index, int64_t M, const int32_t *rows_dev,
                        float *__restrict__ out, __nv_bfloat16 *__restrict__ h1_out, __nv_bfloat16 *__restrict__ h2_out) {
    tower_forward_body<D, NOUT>(W1, B1, W2, B2, Wh, Bh, x, index, M, rows_dev, out, h1_out, h2_out, blockIdx.x, gridDim.x);
}

// Both towers of a policy step in ONE launch: 2 x 512 tiles over 74 + 74 CTAs are 7 rounds instead of 4 + 4, and one kernel
// boundary per step less.  Same per-tower code; the branch is uniform per CTA.
struct TowerFwdArgs {
    const float *W1, *B1; const __nv_bfloat16 *W2; const float *B2, *Wh, *Bh; float *out; __nv_bfloat16 *h1_out, *h2_out;
};
template <int D, int A>
__global__ void __launch_bounds__(kTowerThreads, 1)
tc_tower_forward_dual_kernel(const __grid_constant__ TowerFwdArgs pi, const __grid_constant__ TowerFwdArgs vf, const float *__restrict__ x,
                             const int32_t *__restrict__ index, int64_t M, const int32_t *rows_dev) {
    const int64_t bid = blockIdx.x >> 1, nblk = gridDim.x >> 1;
    if (blockIdx.x & 1) tower_forward_body<D, 1>(vf.W1, vf.B1, vf.W2, vf.B2, vf.Wh, vf.Bh, x, index, M, rows_dev, vf.out, vf.h1_out, vf.h2_out, bid, nblk);
    else tower_forward_body<D, A>(pi.W1, pi.B1, pi.W2, pi.B2, pi.Wh, pi.Bh, x, index, M, rows_dev, pi.out, pi.h1_out, pi.h2_out, bid, nblk);
}

// ------------------------------------------------------------------------------- small helper kernels
__global__ void f32_to_bf16_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __float2bfloat16_rn(src[i]);
}
// W2 [out][in] fp32 -> bf16 copy, bf16 transpose ([in][out]) for the unfused dgrad GEMM, and the 128 KB shared-memory
// operand IMAGE (16-byte chunk (j, kb) at (j/8)*4096 + kb*128 + (j%8)*16) that the fused training kernel pulls in with
// one bulk-TMA load
__global__ void pack_w2_kernel(const float *__restrict__ w2, __nv_bfloat16 *__restrict__ w, __nv_bfloat16 *__restrict__ wt,
                               __nv_bfloat16 *__restrict__ img) {
    __shared__ float tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const float v = w2[(by + j) * H + bx + threadIdx.x];
        tile[j][threadIdx.x] = v;
        w[(by + j) * H + bx + threadIdx.x] = __float2bfloat16_rn(v);
        const int r = by + j, k = bx + threadIdx.x;
        img[(r >> 3) * 2048 + (k >> 3) * 64 + (r & 7) * 8 + (k & 7)] = __float2bfloat16_rn(v);
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) wt[(bx + j) * H + by + threadIdx.x] = __float2bfloat16_rn(tile[threadIdx.x][j]);
}

static int g_attr_done = 0;
static int ensure_attrs() {
    if (g_attr_done) return TMLA_OK;
    TMLA_CUDA(cudaFuncSetAttribute(tc_linear_kernel<EPI_BIAS_TANH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLinearSmem));
    TMLA_CUDA(cudaFuncSetAttribute(tc_linear_kernel<EPI_DTANH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLinearSmem));
    TMLA_CUDA(cudaFuncSetAttribute(tc_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWgradSmem));
    TMLA_CUDA(cudaFuncSetAttribute(tc_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWgradSmem));
    g_attr_done = 1;
    return TMLA_OK;
}
static int sm_count() {
    static int n = 0;
    if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = 148; }
    return n;
}

// launchers shared with mlp_kernels.cu
int tc_linear_launch(int epi, const void *A, const void *W, const float *bias, const void *aux, void *out, int64_t M,
                     const int32_t *rows_dev, cudaStream_t st) {
    int rc = ensure_attrs();
    if (rc) return rc;
    const unsigned grid = (unsigned)std::min<int64_t>((M + 127) / 128, sm_count());
    if (epi == EPI_BIAS_TANH)
        tc_linear_kernel<EPI_BIAS_TANH><<<grid, 256, kLinearSmem, st>>>((const __nv_bfloat16 *)A, (const __nv_bfloat16 *)W, bias,
                                                                        (const __nv_bfloat16 *)aux, (__nv_bfloat16 *)out, M, rows_dev);
    else
        tc_linear_kernel<EPI_DTANH><<<grid, 256, kLinearSmem, st>>>((const __nv_bfloat16 *)A, (const __nv_bfloat16 *)W, bias,
                                                                    (const __nv_bfloat16 *)aux, (__nv_bfloat16 *)out, M, rows_dev);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
int tc_wgrad_launch(const void *X, const void *Y, float *G, int64_t rows, cudaStream_t st) {
    int rc = ensure_attrs();
    if (rc) return rc;
    const unsigned grid = (unsigned)std::min<int64_t>((rows + kgRows - 1) / kgRows, sm_count());
    tc_wgrad_kernel<false><<<grid, 256, kWgradSmem, st>>>((const __nv_bfloat16 *)X, (const __nv_bfloat16 *)Y, G, rows);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
// deterministic form: one partial plane per CTA into `planes` (tc_wgrad_det_planes(rows) of them, all written)
int64_t tc_wgrad_det_planes(int64_t rows) { return std::min<int64_t>((rows + kgRows - 1) / kgRows, sm_count()); }
int tc_wgrad_det_launch(const void *X, const void *Y, float *planes, int64_t rows, cudaStream_t st) {
    int rc = ensure_attrs();
    if (rc) return rc;
    tc_wgrad_kernel<true><<<(unsigned)tc_wgrad_det_planes(rows), 256, kWgradSmem, st>>>((const __nv_bfloat16 *)X, (const __nv_bfloat16 *)Y, planes, rows);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
template <int D, int NOUT>
static int tower_forward_launch_t(const float *W1, const float *B1, const void *W2, const float *B2, const float *Wh, const float *Bh,
                                  const float *x, const int32_t *index, int64_t M, const int32_t *rows_dev, float *out, void *h1,
                                  void *h2, cudaStream_t st) {
    static int attr_done = 0;
    constexpr uint32_t smem = TowerSmem<D, NOUT>::total;
    static_assert(smem <= 232448, "fused tower kernel exceeds the 227 KB shared-memory limit");
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_tower_forward_kernel<D, NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = 1;
    }
    const unsigned grid = (unsigned)std::min<int64_t>((M + 127) / 128, sm_count());
    tc_tower_forward_kernel<D, NOUT><<<grid, kTowerThreads, smem, st>>>(W1, B1, (const __nv_bfloat16 *)W2, B2, Wh, Bh, x, index, M, rows_dev, out,
                                                              (__nv_bfloat16 *)h1, (__nv_bfloat16 *)h2);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
template <int D, int A>
static int tower_forward_dual_launch_t(const TowerFwdArgs &pi, const TowerFwdArgs &vf, const float *x, const int32_t *index, int64_t M,
                                       const int32_t *rows_dev, cudaStream_t st) {
    static int attr_done = 0;
    constexpr uint32_t smem = TowerSmem<D, A>::total > TowerSmem<D, 1>::total ? TowerSmem<D, A>::total : TowerSmem<D, 1>::total;
    static_assert(smem <= 232448, "fused tower kernel exceeds the 227 KB shared-memory limit");
    if (!attr_done) {
        TMLA_CUDA(cudaFuncSetAttribute(tc_tower_forward_dual_kernel<D, A>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = 1;
    }
    const unsigned grid = (unsigned)std::min<int64_t>(2 * ((M + 127) / 128), sm_count() & ~1);
    tc_tower_forward_dual_kernel<D, A><<<grid, kTowerThreads, smem, st>>>(pi, vf, x, index, M, rows_dev);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
// both towers in one launch (policy step of a rollout); W1/B1/W2/B2/Wh/Bh/out/h1/h2 as [2] arrays: policy, value
int tc_tower_forward_dual_launch(int D, int n_actions, const float *const *W1, const float *const *B1, const void *const *W2,
                                 const float *const *B2, const float *const *Wh, const float *const *Bh, const float *x,
                                 const int32_t *index, int64_t M, const int32_t *rows_dev, float *const *out, void *const *h1,
                                 void *const *h2, cudaStream_t st) {
    TowerFwdArgs a[2];
    for (int t = 0; t < 2; ++t)
        a[t] = TowerFwdArgs{W1[t], B1[t], (const __nv_bfloat16 *)W2[t], B2[t], Wh[t], Bh[t], out[t], (__nv_bfloat16 *)h1[t], (__nv_bfloat16 *)h2[t]};
#define TFD(DD, AA) if (D == DD && n_actions == AA) return tower_forward_dual_launch_t<DD, AA>(a[0], a[1], x, index, M, rows_dev, st)
    TFD(6, 5); TFD(4, 5); TFD(4, 4);
#undef TFD
    return TMLA_EINVAL;
}
// fused tower forward for the shapes of the four tasks; returns TMLA_EINVAL for an unsupported (D, NOUT)
int tc_tower_forward_launch(int D, int nout, const float *W1, const float *B1, const void *W2, const float *B2, const float *Wh,
                            const float *Bh, const float *x, const int32_t *index, int64_t M, const int32_t *rows_dev, float *out,
                            void *h1, void *h2, cudaStream_t st) {
#define TF(DD, NN) if (D == DD && nout == NN) return tower_forward_launch_t<DD, NN>(W1, B1, W2, B2, Wh, Bh, x, index, M, rows_dev, out, h1, h2, st)
    TF(6, 5); TF(6, 1); TF(4, 5); TF(4, 4); TF(4, 1);
#undef TF
    return TMLA_EINVAL;
}

int tc_pack_w2_launch(const float *w2, void *w, void *wt, void *img, cudaStream_t st) {
    pack_w2_kernel<<<dim3(H / 32, H / 32), dim3(32, 8), 0, st>>>(w2, (__nv_bfloat16 *)w, (__nv_bfloat16 *)wt, (__nv_bfloat16 *)img);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

extern "C" {

// Test hooks for the tensor-core building blocks (bf16 device buffers, row-major):
//   tmla_tc_linear: out[M,256] = tanh(A.W^T + bias) (epi 0)  |  (A.W^T) * (1 - aux^2) (epi 1);  W is [256 out][256 in]
//   tmla_tc_wgrad : G[256,256] (fp32) += X[rows,256]^T . Y[rows,256]
int tmla_tc_linear(int epi, const void *A, const void *W, const float *bias, const void *aux, void *out, int64_t M,
                   const int32_t *rows_dev, void *stream) {
    TMLA_REQUIRE(A && W && out && M > 0, "bad arguments");
    TMLA_REQUIRE((epi == EPI_BIAS_TANH && bias) || (epi == EPI_DTANH && aux), "epilogue operand missing");
    return tc_linear_launch(epi, A, W, bias, aux, out, M, rows_dev, (cudaStream_t)stream);
}
int tmla_tc_wgrad(const void *X, const void *Y, float *G, int64_t rows, void *stream) {
    TMLA_REQUIRE(X && Y && G && rows > 0, "bad arguments");
    return tc_wgrad_launch(X, Y, G, rows, (cudaStream_t)stream);
}
int tmla_tc_debug(int swap_lbo_sbo) {
    TMLA_CUDA(cudaMemcpyToSymbol(g_desc_swap, &swap_lbo_sbo, sizeof(int)));
    return TMLA_OK;
}
int tmla_f32_to_bf16(const float *src, void *dst, int64_t n, void *stream) {
    TMLA_REQUIRE(src && dst && n > 0, "bad arguments");
    f32_to_bf16_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, (cudaStream_t)stream>>>(src, (__nv_bfloat16 *)dst, n);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

}  // extern "C"
