// det_reduce.cu — the fixed-order sum behind deterministic mode (mlp_common.cuh: DetSeg).
//
// The reducing kernels of the update (fused tower kernel, split-K weight-gradient GEMMs, head / layer-1 backward, loss
// statistics) normally finish with float atomics, whose order follows the scheduler.  Their deterministic instantiations
// store one partial row per CTA instead; this kernel then sums, for every value, rows 0, 1, 2, ... of its segment.
// Block = 8 warps x 32 consecutive values: warp w sums rows w, w+8, w+16, ... in order, warp 0 adds the 8 warp sums in
// order.  The order depends on the row count only, never on timing, so two calls on the same inputs agree bit for bit.
#include "common.cuh"
#include "mlp_common.cuh"

struct DetSegs {
    DetSeg s[kDetMaxSegs];
};

__device__ __forceinline__ float det_rows_sum(const float *src, int64_t stride, int nrows, int64_t e, float (*sh)[32]) {
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    float s = 0.0f;
    for (int r = w; r < nrows; r += 8) s += src[(int64_t)r * stride + e];
    sh[w][l] = s;
    __syncthreads();
    float t = 0.0f;
    if (w == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) t += sh[q][l];
    }
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(256) det_reduce_kernel(const __grid_constant__ DetSegs segs) {
    __shared__ float sh[8][32];
    const DetSeg &g = segs.s[blockIdx.y];
    const int64_t e0 = (int64_t)blockIdx.x * 32;
    if (e0 >= g.len) return;                                   // (block-uniform)
    const int l = threadIdx.x & 31;
    const int64_t e = e0 + l;
    const bool ok = e < g.len;
    float t = det_rows_sum(g.src, g.stride, ok ? g.nrows : 0, e, sh);
    if (g.src2) t += det_rows_sum(g.src2, g.stride2, ok ? g.nrows2 : 0, e, sh);
    if (threadIdx.x < 32 && ok) g.dst[e] = g.assign ? t : g.dst[e] + t;
}

int det_reduce_launch(const DetSeg *segs, int nseg, cudaStream_t st) {
    TMLA_REQUIRE(nseg > 0 && nseg <= kDetMaxSegs, "bad segment count");
    DetSegs a;
    int64_t len = 0;
    for (int i = 0; i < nseg; ++i) {
        a.s[i] = segs[i];
        len = len > segs[i].len ? len : segs[i].len;
    }
    det_reduce_kernel<<<dim3((unsigned)ceil_div64(len, 32), (unsigned)nseg), 256, 0, st>>>(a);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
