// mlp_common.cuh — offsets of the flat fp32 parameter vector (include/tmla.h: policy.parameters() order)
#pragma once
#include <stdint.h>

struct MlpOffsets {
    int64_t w1[2], b1[2], w2[2], b2[2], wh[2], bh[2], total;
    int nout[2];
};
static inline MlpOffsets mlp_offsets(int D, int A, int64_t H = 256) {      // H: hidden width (256, or 64 / 128: mlp_small.cu)
    MlpOffsets o;
    int64_t p = 0;
    for (int t = 0; t < 2; ++t) {
        o.w1[t] = p; p += H * D;
        o.b1[t] = p; p += H;
        o.w2[t] = p; p += H * H;
        o.b2[t] = p; p += H;
    }
    o.wh[0] = p; p += (int64_t)A * H;
    o.bh[0] = p; p += A;
    o.wh[1] = p; p += H;
    o.bh[1] = p; p += 1;
    o.total = p;
    o.nout[0] = A; o.nout[1] = 1;
    return o;
}


// ---- deterministic mode (TMLA_MB_DETERMINISTIC and the *_det entry points): instead of a float atomic, CTA b of a reducing
// kernel stores its partial in row b of a partial buffer (rows of a compile-time stride), and det_reduce_launch sums the rows
// of every segment in row order (det_reduce.cu).  One segment = `len` consecutive values of each of `nrows` rows.
struct DetSeg {
    const float *src;             // row 0 of the partials
    int64_t stride;               // floats between rows
    int nrows, len;
    float *dst;                   // dst[i] += sum of rows (or = with `assign`)
    const float *src2;            // optional second partial set summed after the first (two towers' statistics), else NULL
    int64_t stride2;
    int nrows2, assign;
};
static constexpr int kDetMaxSegs = 12;
int det_reduce_launch(const DetSeg *segs, int nseg, cudaStream_t st);
// partial row of one CTA of the fused tower kernel (mlp_train.cu): W1 | b1 | b2 | Wh | bh | statistics (8)
__host__ __device__ constexpr int64_t det_tower_row(int D, int NOUT, int H = 256) { return (int64_t)H * D + 2 * H + (int64_t)NOUT * H + NOUT + 8; }
// squared-norm partials of clip_grad_norm_: one per CTA of the norm pass, summed in a fixed order by every CTA of the Adam kernel
#define TMLA_NORM_BLOCKS 128
// ppo_kernels.cu: clip + Adam launch shared with the fused all-reduce (comm.cu)
int adam_clip_launch(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                     float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, int zero_grads,
                     void *wpack, int obs_dim, int hidden, int n_actions, void *stream, bool partials_ready);
// comm.cu: the whole optimizer step (optional gradient exchange + clip + Adam) as one cooperative launch; TMLA_EINVAL = shape
// does not fit / disabled, callers fall back to the two-launch path
struct tmla_comm;
int opt_step_launch(tmla_comm *c, float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale, float max_grad_norm,
                    float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out, int zero_grads, void *wpack, int obs_dim,
                    int hidden, int n_actions, void *stream);
