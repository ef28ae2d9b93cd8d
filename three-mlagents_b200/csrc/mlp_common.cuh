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
