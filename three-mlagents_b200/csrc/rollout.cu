// rollout.cu — the PPO rollout as ONE call: tmla_rollout.
//
// Replaces the body of SB3's OnPolicyAlgorithm.collect_rollouts + RolloutBuffer.compute_returns_and_advantage, the loop the
// reference enters from backend/mlagents/training.py:166 (`model.learn`): for each of n_steps steps
//     policy forward -> sample action, log-prob -> VecEnv.step -> timeout bookkeeping -> buffer.add
// then predict_values(last_obs), the timeout bootstrap and the GAE scan.  Here the whole sequence
//     T x { tower forward (both towers, tcgen05) ; step_policy_kernel<Task> } ; last-value forward ; truncation-value forward ;
//     bootstrap_add ; gae_kernel ; step-counter increment
// is recorded ONCE into a CUDA graph per (handle, argument block) and replayed with a single cudaGraphLaunch per PPO
// iteration: no host round trip per step, no per-step launch pacing from the binding.  Every node is a kernel of this
// library; the Philox step index comes from a device-side counter so a replay draws fresh random numbers (same streams as
// the per-step calls: a replay is bit-identical to calling tmla_mlp_forward* + tmla_step_policy T times).
#include <stdlib.h>
#include <string.h>
#include <new>
#include "env_handle.cuh"

namespace {

struct RolloutPlan {
    tmla_rollout_args key;
    const void *ep_log, *ep_log_count;        // the handle's episode log is baked into the recorded step kernels too
    uint64_t seed;
    cudaGraphExec_t exec;
};

void plan_free(void *p) {
    RolloutPlan *plan = static_cast<RolloutPlan *>(p);
    if (plan->exec) cudaGraphExecDestroy(plan->exec);
    delete plan;
}

int forward(const tmla_rollout_args &a, const float *x, int64_t rows, const int32_t *rows_dev, float *logits, float *values, cudaStream_t st) {
    if (a.wpack)
        return tmla_mlp_forward_bf16(a.params, a.wpack, a.obs_dim, a.hidden, a.n_actions, x, nullptr, rows, rows_dev, logits, values, a.act_cache, st);
    return tmla_mlp_forward(a.params, a.obs_dim, a.hidden, a.n_actions, x, nullptr, rows, rows_dev, logits, values, (float *)a.act_cache, st);
}

// the launches of one rollout, in stream order (recorded under capture, or run directly when TMLA_ROLLOUT=launch)
int enqueue(tmla_env *h, const tmla_rollout_args &a, cudaStream_t st) {
    const int64_t n = h->n, D = a.obs_dim;
    const int T = a.n_steps;
    TMLA_CUDA(cudaMemsetAsync(a.trunc_count, 0, sizeof(int32_t), st));
    if (a.ep_stats) TMLA_CUDA(cudaMemsetAsync(a.ep_stats, 0, 4 * sizeof(float), st));
    for (int t = 0; t < T; ++t) {
        int rc = forward(a, a.obs + (int64_t)t * n * D, n, nullptr, a.logits, a.values + (int64_t)t * n, st);
        if (rc) return rc;
        rc = tmla_step_policy(h, a.logits, a.deterministic, t, a.obs + (int64_t)(t + 1) * n * D, a.actions + (int64_t)t * n,
                              a.log_probs + (int64_t)t * n, a.rewards + (int64_t)t * n, a.dones + (int64_t)t * n, a.trunc_count,
                              a.trunc_index, a.trunc_obs, a.trunc_capacity, a.ep_stats, a.step_counter, st);
        if (rc) return rc;
    }
    int rc = forward(a, a.obs + (int64_t)T * n * D, n, nullptr, nullptr, a.last_values, st);       // predict_values(last_obs)
    if (rc) return rc;
    // timeout bootstrap: rewards[idx] += gamma * V(terminal_obs) for the truncation records of this rollout
    rc = forward(a, a.trunc_obs, a.trunc_capacity, a.trunc_count, nullptr, a.trunc_values, st);
    if (rc) return rc;
    rc = tmla_bootstrap_add(a.rewards, a.trunc_count, a.trunc_index, a.trunc_values, a.gamma, a.trunc_capacity, st);
    if (rc) return rc;
    rc = tmla_gae(a.rewards, a.values, a.dones, a.last_values, a.gamma, a.gae_lambda, T, n, a.advantages, a.returns, st);
    if (rc) return rc;
    return tmla_counter_add(a.step_counter, (uint64_t)T, st);
}

}  // namespace

extern "C" {

int tmla_rollout(tmla_env *h, const tmla_rollout_args *args, void *stream) {
    TMLA_REQUIRE(h && args, "handle/args is NULL");
    const tmla_rollout_args &a = *args;
    TMLA_REQUIRE(a.params && a.obs && a.actions && a.log_probs && a.rewards && a.values && a.dones && a.last_values && a.advantages &&
                 a.returns && a.logits && a.step_counter, "NULL rollout buffer");
    TMLA_REQUIRE(a.trunc_count && a.trunc_index && a.trunc_obs && a.trunc_values && a.trunc_capacity > 0, "truncation list is incomplete");
    TMLA_REQUIRE(a.n_steps > 0 && a.obs_dim == tmla_task_obs_dim(h->task) && a.n_actions == tmla_task_num_actions(h->task),
                 "n_steps / obs_dim / n_actions do not match the handle's task");
    TMLA_REQUIRE(a.act_cache || (a.wpack ? a.obs_dim <= 6 : (a.hidden == 64 || a.hidden == 128)),
                 "act_cache may be NULL only on the fused-tower shapes (bf16, obs_dim <= 6) and for the fp32 widths 64 and 128");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    // the device-side step counter the graph's kernels read: (re)synchronised with the handle on every call (8 bytes)
    TMLA_CUDA(cudaMemcpyAsync(a.step_counter, &h->step_count, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    static const bool direct = [] { const char *e = getenv("TMLA_ROLLOUT"); return e && !strcmp(e, "launch"); }();
    if (direct) {                                          // debugging aid: the same launches without a graph
        const int rc = enqueue(h, a, st);
        if (rc) return rc;
        h->step_count += (uint64_t)a.n_steps;
        return TMLA_OK;
    }
    RolloutPlan *plan = static_cast<RolloutPlan *>(h->rollout_plan);
    if (!plan || memcmp(&plan->key, &a, sizeof(a)) != 0 || plan->ep_log != h->ep_log || plan->ep_log_count != h->ep_log_count ||
        plan->seed != h->seed) {
        if (plan) { plan_free(plan); h->rollout_plan = nullptr; }
        // recorded on a private stream (the caller's may be the legacy default stream, which cannot be captured); the
        // instantiated graph is then launched on the caller's stream
        cudaStream_t cap = nullptr;
        TMLA_CUDA(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        cudaError_t ec = cudaStreamBeginCapture(cap, cudaStreamCaptureModeRelaxed);
        int rc = TMLA_OK;
        if (ec == cudaSuccess) {
            rc = enqueue(h, a, cap);
            ec = cudaStreamEndCapture(cap, &graph);
        }
        cudaStreamDestroy(cap);
        if (rc || ec != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            if (!rc) tmla_set_error("tmla_rollout: stream capture failed: %s", cudaGetErrorString(ec));
            cudaGetLastError();
            return rc ? rc : TMLA_ECUDA;
        }
        plan = new (std::nothrow) RolloutPlan();
        if (!plan) { cudaGraphDestroy(graph); tmla_set_error("out of host memory"); return TMLA_ENOMEM; }
        memcpy(&plan->key, &a, sizeof(a));
        plan->ep_log = h->ep_log; plan->ep_log_count = h->ep_log_count; plan->seed = h->seed;
        const cudaError_t ei = cudaGraphInstantiate(&plan->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ei != cudaSuccess) {
            delete plan;
            tmla_set_error("tmla_rollout: cudaGraphInstantiate: %s", cudaGetErrorString(ei));
            return TMLA_ECUDA;
        }
        h->rollout_plan = plan;
        h->rollout_plan_free = plan_free;
    }
    mark_device_path(h, st);
    TMLA_CUDA(cudaGraphLaunch(plan->exec, st));
    h->step_count += (uint64_t)a.n_steps;
    return TMLA_OK;
}

}  // extern "C"
