/*
 * tmla.h — C ABI of libtmla.so, the B200-native (sm_100a) hot path of three-mlagents.
 *
 * The reference (lukehollis/three-mlagents) has no FFI: its hot path is pure Python —
 * `DummyVecEnv.step_wait` looping over `LegacySingleAgentGymAdapter.step`
 * (backend/mlagents/envs.py:125-152) over `Ball3DEnv/GridWorldEnv/PushEnv.step`
 * (backend/examples/ball3d.py:74-113, gridworld.py:67-95, push.py:62-125) and
 * `BasicMoveToGoalEnv.step` (envs.py:60-81), then SB3's RolloutBuffer / PPO.train
 * reached from backend/mlagents/training.py:150,166.  Every entry point below names the
 * reference (or SB3-2.9.0) routine it replaces.  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add to bind them.
 *
 * Conventions
 *   - Every function returns 0 on success or a negative TMLA_E* code; the message is
 *     available from tmla_last_error() (thread-local).  No exceptions cross the ABI.
 *   - Unless a name ends in `_host`, tensor pointers are DEVICE pointers owned by the
 *     caller; the library owns only the packed structure-of-arrays environment state
 *     inside a handle.  `stream` is a cudaStream_t passed as void*; calls enqueue on it
 *     and never synchronise (the `_host` variants synchronise before returning because
 *     they hand results back in host memory).
 *   - A handle is bound to one (task, device); handles are independent; a handle is
 *     not thread-safe.
 *   - There is no CPU fallback anywhere in this library.
 */
#ifndef TMLA_H
#define TMLA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TMLA_VERSION 100          /* major*100 + minor */

#define TMLA_OK            0
#define TMLA_EINVAL       -1      /* bad argument (unknown task, null pointer, n<=0 ...) */
#define TMLA_ECUDA        -2      /* a CUDA runtime call failed */
#define TMLA_ENOMEM       -3
#define TMLA_EACTION      -4      /* an out-of-range action was seen by a step kernel */

typedef enum { TMLA_BASIC = 0, TMLA_BALL3D = 1, TMLA_GRIDWORLD = 2, TMLA_PUSH = 3, TMLA_WALLJUMP = 4, TMLA_BRICKBREAK = 5, TMLA_BICYCLE = 6, TMLA_GLIDER = 7 } tmla_task;
#define TMLA_NUM_TASKS 8

typedef struct tmla_env tmla_env;     /* opaque handle: packed SoA state of n envs on one GPU */

/* Wire format of tmla_get_state / tmla_set_state: array-of-structs, one per env, in DEVICE
 * memory (state injection for parity tests; the resident layout is packed SoA, DESIGN.md). */
typedef struct { int32_t pos, steps; float ep_return; } tmla_basic_state;                                /* envs.py:46-47 */
typedef struct { double rot[2]; float pos[2]; float vel[2]; int32_t steps; float ep_return; int32_t episode, pad_; } tmla_ball3d_state; /* ball3d.py:49-58; episode = auto-reset stream index */
typedef struct { int32_t agent[2], green[2], red[2], goal_type, steps; float ep_return; } tmla_gridworld_state;  /* gridworld.py:46-51 */
typedef struct { int32_t agent[2], box[2], goal_x, steps; float ep_return; } tmla_push_state;                    /* push.py:42-49 */
typedef struct { int32_t agent_x, in_air, wall, steps; float ep_return; } tmla_walljump_state;                   /* walljump.py:39-45 (SURVEY 8(f) #3) */
typedef struct { double pos[2], vel[2], paddle; uint8_t bricks[40]; int32_t steps; float ep_return; } tmla_brickbreak_state; /* brick_break.py:39-46 */
typedef struct { double x, z, theta, phi, phi_dot, delta, goal[2], dist; int32_t steps; float ep_return; } tmla_bicycle_state; /* bicycle.py:22-36 */
typedef struct { double pos[3], vel[3], rot[3], ang_vel[3]; int32_t waypoint, steps; float ep_return; int32_t pad_; } tmla_glider_state; /* glider.py:41-52 */

int         tmla_version(void);
const char *tmla_last_error(void);

/* task metadata — replaces the space declarations in make_*_env (envs.py:38-44,169-199) */
int tmla_task_from_name(const char *name);            /* "basic"|"ball3d"|"gridworld"|"push"|"walljump"|"brickbreak"|"bicycle"|"glider" -> tmla_task or TMLA_EINVAL */
int tmla_task_obs_dim(int task);                      /* 21 / 6 / 4 / 4 / 4 / 45 / 7 / 16 */
int tmla_task_num_actions(int task);                  /* 3 / 5 / 5 / 5 / 4 / 3 */
int tmla_task_max_steps(int task);                    /* 50 / 200 / 100 / 120 / 150 / 2000 */
int tmla_task_state_size(int task);                   /* sizeof(tmla_<task>_state) */

/* make_vector_env (training.py:71-89): n_envs envs whose global ids are
 * [env_id_base, env_id_base+n_envs); all randomness is Philox4x32-10 keyed by `seed`
 * with the global env id as sub-sequence, so trajectories do not depend on sharding. */
int tmla_create(int task, int64_t n_envs, uint64_t seed, uint64_t env_id_base, int device, tmla_env **out);
int tmla_destroy(tmla_env *h);                        /* VecEnv.close (training.py:223) */
int tmla_seed(tmla_env *h, uint64_t seed);            /* VecEnv.seed */
int64_t  tmla_num_envs(const tmla_env *h);
uint64_t tmla_step_count(const tmla_env *h);          /* global step index (host copy) */

/* VecEnv.reset(): re-draw every env (adapter.reset, envs.py:110-123) and write obs[n,D]. */
int tmla_reset(tmla_env *h, float *obs, void *stream);

/* VecEnv.step() = DummyVecEnv.step_wait: one fused launch doing
 * transition + reward + terminated/truncated + Monitor accumulation + terminal-obs capture +
 * Philox auto-reset + observation write.
 *   actions      int32[n]
 *   obs          float[n,D]   observation AFTER auto-reset (what VecEnv.step returns)
 *   reward       float[n]
 *   done         uint8[n]     terminated|truncated
 *   truncated    uint8[n]     infos[i]["TimeLimit.truncated"]
 *   terminal_obs float[n,D]   written only where done (infos[i]["terminal_observation"])
 *   ep_return    float[n]     written only where done (Monitor "r")
 *   ep_length    int32[n]     written only where done (Monitor "l")
 * terminal_obs / ep_return / ep_length may be NULL. */
int tmla_step(tmla_env *h, const int32_t *actions, float *obs, float *reward, uint8_t *done,
              uint8_t *truncated, float *terminal_obs, float *ep_return, int32_t *ep_length, void *stream);

/* Same call with HOST buffers (the SB3 VecEnv contract is NumPy in / NumPy out): stages through
 * pinned memory owned by the handle, H2D actions -> kernel -> D2H results, synchronises.
 * *n_done receives the number of finished episodes (so callers only touch infos when >0). */
int tmla_step_host(tmla_env *h, const int32_t *actions, float *obs, float *reward, uint8_t *done,
                   uint8_t *truncated, float *terminal_obs, float *ep_return, int32_t *ep_length,
                   int64_t *n_done);
int tmla_reset_host(tmla_env *h, float *obs);
/* Zero-copy variant for language bindings: the handle owns one pinned host block; tmla_host_views hands
 * out the pointers into it (valid for the life of the handle; any may be NULL).  The caller writes
 * int32 actions into *actions, calls tmla_step_pinned, and reads the results in place: obs/reward/done/
 * truncated after every call, terminal_obs/ep_return/ep_length valid where done when *n_done > 0. */
int tmla_host_views(tmla_env *h, int32_t **actions, float **obs, float **reward, uint8_t **done,
                    uint8_t **truncated, float **terminal_obs, float **ep_return, int32_t **ep_length);
int tmla_step_pinned(tmla_env *h, int64_t *n_done);
/* The same episode-end payload as *n_done compact records in the pinned block, in no particular order:
 * {int32 env index, float ep_return, int32 ep_length, float terminal_obs[D], zero padding} = *floats_per_record 32-bit words
 * each (3 + D rounded up to a multiple of 4, so the kernel writes a record as 128-bit stores) — what a
 * binding should read instead of scanning `done` (Monitor / infos of the finished envs only). */
int tmla_host_records(tmla_env *h, const float **records, int32_t *floats_per_record);
/* Result blocks: pinned host memory a binding hands out to ITS caller, so that the GPU writes a step's results
 * straight into the arrays the caller receives (no copy out of a staging block).  How they get there is selected by the
 * environment variable TMLA_HOST_STEP, read once per process (all tmla_step_host / _pinned / _block calls):
 *   unset / "poll": the step kernel reads the actions from and stores the results to pinned memory itself (zero-copy over
 *                   PCIe), the last CTA publishes {n_done, bad_action, sequence} and the host polls the sequence word;
 *   "sync"        : the same stores, completion by cudaStreamSynchronize;
 *   "copy"        : H2D actions -> kernel -> ONE D2H of obs..flags + the head of the record area (copy engines).
 * Layout, as byte offsets from the block:
 * offsets[0..5] = obs f32[n,D], reward f32[n], done u8[n], truncated u8[n], flags i32[4] {n_done, bad_action, sequence, -},
 * records (stride as tmla_host_records reports it); *bytes = size of a block.  tmla_step_block is tmla_step_pinned with the
 * results (and the n_done compact records) landing in `block`; the actions still come from the pinned action view.
 * The reference's DummyVecEnv returns fresh copies each step (SB3 dummy_vec_env.py step_wait): a binding keeps a small
 * pool of blocks and reuses one only when its caller has dropped every array over it (vec_env.py does this by refcount). */
/* Actions of the next host step (tmla_step_pinned / tmla_step_block), range-checked and narrowed in one pass over the caller's
 * array into the pinned action stage as ONE BYTE per action: a quarter of the PCIe reads of int32, and an out-of-range action
 * returns TMLA_EACTION before anything is launched — the reference's ACTION_DELTAS[action] (examples/ball3d.py:76) raises
 * before any state change.  elem_bytes = 4 (int32) or 8 (int64, what SB3 passes to VecEnv.step).  A caller that writes
 * int32 actions straight into the tmla_host_views action view instead is checked by the kernel (after the step). */
int tmla_stage_actions(tmla_env *h, const void *actions, int elem_bytes);
int tmla_result_block_layout(tmla_env *h, int64_t offsets[6], int64_t *bytes);
int tmla_result_block_alloc(tmla_env *h, void **block);
int tmla_result_block_free(void *block);
int tmla_step_block(tmla_env *h, void *block, int64_t *n_done);
/* VecEnv.step_async / step_wait (SB3 vec_env/base_vec_env.py; what DummyVecEnv.step_wait does serially over
 * backend/mlagents/envs.py:123-152) on the CALLER'S action array.  For int64 actions above 16 384 envs _begin launches the step
 * kernel first and then, chunk by chunk (TMLA_HOST_CHUNKS; default 4 for int64, 1 = stage-then-launch for int32), range-checks +
 * narrows the actions and publishes a ready word in mapped pinned memory that the chunk's first CTA polls: the host's staging
 * pass runs behind the launch latency and the earlier chunks' PCIe traffic.  _end waits for the sequence word of the batch and
 * returns n_done / TMLA_EACTION like tmla_step_block.  An out-of-range action in ANY chunk makes _begin return TMLA_EACTION
 * with every env in its pre-step state (chunks not yet released leave untouched, chunks already stepped are rolled back from
 * shadow state planes) — the reference's ACTION_DELTAS[action] raises before any state change.  One step in flight per handle. */
int tmla_step_block_begin(tmla_env *h, const void *actions, int elem_bytes, void *block);
int tmla_step_block_end(tmla_env *h, void *block, int64_t *n_done);

/* state injection / extraction (parity tests): `aos` is n structs of the task's wire type. */
int tmla_get_state(tmla_env *h, void *aos, void *stream);
int tmla_set_state(tmla_env *h, const void *aos, void *stream);
/* out-of-range action flag, read back from the device (synchronises `stream`). */
int tmla_check_actions(tmla_env *h, void *stream);

/* Fused T-step random-policy rollout, ONE launch, state held in registers for all T steps
 * (DummyVecEnv loop with `action_space.sample()`-style uniform actions from the TAG_ACTION
 * Philox stream).  Buffers are [T,n,...] as SB3's RolloutBuffer lays them out:
 *   obs_buf float[T,n,D] observation the action was taken on;  act_buf int32[T,n];
 *   rew_buf float[T,n];  done_buf uint8[T,n].  Any of them may be NULL (not written). */
int tmla_rollout_random(tmla_env *h, int T, float *obs_buf, int32_t *act_buf, float *rew_buf,
                        uint8_t *done_buf, void *stream);

/* Policy-driven step of the PPO rollout (OnPolicyAlgorithm.collect_rollouts body):
 * sample a ~ Categorical(logits) with the TAG_SAMPLE Philox stream (or argmax when
 * deterministic!=0), log-prob, env step, auto-reset, rollout-row write.
 *   logits float[n,A] ; obs_next float[n,D] (row t+1 of the obs buffer) ; act/logp/rew/done rows of
 *   the [T,n] buffers ; truncation records (terminal obs + flat index) are appended to trunc_*;
 *   step_base: optional DEVICE uint64 added to the handle's step index (CUDA-graph replay). */
int tmla_step_policy(tmla_env *h, const float *logits, int deterministic, int32_t row_index,
                     float *obs_next, int32_t *act, float *logp, float *rew, uint8_t *done,
                     int32_t *trunc_count, int32_t *trunc_index, float *trunc_obs, int32_t trunc_capacity,
                     float *ep_stats /* [4]: sum return, sum length, episodes, (unused) */,
                     const uint64_t *step_base, void *stream);
/* The whole PPO rollout as ONE call — OnPolicyAlgorithm.collect_rollouts + RolloutBuffer.compute_returns_and_advantage of
 * SB3 2.9.0, the loop the reference enters from backend/mlagents/training.py:166 (SURVEY.md A.2/A.3; §8(b) `tmla_rollout`):
 *   for t in [0, n_steps): logits, values[t] = policy(obs[t]); a ~ Categorical(logits) (TAG_SAMPLE Philox stream);
 *                          obs[t+1], rewards[t], dones[t] = VecEnv.step(a) with auto-reset; timeouts recorded in trunc_*
 *   last_values = V(obs[n_steps]);  rewards[idx] += gamma * V(terminal_obs) for the timeouts;  GAE -> advantages, returns.
 * The launches (tower forward on tcgen05 + step_policy_kernel per step, value forwards, bootstrap, GAE scan) are recorded
 * once per (handle, argument block) into a CUDA graph and replayed with one cudaGraphLaunch per call: no host round trip
 * per step.  A call is bit-identical to n_steps x {tmla_mlp_forward[_bf16] + tmla_step_policy} + tmla_bootstrap_add +
 * tmla_gae issued one by one (environment variable TMLA_ROLLOUT=launch does exactly that, for debugging).
 * Every pointer is DEVICE memory owned by the caller; the struct has no padding (it is compared bytewise to reuse the graph).
 *   params/wpack/act_cache  as tmla_mlp_forward_bf16 (wpack NULL = fp32 CUDA-core path, act_cache then float); act_cache holds
 *                           4 x max(n, trunc_capacity) x hidden elements, NULL allowed where tmla_mlp_forward_bf16 allows it
 *                           and, with wpack NULL, for hidden 64 and 128
 *   obs [n_steps+1,n,D]     row 0 = current observations (input), rows 1.. written
 *   actions/log_probs/rewards/values/dones/advantages/returns [n_steps,n];  last_values [n];  logits [n,A] scratch
 *   trunc_count int32[1], trunc_index int32[cap], trunc_obs float[cap,D], trunc_values float[cap]: timeout records
 *   ep_stats float[4] (sum return, sum length, episodes, -) or NULL;  step_counter: device uint64 scratch */
typedef struct {
    const float *params; const void *wpack; void *act_cache;
    float *obs; int32_t *actions; float *log_probs; float *rewards; float *values; uint8_t *dones;
    float *last_values; float *advantages; float *returns; float *logits;
    int32_t *trunc_count; int32_t *trunc_index; float *trunc_obs; float *trunc_values;
    float *ep_stats; uint64_t *step_counter;
    double gamma, gae_lambda;
    int32_t obs_dim, hidden, n_actions, n_steps, deterministic, trunc_capacity;
} tmla_rollout_args;
int tmla_rollout(tmla_env *h, const tmla_rollout_args *args, void *stream);

/* Monitor (training.py:83: `Monitor(env, filename=...)` logs {r, l, t} per episode) for the policy-driven device path: while a
 * log is attached, every episode that ends inside tmla_step_policy / tmla_rollout appends {ep_return, float(ep_length)} at slot
 * atomicAdd(count); records float[capacity][2] and count int32 are DEVICE memory owned by the caller, who reads and re-zeroes
 * count between rollouts (slots >= capacity are counted, not written).  records = count = NULL detaches. */
int tmla_set_episode_log(tmla_env *h, float *records, int32_t capacity, int32_t *count);
/* advance the handle's host step counter after a graph replay of T tmla_step_policy launches,
 * and the matching device-side counter increment to put at the end of the captured graph */
int tmla_advance_steps(tmla_env *h, uint64_t n);
int tmla_counter_add(uint64_t *counter, uint64_t n, void *stream);
/* test hook: exhaustive check of the kernels' hand-rolled correctly-rounded x/3, x/5 and the short double
 * sin polynomial against the IEEE intrinsics; out3 = DEVICE uint64[3] {x/3 mismatches over [0,8),
 * k/5 mismatches over k in [-5,5], max ulp distance of sin over [-25deg, 25deg]} */
int tmla_selftest_arith(uint64_t *out3, void *stream);

/* rewards[idx] += gamma * values[i] for the truncation records (collect_rollouts timeout bootstrap) */
int tmla_bootstrap_add(float *rew_buf, const int32_t *trunc_count, const int32_t *trunc_index,
                       const float *trunc_values, double gamma, int32_t capacity, void *stream);

/* RolloutBuffer.compute_returns_and_advantage (SB3 2.9.0), float32, same operation order:
 * rewards/values float[T,n], dones uint8[T,n] (done after step t == episode_starts[t+1]),
 * last_values float[n]  ->  advantages, returns float[T,n].  gamma/gae_lambda are doubles because
 * NumPy multiplies the two Python floats in double before rounding to float32 (SURVEY.md A.3). */
int tmla_gae(const float *rewards, const float *values, const uint8_t *dones, const float *last_values,
             double gamma, double gae_lambda, int T, int64_t n, float *advantages, float *returns, void *stream);

/* RolloutBuffer.get: pseudo-random permutation of [0,total) (keyed Feistel + cycle walking), written
 * as SB3's flat sample index env*T+t converted to buffer offset t*n+env.  out int32[total]. */
int tmla_permutation(uint64_t seed, uint64_t epoch, int64_t total, int T, int64_t n, int32_t *out, void *stream);

/* ---- policy / value network: MlpPolicy with net_arch dict(pi=[H,H], vf=[H,H]), tanh ------------
 * Flat fp32 parameter vector in SB3's policy.parameters() order:
 *   pi.W1[H,D] pi.b1[H] pi.W2[H,H] pi.b2[H] vf.W1[H,D] vf.b1[H] vf.W2[H,H] vf.b2[H] Wa[A,H] ba[A] Wv[1,H] bv[1]
 * hidden H: 256, 64 or 128 for tmla_mlp_num_params / tmla_mlp_forward / tmla_mlp_backward(_scratch) (64 and 128 run the
 * float32 kernels of csrc/mlp_small.cu); any other width is TMLA_EINVAL.  The bf16 entry points take 256 only.
 */
int64_t tmla_mlp_num_params(int obs_dim, int hidden, int n_actions);

/* ActorCriticPolicy.forward / evaluate_actions / predict_values.
 *   x float[rows,D] gathered through `index` (int32[rows], may be NULL = identity);
 *   logits float[rows,A] (NULL: value tower only), values float[rows] (NULL: policy tower only);
 *   act_cache: float[4,rows,H] (pi.h1, pi.h2, vf.h1, vf.h2) kept for tmla_mlp_backward (workspace at H = 256; at H = 64 / 128
 *   NULL = inference, no activations kept);
 *   rows_dev: optional DEVICE int32 row count overriding `rows` as an upper bound (rows<=capacity). */
int tmla_mlp_forward(const float *params, int obs_dim, int hidden, int n_actions, const float *x,
                     const int32_t *index, int64_t rows, const int32_t *rows_dev, float *logits,
                     float *values, float *act_cache, void *stream);

/* backward of the above: dlogits float[rows,A], dvalues float[rows] -> grads (flat, same order as
 * params; OVERWRITTEN, not accumulated).  scratch: float[tmla_mlp_backward_scratch(...)] (H = 64 / 128: per-chunk partial
 * gradients, summed in a fixed order, so two calls on the same inputs give bit-identical gradients) */
int64_t tmla_mlp_backward_scratch(int obs_dim, int hidden, int n_actions, int64_t rows);
int tmla_mlp_backward(const float *params, int obs_dim, int hidden, int n_actions, const float *x,
                      const int32_t *index, int64_t rows, const float *act_cache, const float *dlogits,
                      const float *dvalues, float *grads, float *scratch, void *stream);

/* bf16 / tensor-core variant of the same network (csrc/mlp_tc.cu): identical semantics, the 256x256 hidden
 * layers run on tcgen05 with bf16 operands and fp32 accumulation, activations (act_cache, scratch) are bf16.
 * hidden must be 256 (other widths: TMLA_EINVAL with a message naming the float32 entry points).
 *   wpack: bf16[TMLA_WPACK_MATRICES][256][256] = {pi.W2, pi.W2^T, vf.W2, vf.W2^T, pi.W2 image, vf.W2 image} (image = the
 *   shared-memory operand layout the fused minibatch kernel loads with one bulk-TMA copy), refreshed by tmla_mlp_pack_bf16 after every
 *   optimizer step.  act_cache: bf16[4,rows,256] (forward: may be NULL when obs_dim <= 6 = inference only, the
 *   fused tower kernel then keeps no activations); scratch: bf16[2,rows,256]. */
#define TMLA_WPACK_MATRICES 6
int tmla_mlp_pack_bf16(const float *params, int obs_dim, int hidden, int n_actions, void *wpack, void *stream);
int tmla_mlp_forward_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *x,
                          const int32_t *index, int64_t rows, const int32_t *rows_dev, float *logits, float *values,
                          void *act_cache, void *stream);
int tmla_mlp_backward_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *x,
                           const int32_t *index, int64_t rows, const void *act_cache, const float *dlogits,
                           const float *dvalues, float *grads, void *scratch, void *stream);

/* PPO.train, one minibatch, loss head (SB3 2.9.0 ppo.py): advantage normalisation statistics,
 * then clipped surrogate + value MSE + entropy, forward and backward in one pass.
 *   stats_out float[8]: pg_loss, value_loss, entropy_loss, approx_kl, clip_fraction, loss, adv_mean, adv_std
 *   adv_sums double[3] device scratch (sum, sum of squares, count) — filled by tmla_adv_stats;
 *   with world_size>1 the caller all-reduces adv_sums between the two calls (global-minibatch
 *   normalisation) and passes the global row count to tmla_ppo_loss. */
int tmla_adv_stats(const float *advantages, const int32_t *index, int64_t rows, double *adv_sums, void *stream);
/* the same statistics for every minibatch of an epoch in one launch: minibatch m covers index[m*mb_rows, min(total,
 * (m+1)*mb_rows)); adv_sums double[ceil(total/mb_rows)][3].  One all-reduce per epoch then replaces one per minibatch. */
int tmla_adv_stats_batched(const float *advantages, const int32_t *index, int64_t total, int64_t mb_rows, double *adv_sums,
                           void *stream);
int tmla_ppo_loss(const float *logits, const float *values, const int32_t *actions, const float *advantages,
                  const float *old_logp, const float *returns, const int32_t *index, int64_t rows,
                  int64_t global_rows, int n_actions, const double *adv_sums, int normalize_advantage,
                  float clip_range, float ent_coef, float vf_coef, float *dlogits, float *dvalues,
                  float *stats_out, void *stream);
/* A2C.train's loss head (SB3 2.9.0 a2c.py), the same pass for the whole rollout as ONE batch:
 *   policy_loss = -(adv * log_prob).mean(), value_loss = mse(returns, values), entropy_loss = -mean(entropy),
 *   loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss; advantages normalised (as tmla_ppo_loss) only when
 *   normalize_advantage != 0 (A2C's default is off).  Arguments as tmla_ppo_loss without old_logp and clip_range;
 *   stats_out float[8] in tmla_ppo_loss's layout with approx_kl and clip_fraction left 0. */
int tmla_a2c_loss(const float *logits, const float *values, const int32_t *actions, const float *advantages, const float *returns,
                  const int32_t *index, int64_t rows, int64_t global_rows, int n_actions, const double *adv_sums,
                  int normalize_advantage, float ent_coef, float vf_coef, float *dlogits, float *dvalues, float *stats_out,
                  void *stream);

/* clip_grad_norm_(max_norm) + Adam.step fused (after the gradient all-reduce).
 *   grad_scale multiplies the gradient first; state m,v float[np]; step is the 1-based Adam step;
 *   norm_out float[TMLA_ADAM_SCRATCH]: [0] receives the pre-clip global norm, [1, 129) is scratch for the
 *   fixed-order (bit-reproducible across data-parallel replicas) reduction of the squared norm, [129, 131) are the two words of
 *   the one-launch optimizer step's grid barrier — the caller zeroes the buffer ONCE when it allocates it. */
#define TMLA_ADAM_SCRATCH 132
int tmla_adam_clip(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale,
                   float max_grad_norm, float lr, float beta1, float beta2, float eps, int64_t step,
                   float *norm_out, void *stream);
/* Same step; zero_grads != 0 also clears `grads` once consumed, so that the next tmla_ppo_minibatch_bf16 call can run with
 * TMLA_MB_GRADS_ZEROED (no memset launch between minibatches). */
int tmla_adam_clip_zero(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale,
                        float max_grad_norm, float lr, float beta1, float beta2, float eps, int64_t step,
                        float *norm_out, int zero_grads, void *stream);
/* ... and, with wpack != NULL (the buffer of tmla_mlp_pack_bf16), also refreshes the bf16 OPERAND IMAGES of the two hidden-layer
 * matrices — all the fused minibatch kernel reads — so no repack launch is needed between minibatches; the row-major bf16
 * copies the rollout's forward uses are NOT refreshed: call tmla_mlp_pack_bf16 once when the update loop ends. */
int tmla_adam_clip_fused(float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale,
                         float max_grad_norm, float lr, float beta1, float beta2, float eps, int64_t step,
                         float *norm_out, int zero_grads, void *wpack, int obs_dim, int hidden, int n_actions, void *stream);

/* ---- the one collective of the path, fused with the optimizer step (csrc/comm.cu) -------------------------------------
 * Data-parallel PPO (one process per GPU, DESIGN.md §7) sums the flat gradient over the ranks once per minibatch.  The reference
 * is single-process (no collective anywhere in backend/); this replaces the `torch.distributed.all_reduce(grads)` +
 * tmla_adam_clip_fused pair with a one-shot all-reduce over NVLink peer memory inside the clip + Adam launches: every rank
 * publishes its gradient in an IPC-exported slot, waits on flags the peers store into ITS memory, reads all slots directly and
 * sums them in rank order (replicas stay bit-identical), producing clip_grad_norm_'s partial sums in the same pass.
 *   tmla_comm_create : allocates this rank's exchange memory on `device` (num_floats >= num_params); handle_out receives the
 *                      64-byte CUDA IPC handle the caller gathers from all ranks (any transport: torch.distributed, MPI, files)
 *   tmla_comm_connect: all_handles = world x 64 bytes, rank-major; maps every peer's exchange memory
 *   tmla_adam_clip_allreduce: arguments as tmla_adam_clip_fused; `step` doubles as the exchange sequence number, so all ranks
 *                      must call it the same number of times with the same step.  Waits are bounded (TMLA_COMM_TIMEOUT_MS, default
 *                      5000): a rank that never shows up sets an error word instead of hanging the GPU — tmla_comm_check
 *                      (synchronises `stream`) turns it into TMLA_ECUDA. */
typedef struct tmla_comm tmla_comm;
int tmla_comm_create(int rank, int world, int device, int64_t num_floats, tmla_comm **out, void *handle_out);
int tmla_comm_connect(tmla_comm *c, const void *all_handles);
int tmla_comm_destroy(tmla_comm *c);
int tmla_comm_check(tmla_comm *c, void *stream);
int tmla_adam_clip_allreduce(tmla_comm *c, float *params, float *grads, float *m, float *v, int64_t num_params, float grad_scale,
                             float max_grad_norm, float lr, float beta1, float beta2, float eps, int64_t step, float *norm_out,
                             int zero_grads, void *wpack, int obs_dim, int hidden, int n_actions, void *stream);

/* clip_grad_norm_(max_norm) + torch.optim.RMSprop.step (A2C's optimizer: alpha 0.99, eps 1e-5, not centred, no momentum, no
 * weight decay), in ONE launch (csrc/comm.cu):  square_avg = alpha * square_avg + (1 - alpha) * g^2;  p -= lr * g / (sqrt(square_avg) + eps)
 * (eps after the square root: torch's rule).  alpha is a double because 1 - alpha is formed from it before rounding to float,
 * as torch does with the Python float it is given (from a float 0.99 the factor would be 8 ulp off).  Arguments as tmla_adam_clip_fused with the one state vector sq_avg float[np]
 * instead of m, v; the allreduce form as tmla_adam_clip_allreduce (`step` = exchange sequence number).  There is no two-launch
 * form: a shape the one launch does not cover (more than 262 144 parameters, buffers not 16-byte aligned, a world other than
 * 1, 2, 4, 8) returns TMLA_EINVAL. */
int tmla_rmsprop_clip_fused(float *params, float *grads, float *sq_avg, int64_t num_params, float grad_scale, float max_grad_norm, float lr,
                            double alpha, float eps, float *norm_out, int zero_grads, void *wpack, int obs_dim, int hidden, int n_actions,
                            void *stream);
int tmla_rmsprop_clip_allreduce(tmla_comm *c, float *params, float *grads, float *sq_avg, int64_t num_params, float grad_scale,
                                float max_grad_norm, float lr, double alpha, float eps, int64_t step, float *norm_out, int zero_grads,
                                void *wpack, int obs_dim, int hidden, int n_actions, void *stream);

/* ---- tensor-core building blocks (csrc/mlp_tc.cu: tcgen05.mma, TMEM accumulators), bf16 row-major device
 * buffers.  Used by the bf16 MLP path; exported so the parity tests can exercise them in isolation.
 *   tmla_tc_linear: out[M,256] = tanh(A . W^T + bias)            (epi 0; layer-2 forward of a tower)
 *                   out[M,256] = (A . W^T) * (1 - aux^2)          (epi 1; dgrad through tanh, W = W2^T)
 *                   A, aux, out bf16 [M,256]; W bf16 [256 out][256 in]; bias fp32[256]
 *   tmla_tc_wgrad : G[256,256] (fp32, accumulated) += X[rows,256]^T . Y[rows,256]
 *   tmla_f32_to_bf16: elementwise conversion;  tmla_tc_debug: descriptor-field experiment switch (tests only) */
int tmla_tc_linear(int epi, const void *A, const void *W, const float *bias, const void *aux, void *out, int64_t M,
                   const int32_t *rows_dev, void *stream);
int tmla_tc_wgrad(const void *X, const void *Y, float *G, int64_t rows, void *stream);
int tmla_f32_to_bf16(const float *src, void *dst, int64_t n, void *stream);
int tmla_tc_debug(int swap_lbo_sbo);

/* ---- PPO.train, one minibatch, fully fused (csrc/mlp_train.cu) ------------------------------------------------
 * Replaces, per minibatch of SB3's PPO.train (reached from backend/mlagents/training.py:166; hyper-parameters
 * training.py:379-389; policy built at training.py:150 with net_arch training.py:363-365), the sequence
 *     evaluate_actions -> advantage normalisation -> clipped surrogate + value MSE + entropy -> loss.backward()
 * i.e. tmla_mlp_forward_bf16 + tmla_ppo_loss + tmla_mlp_backward_bf16 with identical semantics, but as one
 * persistent kernel per tower (forward, loss and backward on chip; tcgen05 for the 256x256 layers) plus one
 * split-K weight-gradient GEMM per tower.  Arguments as in those three calls:
 *   obs float[total,D], index int32[rows] (NULL = identity) selects the minibatch rows of obs AND of the
 *   [T*N] buffers actions/advantages/old_logp/returns;  adv_sums from tmla_adv_stats (all-reduced by the caller
 *   when world_size>1), global_rows = rows summed over ranks;
 *   grads float[num_params] OVERWRITTEN;  scratch bf16[tmla_ppo_minibatch_scratch(hidden, rows)] (tile images);
 *   stats_out float[8] as tmla_ppo_loss;  logits_out float[rows,A] / values_out float[rows]: optional (NULL);
 *   flags: TMLA_MB_GRADS_ZEROED — the caller guarantees grads is all zeros (tmla_adam_clip_zero left it so): no memset;
 *          TMLA_MB_ACCUMULATE_STATS — stats_out is added to instead of overwritten (a running sum over minibatches);
 *          TMLA_MB_DETERMINISTIC — bit-reproducible sums (see "deterministic mode" below; needs the larger scratch).
 * tmla_ppo_minibatch_supported: 1 when the fused path covers (obs_dim, hidden, n_actions) — ball3d, gridworld,
 * push, walljump, bicycle at hidden 256; callers use the three-call sequence otherwise (basic: obs_dim 21, 3 actions; every
 * shape at hidden 64 / 128, where it returns 0). */
#define TMLA_MB_GRADS_ZEROED 1
#define TMLA_MB_ACCUMULATE_STATS 2
int tmla_ppo_minibatch_supported(int obs_dim, int hidden, int n_actions);
int64_t tmla_ppo_minibatch_scratch(int hidden, int64_t rows);
int tmla_ppo_minibatch_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *obs,
                            const int32_t *index, int64_t rows, int64_t global_rows, const int32_t *actions,
                            const float *advantages, const float *old_logp, const float *returns, const double *adv_sums,
                            int normalize_advantage, float clip_range, float ent_coef, float vf_coef, float *grads,
                            void *scratch, float *stats_out, float *logits_out, float *values_out, int flags, void *stream);
/* A2C.train (SB3 2.9.0 a2c.py: rollout_buffer.get(batch_size=None), one gradient step per rollout) fused the same way: the
 * policy tower runs tmla_a2c_loss's loss instead of the clipped surrogate and reads no old log-probabilities.  Arguments as
 * tmla_ppo_minibatch_bf16 without old_logp and clip_range; index is normally NULL (the whole rollout, row order irrelevant);
 * the same shapes as tmla_ppo_minibatch_supported; stats_out as tmla_a2c_loss. */
int tmla_a2c_batch_bf16(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *obs,
                        const int32_t *index, int64_t rows, int64_t global_rows, const int32_t *actions, const float *advantages,
                        const float *returns, const double *adv_sums, int normalize_advantage, float ent_coef, float vf_coef,
                        float *grads, void *scratch, float *stats_out, float *logits_out, float *values_out, int flags, void *stream);

/* test hooks of csrc/mlp_train.cu:
 *   tmla_tc_wgrad_tiled: G[256,256] (fp32, accumulated) += X^T . Y where X and Y are given as TILE IMAGES — per 128
 *                     rows one 64 KB block in the shared-memory operand layout, 16-byte chunk (r, cb) of a tile at
 *                     byte (r/8)*4096 + cb*128 + (r%8)*16 — exactly what the fused training kernel writes with one
 *                     bulk-TMA store per tile; operands are read through MN-major UMMA descriptors;
 *   tmla_tc_probe   : one-CTA descriptor check, A bf16[128,256], B bf16[256,256]:
 *                     mode 0 out[128,256] = A.B^T | mode 1 out[128,256] = A.B | mode 2 out[256,256] = A^T.B[0:128] */
int tmla_tc_wgrad_tiled(const void *Xt, const void *Yt, float *G, int64_t rows_padded, void *stream);
int tmla_tc_probe(const void *A, const void *B, float *out, int mode, void *stream);
/* measurement hook: do tcgen05.ld reads of TMEM columns [256,512) overlap tcgen05.mma (M128 N=n K16) already queued on columns
 * [0,n)?  out8 = DEVICE uint64[8] cycle counts {MMAs alone, loads alone, MMAs with loads running, loads under queued MMAs,
 * cycles the issuing lane spent inside the tcgen05.mma instructions, -, -, -}  (profiles/tc_overlap.py) */
int tmla_tc_overlap_probe(uint64_t *out8, int n, int n_mma, int n_ld, void *stream);

/* ---- deterministic mode ---------------------------------------------------------------------------------------------------
 * The default update kernels finish their sums over rows with float atomics, so their last bits depend on scheduling.  The
 * forms below compute the same quantities, but every CTA stores its partial sum in a scratch row of its own and one more launch
 * adds the rows in CTA order: two calls on the same inputs (same build, same GPU model) give bit-identical results.
 *   TMLA_MB_DETERMINISTIC (flags of tmla_ppo_minibatch_bf16 / tmla_a2c_batch_bf16): scratch then holds the
 *       tmla_ppo_minibatch_scratch(hidden, rows) bf16 tile-image elements followed by tmla_det_scratch_bytes(...) bytes of partials;
 *   tmla_mlp_backward_bf16_det, tmla_ppo_loss_det, tmla_a2c_loss_det: as their default forms plus `partials`, a device buffer of
 *       tmla_det_scratch_bytes(obs_dim, hidden, n_actions, rows) bytes (one size serves every call of up to `rows` rows: it never
 *       decreases as rows grow);
 *   tmla_adv_stats_batched_det: as tmla_adv_stats_batched plus `partials` of tmla_adv_stats_det_scratch_bytes(total, mb_rows)
 *       bytes (a single batch: mb_rows = total).
 * Not covered: the float32 256-wide path (tmla_mlp_backward's split-K GEMM) and the gradient exchange between ranks. */
#define TMLA_MB_DETERMINISTIC 4
int64_t tmla_det_scratch_bytes(int obs_dim, int hidden, int n_actions, int64_t rows);
int64_t tmla_adv_stats_det_scratch_bytes(int64_t total, int64_t mb_rows);
int tmla_mlp_backward_bf16_det(const float *params, const void *wpack, int obs_dim, int hidden, int n_actions, const float *x,
                               const int32_t *index, int64_t rows, const void *act_cache, const float *dlogits,
                               const float *dvalues, float *grads, void *scratch, void *partials, void *stream);
int tmla_adv_stats_batched_det(const float *advantages, const int32_t *index, int64_t total, int64_t mb_rows, double *adv_sums,
                               void *partials, void *stream);
int tmla_ppo_loss_det(const float *logits, const float *values, const int32_t *actions, const float *advantages,
                      const float *old_logp, const float *returns, const int32_t *index, int64_t rows, int64_t global_rows,
                      int n_actions, const double *adv_sums, int normalize_advantage, float clip_range, float ent_coef,
                      float vf_coef, float *dlogits, float *dvalues, float *stats_out, void *partials, void *stream);
int tmla_a2c_loss_det(const float *logits, const float *values, const int32_t *actions, const float *advantages, const float *returns,
                      const int32_t *index, int64_t rows, int64_t global_rows, int n_actions, const double *adv_sums,
                      int normalize_advantage, float ent_coef, float vf_coef, float *dlogits, float *dvalues, float *stats_out,
                      void *partials, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TMLA_H */
