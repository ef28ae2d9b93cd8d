// env_kernels.cu — batched environment stepping for basic / ball3d / gridworld / push / walljump / brickbreak / bicycle / glider (sm_100a).
//
// Replaces SB3 `DummyVecEnv.step_wait` (a serial Python loop over envs) + `Monitor` + the reference's
// `LegacySingleAgentGymAdapter.step/reset` (backend/mlagents/envs.py:110-152) and the task dynamics
// (envs.cuh).  One thread per environment; state lives in packed structure-of-arrays planes in HBM
// (128-bit loads/stores for ball3d, one 64-bit word per env for the integer tasks) and is kept in
// registers for all T steps by the fused rollout kernel.  Observation rows are staged through shared
// memory and leave the SM as coalesced 128-bit stores (ball3d's fused rollout: straight from each lane).
//
// These kernels are HBM-bound integer/byte/float32 work: no tensor cores, no GEMM reshaping.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <type_traits>
#if defined(__x86_64__)
#include <immintrin.h>
#endif
#include "envs.cuh"
#include "env_handle.cuh"

// the host path runs on own_stream: make it wait for whatever the device path enqueued on the caller's stream
static int order_after_device_path(tmla_env *h) {
    if (!h->dev_dirty) return TMLA_OK;
    h->dev_dirty = false;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(h->dev_stream, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone ||
        cudaEventRecord(h->dev_evt, h->dev_stream) != cudaSuccess) {
        cudaGetLastError();                               // stale / capturing stream: fall back to a device-wide wait
        TMLA_CUDA(cudaDeviceSynchronize());
        return TMLA_OK;
    }
    TMLA_CUDA(cudaStreamWaitEvent(h->own_stream, h->dev_evt, 0));
    return TMLA_OK;
}

struct EnvPtrs { void *buf[4]; };

static constexpr int kBlock = 128;

// ------------------------------------------------------------------------- cooperative obs store
// Threads of a block have written BLOCK*D floats (row-major [env][D]) to shared memory; write the
// valid prefix to `dst` as 128-bit stores when the destination is 16-byte aligned.
template <int D, int BLOCK, bool STREAMING>
__device__ __forceinline__ void block_store_obs(const float *s_obs, float *dst, int valid_envs) {
    const int total = valid_envs * D;
    if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        const int nvec = total >> 2;
        const float4 *s4 = reinterpret_cast<const float4 *>(s_obs);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        for (int v = threadIdx.x; v < nvec; v += BLOCK) {
            if (STREAMING) st_stream_f4(d4 + v, s4[v]);
            else d4[v] = s4[v];
        }
        for (int e = (nvec << 2) + threadIdx.x; e < total; e += BLOCK) dst[e] = s_obs[e];
    } else {
        for (int e = threadIdx.x; e < total; e += BLOCK) dst[e] = s_obs[e];
    }
}

template <int D>
__device__ __forceinline__ void thread_store_obs(const float *o, float *dst) {   // rare paths (terminal obs)
#pragma unroll
    for (int j = 0; j < D; ++j) dst[j] = o[j];
}

// ---------------------------------------------------------------------------------- reset / state
template <class Task>
__global__ void __launch_bounds__(kBlock) reset_kernel(EnvPtrs p, int64_t n, uint64_t seed, uint64_t env_base,
                                                       uint64_t k, uint32_t tag, float *obs) {
    __shared__ __align__(16) float s_obs[kBlock * Task::D];
    const int64_t i0 = (int64_t)blockIdx.x * kBlock, i = i0 + threadIdx.x;
    if (i < n) {
        typename Task::State s;
        Task::reset(s, seed, env_base + (uint64_t)i, k, tag);
        Task::store(p.buf, i, s);
        float o[Task::D];
        Task::observe(s, o);
#pragma unroll
        for (int j = 0; j < Task::D; ++j) s_obs[threadIdx.x * Task::D + j] = o[j];
    }
    __syncthreads();
    if (obs) block_store_obs<Task::D, kBlock, false>(s_obs, obs + i0 * Task::D, (int)min((int64_t)kBlock, n - i0));
}

template <class Task>
__global__ void get_state_kernel(EnvPtrs p, int64_t n, typename Task::Wire *aos) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) aos[i] = Task::to_wire(Task::load(p.buf, i));
}
template <class Task>
__global__ void set_state_kernel(EnvPtrs p, int64_t n, const typename Task::Wire *aos) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) Task::store(p.buf, i, Task::from_wire(aos[i]));
}

// ------------------------------------------------------------------------------------ VecEnv.step
template <class Task>
__global__ void __launch_bounds__(kBlock)
step_kernel(EnvPtrs p, int64_t n, uint64_t seed, uint64_t env_base, uint64_t step_index,
            const int32_t *__restrict__ actions, float *__restrict__ obs, float *__restrict__ reward,
            uint8_t *__restrict__ done, uint8_t *__restrict__ truncated, float *__restrict__ terminal_obs,
            float *__restrict__ ep_return, int32_t *__restrict__ ep_length, int32_t *n_done, int *err_flag,
            float *__restrict__ compact, int32_t *__restrict__ host_flags, int host_seq, int act_u8,
            const int32_t *ready, int32_t *dev_ready, int chunk_ctas, EnvPtrs shadow) {
    // ready != NULL (chunked host step, tmla_step_block_begin): the kernel is launched BEFORE the host has staged the actions;
    // the CTAs of chunk c = blockIdx.x / chunk_ctas wait until the host publishes ready[c] == host_seq in mapped pinned memory
    // (its range check + narrowing of that chunk is done; the chunk's first CTA polls it and republishes it in dev_ready[c])
    // and leave without touching anything on ready[c] == ~host_seq (a chunk was rejected) or after a bounded wait.  shadow.buf[0] != NULL: the state every env had BEFORE this step is kept in
    // the shadow planes, so that the chunks already stepped can be rolled back.
    // compact != NULL (host-facing step): finished envs append one record {env index, ep_return, ep_length, terminal_obs[D]}
    // at slot atomicAdd(n_done): the host then fetches n_done records instead of three dense [n] arrays.
    // host_flags != NULL (zero-copy host step): the last CTA to finish publishes {n_done, bad_action, host_seq} to mapped host
    // memory and re-arms the device counters n_done[0..2] (count, bad action, ticket): the step needs no memset and no flag
    // copy, and the host can poll host_flags[2] for host_seq instead of synchronising the stream (every CTA fences its
    // result stores at system scope before taking its ticket, so the sequence word is the last thing to become visible).
    constexpr int D = Task::D;
    __shared__ __align__(16) float s_obs[kBlock * D];
    __shared__ __align__(16) float s_rew[kBlock];
    __shared__ __align__(16) uint8_t s_flag[2 * kBlock];          // done[kBlock] | truncated[kBlock]
    const int64_t i0 = (int64_t)blockIdx.x * kBlock, i = i0 + threadIdx.x;
    if (ready) {
        // ONE CTA per chunk polls the host word over PCIe and republishes it in device memory for the others (512 CTAs polling
        // pinned memory directly saturate the non-posted PCIe reads: 400-540 us per step instead of 80)
        __shared__ int s_go;
        if (threadIdx.x == 0) {
            const int c = blockIdx.x / chunk_ctas;
            const bool leader = blockIdx.x == (unsigned)(c * chunk_ctas);
            const volatile int32_t *f = leader ? ready + c : dev_ready + c;
            unsigned long long t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            int v;
            while ((v = *f) != host_seq && v != ~host_seq) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > 2000000000ull) { v = ~host_seq; break; }      // 2 s: the host never finished staging
                if (leader) __nanosleep(100);
            }
            if (leader) { __threadfence_system(); *(volatile int32_t *)(dev_ready + c) = v; }
            __threadfence_system();                                          // the staged actions are read after the flag
            s_go = v == host_seq;
        }
        __syncthreads();
        if (!s_go) return;
    }
    // full block with 16-byte aligned rows: reward / done / truncated leave as 128-bit stores too (40 per CTA instead of 384
    // scalar ones — they may travel over PCIe to a pinned result block, where a 1-byte store per lane is a 32-byte write)
    const bool wide = (n - i0 >= kBlock) && (((reinterpret_cast<uintptr_t>(reward + i0) | reinterpret_cast<uintptr_t>(done + i0) |
                                               reinterpret_cast<uintptr_t>(truncated + i0)) & 15u) == 0);
    if (i < n) {
        const typename Task::Consts cst = Task::load_consts();
        typename Task::State s = Task::load(p.buf, i);
        if (shadow.buf[0]) Task::store(shadow.buf, i, s);
        int a = act_u8 ? (int)reinterpret_cast<const uint8_t *>(actions)[i] : actions[i];   // host step: one byte per action on the wire
        if ((unsigned)a >= (unsigned)Task::A) { *err_flag = 1; a = min(max(a, 0), Task::A - 1); }
        float r; bool term, trunc;
        Task::step(cst, s, a, r, term, trunc);
        s.ep_ret = __fadd_rn(s.ep_ret, r);                       // Monitor: episode return
        const bool d = term || trunc;
        if (wide) {
            s_rew[threadIdx.x] = r;
            s_flag[threadIdx.x] = d ? 1 : 0;
            s_flag[kBlock + threadIdx.x] = (trunc && !term) ? 1 : 0;
        } else {
            reward[i] = r;
            done[i] = d ? 1 : 0;
            truncated[i] = (trunc && !term) ? 1 : 0;             // infos["TimeLimit.truncated"]
        }
        float o[D];
        Task::observe(s, o);
        if (d) {                                                 // DummyVecEnv: keep terminal obs, auto-reset
            if (terminal_obs) thread_store_obs<D>(o, terminal_obs + i * D);
            if (ep_return) ep_return[i] = s.ep_ret;
            if (ep_length) ep_length[i] = s.steps;
            int slot = 0;
            if (n_done) slot = atomicAdd(n_done, 1);
            if (compact) {
                // records are padded to a multiple of 4 words and written as 128-bit stores (they may go over PCIe)
                constexpr int RW = (3 + D + 3) & ~3;
                float rec[RW];
                rec[0] = __int_as_float((int)i); rec[1] = s.ep_ret; rec[2] = __int_as_float(s.steps);
#pragma unroll
                for (int j = 0; j < D; ++j) rec[3 + j] = o[j];
#pragma unroll
                for (int j = 3 + D; j < RW; ++j) rec[j] = 0.0f;
                float4 *dst = reinterpret_cast<float4 *>(compact + (int64_t)slot * RW);
#pragma unroll
                for (int q = 0; q < RW / 4; ++q) dst[q] = make_float4(rec[4 * q], rec[4 * q + 1], rec[4 * q + 2], rec[4 * q + 3]);
            }
            Task::reset(s, seed, env_base + (uint64_t)i, step_index + 1, TMLA_TAG_RESET);
            Task::observe(s, o);
        }
        Task::store(p.buf, i, s);
#pragma unroll
        for (int j = 0; j < D; ++j) s_obs[threadIdx.x * D + j] = o[j];
    }
    __syncthreads();
    block_store_obs<D, kBlock, false>(s_obs, obs + i0 * D, (int)min((int64_t)kBlock, n - i0));
    if (wide) {
        const int t = threadIdx.x;
        if (t < kBlock / 4) reinterpret_cast<float4 *>(reward + i0)[t] = reinterpret_cast<const float4 *>(s_rew)[t];
        else if (t < kBlock / 4 + kBlock / 16) reinterpret_cast<uint4 *>(done + i0)[t - kBlock / 4] = reinterpret_cast<const uint4 *>(s_flag)[t - kBlock / 4];
        else if (t < kBlock / 4 + kBlock / 8) reinterpret_cast<uint4 *>(truncated + i0)[t - kBlock / 4 - kBlock / 16] = reinterpret_cast<const uint4 *>(s_flag + kBlock)[t - kBlock / 4 - kBlock / 16];
    }
    if (host_flags) {
        __syncthreads();                         // every thread's result stores (obs included) precede thread 0's fence
        if (threadIdx.x == 0) {
            __threadfence_system();
            if (atomicAdd(n_done + 2, 1) == (int)gridDim.x - 1) {
                __threadfence();
                host_flags[0] = *(volatile int32_t *)n_done;
                host_flags[1] = *(volatile int32_t *)(n_done + 1);
                n_done[0] = 0; n_done[1] = 0; n_done[2] = 0;
                __threadfence_system();
                *(volatile int32_t *)(host_flags + 2) = host_seq;
            }
        }
    }
}

// --------------------------------------------------------------- fused T-step random-policy rollout
// State stays in registers for all T steps; per step and env the kernel writes obs (D floats, via the
// double-buffered shared-memory stage -> st.global.cs.v4; ball3d: st.global.cs.v2 per lane), action, reward and done: the [T,N] rollout
// buffer is write-once streaming traffic, 33 B/env-step for ball3d (SURVEY.md §8(d)).
// One warp per CTA: 65 536 envs -> 2048 CTAs = 13.8 per SM (tail imbalance < 2 %); the obs stage is
// private to the warp, so __syncwarp() replaces the CTA barrier (measured 78.6 -> 73.1 us vs 64-thread CTAs).
static constexpr int kRollBlock = 32;

template <int D>
__device__ __forceinline__ void stage_obs(float *stage, const float *o) {     // row-major [env][D] in shared memory
    if (D % 2 == 0) {                                                          // 64-bit stores: conflict-free for D=6
        float2 *s2 = reinterpret_cast<float2 *>(stage + threadIdx.x * D);
#pragma unroll
        for (int j = 0; j < D / 2; ++j) s2[j] = make_float2(o[2 * j], o[2 * j + 1]);
    } else {
#pragma unroll
        for (int j = 0; j < D; ++j) stage[threadIdx.x * D + j] = o[j];
    }
}

template <class Task>
__global__ void __launch_bounds__(kRollBlock)
rollout_random_kernel(EnvPtrs p, int64_t n, uint64_t seed, uint64_t env_base, uint64_t step0, int T,
                      float *__restrict__ obs_buf, int32_t *__restrict__ act_buf, float *__restrict__ rew_buf,
                      uint8_t *__restrict__ done_buf) {
    constexpr int D = Task::D, BLOCK = kRollBlock;
    constexpr bool STAGED = (D != 4);                     // D == 4: one float4 per env straight from registers
    constexpr int NVEC = BLOCK * D / 4;                   // float4 per full block row
    __shared__ __align__(16) float s_obs[STAGED ? 2 * BLOCK * D : 4];
    const int64_t i0 = (int64_t)blockIdx.x * BLOCK, i = i0 + threadIdx.x;
    const bool active = i < n;
    const int valid = (int)min((int64_t)BLOCK, n - i0);
    const uint64_t env_id = env_base + (uint64_t)i;
    const int64_t row_floats = n * D;
    // block-uniform fast path: full block, 16-byte aligned rows
    const bool vec_ok = obs_buf && valid == BLOCK && ((reinterpret_cast<uintptr_t>(obs_buf + i0 * D) & 15u) == 0) &&
                        ((row_floats & 3) == 0);
    const typename Task::Consts cst = Task::load_consts();
    typename Task::State s;
    TmlaActionStream as;
    if (active) {
        s = Task::load(p.buf, i);
        as.seek(seed, env_id, step0, Task::A);
    }
    float *orow = obs_buf ? obs_buf + i0 * D : nullptr;   // block's slice of row t
    int64_t off = i;                                      // t*n + i
    for (int t = 0; t < T; ++t) {
        const uint64_t k = step0 + (uint64_t)t;
        float *stage = STAGED ? s_obs + (t & 1) * BLOCK * D : s_obs;
        if (active) {
            float o[D];
            Task::observe(s, o);                          // observation the action is taken on
            if (STAGED) stage_obs<D>(stage, o);
            else if (obs_buf) {
                float *dst = obs_buf + off * 4;
                if ((reinterpret_cast<uintptr_t>(obs_buf) & 15u) == 0) st_stream_f4(reinterpret_cast<float4 *>(dst), make_float4(o[0], o[1], o[2], o[3]));
                else { dst[0] = o[0]; dst[1] = o[1]; dst[2] = o[2]; dst[3] = o[3]; }
            }
            const int a = as.next(seed, env_id, step0, (uint32_t)t, Task::A);
            float r; bool term, trunc;
            Task::step(cst, s, a, r, term, trunc);
            s.ep_ret = __fadd_rn(s.ep_ret, r);
            const bool d = term || trunc;
            if (act_buf) __stcs(act_buf + off, a);
            if (rew_buf) __stcs(rew_buf + off, r);
            if (done_buf) __stcs(done_buf + off, (uint8_t)(d ? 1 : 0));
            if (d) Task::reset(s, seed, env_id, k + 1, TMLA_TAG_RESET);
        }
        if (STAGED) {
            __syncthreads();
            if (vec_ok) {
                const float4 *s4 = reinterpret_cast<const float4 *>(stage);
                float4 *d4 = reinterpret_cast<float4 *>(orow);
#pragma unroll
                for (int v = 0; v < (NVEC + BLOCK - 1) / BLOCK; ++v) {
                    const int e = v * BLOCK + threadIdx.x;
                    if ((v + 1) * BLOCK <= NVEC || e < NVEC) st_stream_f4(d4 + e, s4[e]);
                }
            } else if (obs_buf) {
                block_store_obs<D, BLOCK, true>(stage, orow, valid);
            }
            if (orow) orow += row_floats;
        }
        off += n;
    }
    if (active) Task::store(p.buf, i, s);
}

// Fast path of the fused rollout (what bench.py times): every block full (n % 32 == 0), all four buffers present,
// 16-byte aligned rows, fewer than 2^31 float4 of observations.  Same arithmetic as the generic kernel above (the tests compare them bit
// for bit) with the loop bookkeeping stripped down, because at 13.8 one-warp CTAs per SM the launch time follows the
// instructions each warp issues per step:
//   - The loop runs over the 16-step blocks of the action stream.  Each block's Philox draw is expanded once into 16
//     packed 4-bit digits, so a step's action is one shift and one mask, with no per-step branch.  A step0 that is not a
//     multiple of 16 starts with a partial block.
//   - For tasks with an episode-indexed reset stream (ball3d) the next initial state is drawn ahead of time (`Spare`) at a
//     block boundary every kSpareEvery steps, so the two Philox blocks of a reset no longer sit inside a divergent branch
//     that ~23 % of the warps enter on every step.  A second reset inside one window draws out of line (draw_spare), which
//     keeps the step loop's code short and contiguous.
//   - Row pointers are bumped once per step and shared memory is indexed directly (no generic pointers).
// Refill period of the ahead-of-time reset draws.  The draw is indexed by the env's episode counter, not by time, so the
// period changes no result — only how often a warp pays two Philox blocks for its consumed lanes (TMLA_SPARE_EVERY).
#ifndef TMLA_SPARE_EVERY
#define TMLA_SPARE_EVERY 64   /* measured on 128-step launches: 16 -> 66.3 us, 32 -> 64.6, 64 -> 63.9, 128 -> 66.7; with the spare carrying its sin products: 32 -> 61.5, 64 -> 61.4, 128 -> 63.9 */
#endif
static constexpr int kSpareEvery = TMLA_SPARE_EVERY;
#ifndef TMLA_ROLLOUT_UNROLL
#define TMLA_ROLLOUT_UNROLL 2
#endif
static constexpr int kRollUnroll = TMLA_ROLLOUT_UNROLL;
static_assert(kSpareEvery % 16 == 0 && ((kSpareEvery / 16) & (kSpareEvery / 16 - 1)) == 0, "a power-of-two number of action blocks");
static_assert(16 % kRollUnroll == 0, "the unrolled step loop covers whole action blocks");

template <class Task>
__device__ __noinline__ typename Task::Spare draw_spare(uint64_t seed, uint64_t env_id, uint32_t episode) {
    return Task::draw(seed, env_id, episode, TMLA_TAG_RESET);
}

template <class Task>
__global__ void __launch_bounds__(kRollBlock)
rollout_fast_kernel(EnvPtrs p, uint32_t n, uint64_t seed, uint64_t env_base, uint64_t step0, int T,
                    float4 *__restrict__ obs4, int32_t *__restrict__ act_buf, float *__restrict__ rew_buf,
                    uint8_t *__restrict__ done_buf) {
    constexpr int D = Task::D, BLOCK = kRollBlock, NVEC = BLOCK * D / 4;
    static_assert(Task::A <= 16, "actions are packed as 4-bit digits");
    // ball3d (D = 6): each lane writes its own 24-byte row as three streaming 64-bit stores.  Measured on B200: 57.4 against
    // 61.5 us per launch when the rows go through the shared-memory stage and leave as 128-bit stores (the __syncwarp and the
    // LDS round trip sit in every step).  The other tasks keep the stage (not measured).
    constexpr bool DIRECT = (D == 6);
    constexpr bool STAGED = (D != 4) && !DIRECT;
    static_assert((BLOCK * D) % 4 == 0, "block rows must be whole float4s");
    __shared__ __align__(16) float s_stage[STAGED ? 2 * BLOCK * D : 4];
    const uint32_t tid = threadIdx.x, i = blockIdx.x * BLOCK + tid;
    const uint64_t env_id = env_base + (uint64_t)i;
    const typename Task::Consts cst = Task::load_consts();
    typename Task::State s = Task::load(p.buf, i);
    // Row pointers of step t, bumped once per step: a 64-bit add each.  A 32-bit element offset scaled into four 64-bit
    // addresses costs more instructions per step (and so does forcing the bumps into IMAD.WIDE, which ptxas splits).
    float *orow = reinterpret_cast<float *>(obs4) + (size_t)i * D;                       // this env's obs (unstaged tasks)
    float4 *vrow = obs4 + blockIdx.x * NVEC + tid;      // this thread's first float4 of the block's rows (staged tasks)
    int32_t *arow = act_buf + i;
    float *rrow = rew_buf + i;
    uint8_t *drow = done_buf + i;
    const uint32_t rowfloats = n * D;                   // floats per obs row (n % 32 == 0)
    uint32_t sb = 0;                                    // stage buffer toggle: 0 / BLOCK*D
    [[maybe_unused]] typename Task::Spare sp;
    [[maybe_unused]] bool have_spare = false;
    // one step with digit j of the current action block; kb: absolute index of the block's first step
    auto step = [&](uint64_t digits, uint32_t j, uint64_t kb) {
        float o[D];
        Task::observe(s, o);                            // observation the action is taken on
        if constexpr (STAGED) {
            if constexpr (D % 2 == 0) {
                float2 *s2 = reinterpret_cast<float2 *>(s_stage + sb + tid * D);
#pragma unroll
                for (int q = 0; q < D / 2; ++q) s2[q] = make_float2(o[2 * q], o[2 * q + 1]);
            } else {
#pragma unroll
                for (int q = 0; q < D; ++q) s_stage[sb + tid * D + q] = o[q];
            }
        } else if constexpr (DIRECT) {
            float2 *d2 = reinterpret_cast<float2 *>(orow);
#pragma unroll
            for (int q = 0; q < D / 2; ++q) __stcs(d2 + q, make_float2(o[2 * q], o[2 * q + 1]));
        } else {
            st_stream_f4(reinterpret_cast<float4 *>(orow), make_float4(o[0], o[1], o[2], o[3]));
        }
        const int a = (int)((uint32_t)(digits >> (4 * j)) & 15u);
        float r; bool term, trunc;
        Task::step(cst, s, a, r, term, trunc);
        s.ep_ret = __fadd_rn(s.ep_ret, r);
        const bool d = term || trunc;
        __stcs(arow, a);
        __stcs(rrow, r);
        __stcs(drow, (uint8_t)(d ? 1 : 0));
        if (d) {
            if constexpr (Task::HAS_SPARE) {
                const uint32_t e = Task::next_episode(s);
                if (!have_spare) sp = draw_spare<Task>(seed, env_id, e);   // second reset inside one window
                Task::begin_episode(s, sp, e);
                have_spare = false;
            } else {
                Task::reset(s, seed, env_id, kb + j + 1, TMLA_TAG_RESET);
            }
        }
        if constexpr (STAGED) {
            if constexpr (BLOCK == 32) __syncwarp(); else __syncthreads();   // one warp per CTA: no CTA barrier needed
            const float4 *s4 = reinterpret_cast<const float4 *>(s_stage + sb);
#pragma unroll
            for (int v = 0; v < (NVEC + BLOCK - 1) / BLOCK; ++v) {
                const int e = v * BLOCK + tid;
                if ((v + 1) * BLOCK <= NVEC || e < NVEC) st_stream_f4(vrow + v * BLOCK, s4[e]);
            }
            sb ^= BLOCK * D;
            vrow += rowfloats / 4;
        } else {
            orow += rowfloats;
        }
        arow += n; rrow += n; drow += n;
    };
    uint64_t kb = step0 & ~(uint64_t)15;                // first step of the current action block
    uint32_t j = (uint32_t)step0 & 15u;                 // digit of the next step within it
    uint32_t left = (uint32_t)T;                        // steps still to run
    for (uint32_t nb = 0; left != 0; ++nb, kb += 16, j = 0) {
        const uint64_t digits = TmlaActionStream::block_digits(seed, env_id, kb >> 4, Task::A);
        if constexpr (Task::HAS_SPARE) {
            if ((nb & (kSpareEvery / 16 - 1)) == 0 && !have_spare) {   // refill consumed spares
                sp = Task::draw(seed, env_id, Task::next_episode(s), TMLA_TAG_RESET);
                have_spare = true;
            }
        }
        if (j == 0 && left >= 16) {
#pragma unroll kRollUnroll   // round 1: 73.2 us (no unroll) / 70.8 us (2) / 72.1 us (4); end of round 2: 63.6 (1) / 61.5-61.8 (2) / 64.2 (3) / 61.6-62.5 (4)
            for (uint32_t q = 0; q < 16; ++q) step(digits, q, kb);
            left -= 16;
        } else {                                        // partial block: step0 % 16 != 0, or the rollout ends inside it
            const uint32_t je = min(16u, j + left);
            left -= je - j;
#pragma unroll 1
            for (; j < je; ++j) step(digits, j, kb);
        }
    }
    Task::store(p.buf, i, s);
}

// ------------------------------------------------------------- policy-driven step (PPO rollout row)
template <int A>
__device__ __forceinline__ void categorical(const float *l, bool deterministic, float u, int &action, float &logp) {
    float m = l[0];
#pragma unroll
    for (int j = 1; j < A; ++j) m = fmaxf(m, l[j]);
    float e[A], sum = 0.0f;
#pragma unroll
    for (int j = 0; j < A; ++j) { e[j] = expf(l[j] - m); sum += e[j]; }
    int a = 0;
    if (deterministic) {                                   // argmax(probs), first maximum wins (torch.argmax)
#pragma unroll
        for (int j = 1; j < A; ++j) if (l[j] > l[a]) a = j;
    } else {                                               // inverse CDF on the unnormalised weights
        const float target = u * sum;
        float c = 0.0f;
        a = A - 1;                                         // guards against target == sum after rounding
        bool found = false;
#pragma unroll
        for (int j = 0; j < A; ++j) {
            c += e[j];
            if (!found && target < c) { a = j; found = true; }
        }
    }
    action = a;
    logp = (l[a] - m) - logf(sum);                         // log_softmax(logits)[a]
}

template <class Task>
__global__ void __launch_bounds__(kBlock)
step_policy_kernel(EnvPtrs p, int64_t n, uint64_t seed, uint64_t env_base, uint64_t step_index,
                   const uint64_t *__restrict__ step_base, const float *__restrict__ logits, int deterministic,
                   int64_t row_index, float *__restrict__ obs_next, int32_t *__restrict__ act, float *__restrict__ logp_out,
                   float *__restrict__ rew, uint8_t *__restrict__ done, int32_t *trunc_count,
                   int32_t *__restrict__ trunc_index, float *__restrict__ trunc_obs, int32_t trunc_capacity,
                   float *ep_stats, float2 *__restrict__ ep_log, int32_t ep_log_cap, int32_t *ep_log_count) {
    constexpr int D = Task::D, A = Task::A;
    __shared__ __align__(16) float s_obs[kBlock * D];
    __shared__ float s_ep[3];                              // CTA sums of the finished episodes: return, length, count
    const int64_t i0 = (int64_t)blockIdx.x * kBlock, i = i0 + threadIdx.x;
    const uint64_t k = step_base ? (*step_base + (uint64_t)row_index) : step_index;
    const unsigned lane = threadIdx.x & 31u, lanes_below = (1u << lane) - 1u;
    if (threadIdx.x < 3) s_ep[threadIdx.x] = 0.0f;
    __syncthreads();
    const bool live = i < n;
    const uint64_t env_id = env_base + (uint64_t)i;
    typename Task::State s;
    float o[D];
    bool d = false, trunc_only = false;
    float ep_r = 0.0f, ep_l = 0.0f;
    if (live) {
        const typename Task::Consts cst = Task::load_consts();
        s = Task::load(p.buf, i);
        float l[A];
#pragma unroll
        for (int j = 0; j < A; ++j) l[j] = logits[i * A + j];
        float u = 0.0f;
        if (!deterministic) u = tmla_u24(tmla_stream_block(seed, env_id, k, TMLA_TAG_SAMPLE, 0).x);
        int a; float lp;
        categorical<A>(l, deterministic != 0, u, a, lp);
        float r; bool term, trunc;
        Task::step(cst, s, a, r, term, trunc);
        s.ep_ret = __fadd_rn(s.ep_ret, r);
        d = term || trunc;
        trunc_only = trunc && !term;
        if (act) act[i] = a;
        if (logp_out) logp_out[i] = lp;
        rew[i] = r;
        done[i] = d ? 1 : 0;
        Task::observe(s, o);
        if (d) { ep_r = s.ep_ret; ep_l = (float)s.steps; }
    }
    // Episode-end bookkeeping, aggregated: a policy that ends episodes quickly (gridworld: ~4 000 of 32 768 envs per step) used to
    // issue three float atomics per finished episode on the SAME three words — ~15 us per step of serialised L2 atomics.  Slots
    // (truncation records, Monitor rows) are now claimed once per warp, the Monitor sums leave once per CTA.  All 32 lanes of
    // every warp get here (kBlock is a multiple of 32; lanes past n carry d = false).
    if (trunc_count) {                                       // collect_rollouts: bootstrap with V(terminal_obs)
        const unsigned m = __ballot_sync(0xffffffffu, trunc_only);
        if (m) {
            const int leader = __ffs(m) - 1;
            int base = 0;
            if ((int)lane == leader) base = atomicAdd(trunc_count, __popc(m));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (trunc_only) {
                const int slot = base + __popc(m & lanes_below);
                if (slot < trunc_capacity) {
                    trunc_index[slot] = (int32_t)(row_index * n + i);
                    thread_store_obs<D>(o, trunc_obs + (int64_t)slot * D);
                }
            }
        }
    }
    const unsigned dm = __ballot_sync(0xffffffffu, d);
    if (dm) {
        if (ep_stats) {                                      // Monitor -> rollout/ep_rew_mean, ep_len_mean
            float wr = ep_r, wl = ep_l;
#pragma unroll
            for (int sh = 16; sh > 0; sh >>= 1) { wr += __shfl_xor_sync(0xffffffffu, wr, sh); wl += __shfl_xor_sync(0xffffffffu, wl, sh); }
            if (lane == 0) { atomicAdd(s_ep + 0, wr); atomicAdd(s_ep + 1, wl); atomicAdd(s_ep + 2, (float)__popc(dm)); }
        }
        if (ep_log) {                                        // Monitor rows of the device path: one (r, l) record per episode
            const int leader = __ffs(dm) - 1;
            int base = 0;
            if ((int)lane == leader) base = atomicAdd(ep_log_count, __popc(dm));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (d) {
                const int slot = base + __popc(dm & lanes_below);
                if (slot < ep_log_cap) ep_log[slot] = make_float2(ep_r, ep_l);
            }
        }
    }
    if (live) {
        if (d) {
            Task::reset(s, seed, env_id, k + 1, TMLA_TAG_RESET);
            Task::observe(s, o);
        }
        Task::store(p.buf, i, s);
#pragma unroll
        for (int j = 0; j < D; ++j) s_obs[threadIdx.x * D + j] = o[j];
    }
    __syncthreads();
    if (ep_stats && threadIdx.x == 0 && s_ep[2] > 0.0f) {
        atomicAdd(ep_stats + 0, s_ep[0]);
        atomicAdd(ep_stats + 1, s_ep[1]);
        atomicAdd(ep_stats + 2, s_ep[2]);
    }
    block_store_obs<D, kBlock, false>(s_obs, obs_next + i0 * D, (int)min((int64_t)kBlock, n - i0));
}

__global__ void counter_add_kernel(uint64_t *c, uint64_t n) { *c += n; }

// ---- arithmetic self-test (test hook): the hand-rolled correctly-rounded divisions and the short sin
// polynomial against the IEEE intrinsics / libdevice over every input the tasks can produce.
//   out[0] div3_rn != __fdiv_rn(x,3) count over all floats in [0, 8)      (ball3d |pos| <= ~4.3)
//   out[1] div5_rn != __fdiv_rn(k,5) count over k in [-5,5]
//   out[2] max ulp distance of sin_small vs sin() over 2^22 points of [-MAX_TILT, MAX_TILT]
__global__ void selftest_arith_kernel(unsigned long long *out) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    unsigned long long bad3 = 0;
    for (uint32_t bits = tid; bits < 0x41000000u; bits += nth) {
        const float x = __uint_as_float(bits);
        bad3 += (__float_as_uint(div3_rn(x)) != __float_as_uint(__fdiv_rn(x, 3.0f)));
    }
    if (bad3) atomicAdd(out + 0, bad3);
    if (tid < 11) {
        const float k = (float)((int)tid - 5);
        if (__float_as_uint(div5_rn(k)) != __float_as_uint(__fdiv_rn(k, 5.0f))) atomicAdd(out + 1, 1ull);
    }
    unsigned long long worst = 0;
    for (uint32_t j = tid; j < (1u << 22); j += nth) {
        const double x = kB3.max_tilt * (2.0 * ((double)j + 0.5) / 4194304.0 - 1.0);
        const long long a = __double_as_longlong(sin_small(x)), b = __double_as_longlong(sin(x));
        const unsigned long long d = (unsigned long long)(a > b ? a - b : b - a);
        worst = d > worst ? d : worst;
    }
    atomicMax(out + 2, worst);
}

// ------------------------------------------------------------------------------------ dispatch
#define TASK_SWITCH(task, CALL)                                   \
    switch (task) {                                               \
        case TMLA_BASIC: { using TaskT = BasicTask; CALL; } break;        \
        case TMLA_BALL3D: { using TaskT = Ball3DTask; CALL; } break;      \
        case TMLA_GRIDWORLD: { using TaskT = GridWorldTask; CALL; } break; \
        case TMLA_PUSH: { using TaskT = PushTask; CALL; } break;          \
        case TMLA_WALLJUMP: { using TaskT = WallJumpTask; CALL; } break;  \
        case TMLA_BRICKBREAK: { using TaskT = BrickBreakTask; CALL; } break; \
        case TMLA_BICYCLE: { using TaskT = BicycleTask; CALL; } break;       \
        case TMLA_GLIDER: { using TaskT = GliderTask; CALL; } break;         \
        default: tmla_set_error("unknown task %d", task); return TMLA_EINVAL; \
    }

static EnvPtrs ptrs_of(const tmla_env *h) {
    EnvPtrs p;
    for (int b = 0; b < 4; ++b) p.buf[b] = h->buf[b];
    return p;
}
static inline unsigned grid_for(int64_t n) { return (unsigned)ceil_div64(n, kBlock); }

static const int kObsDim[TMLA_NUM_TASKS] = {BasicTask::D, Ball3DTask::D, GridWorldTask::D, PushTask::D, WallJumpTask::D, BrickBreakTask::D, BicycleTask::D, GliderTask::D};
static const int kNumActions[TMLA_NUM_TASKS] = {BasicTask::A, Ball3DTask::A, GridWorldTask::A, PushTask::A, WallJumpTask::A, BrickBreakTask::A, BicycleTask::A, GliderTask::A};
static const int kMaxSteps[TMLA_NUM_TASKS] = {BasicTask::MAX_STEPS, Ball3DTask::MAX_STEPS, GridWorldTask::MAX_STEPS, PushTask::MAX_STEPS,
                                              WallJumpTask::MAX_STEPS, BrickBreakTask::MAX_STEPS, BicycleTask::MAX_STEPS, GliderTask::MAX_STEPS};
static const int kStateSize[TMLA_NUM_TASKS] = {(int)sizeof(tmla_basic_state), (int)sizeof(tmla_ball3d_state), (int)sizeof(tmla_gridworld_state),
                                               (int)sizeof(tmla_push_state), (int)sizeof(tmla_walljump_state), (int)sizeof(tmla_brickbreak_state),
                                               (int)sizeof(tmla_bicycle_state), (int)sizeof(tmla_glider_state)};

// staging layout shared by the device block and its pinned host mirror (16-byte aligned sections):
//   actions i32[n] | obs f32[n,D] | reward f32[n] | done u8[n] | truncated u8[n] | flags i32[4] {n_done, bad_action}
//   | compact records f32[n,3+D] | terminal_obs f32[n,D] | ep_return f32[n] | ep_length i32[n]   (the last three host-only)
// obs..flags plus the head of the record area is one contiguous span -> ONE device-to-host copy per step.  The same span,
// re-based at `obs`, is the layout of a RESULT BLOCK (tmla_result_block_*): pinned memory a binding hands out to its caller,
// so that the copy engine writes a step's results straight into the arrays the caller receives.  The episode-end payload
// travels as n_done compact records (36 B each for ball3d); the dense terminal_obs/ep_return/ep_length views of
// tmla_step_pinned are filled from them on the host: only the entries of envs whose `done` flag is set are meaningful.
static inline int record_words(int D) { return (3 + D + 3) & ~3; }      // {idx, ret, len, tobs[D]} padded to whole 16-byte chunks
struct StageLayout { size_t act, obs, rew, done, trunc, flags, crec, tobs, ret, len, end; };
static StageLayout stage_layout(int64_t n, int D) {
    auto up = [](size_t x) { return (x + 15) & ~(size_t)15; };
    StageLayout L;
    L.act = 0;
    L.obs = up(L.act + 4 * n);
    L.rew = L.obs + 4 * n * D;
    L.done = L.rew + 4 * n;
    L.trunc = L.done + n;
    L.flags = up(L.trunc + n);
    L.crec = L.flags + 16;                      // compact episode-end records {idx, ret, len, tobs[D]}, at most n of them
    L.tobs = up(L.crec + 4 * n * record_words(D));
    L.ret = L.tobs + 4 * n * D;
    L.len = L.ret + 4 * n;
    L.end = L.len + 4 * n;
    return L;
}


#if defined(__x86_64__)
// host-side action staging (tmla_stage_actions): AVX2 bodies, selected at run time; they return how many elements they handled
__attribute__((target("avx2"))) static int64_t stage_actions32_avx2(const int32_t *src, uint8_t *dst, int64_t n, uint64_t *ored, uint32_t *mx) {
    __m256i acc = _mm256_setzero_si256(), vmx = _mm256_setzero_si256();
    const __m256i perm = _mm256_setr_epi32(0, 4, 1, 5, 2, 6, 3, 7);
    int64_t i = 0;
    for (; i + 32 <= n; i += 32) {
        const __m256i a = _mm256_loadu_si256((const __m256i *)(src + i)), b = _mm256_loadu_si256((const __m256i *)(src + i + 8));
        const __m256i c = _mm256_loadu_si256((const __m256i *)(src + i + 16)), d = _mm256_loadu_si256((const __m256i *)(src + i + 24));
        acc = _mm256_or_si256(acc, _mm256_or_si256(_mm256_or_si256(a, b), _mm256_or_si256(c, d)));
        __m256i p = _mm256_packus_epi16(_mm256_packs_epi32(a, b), _mm256_packs_epi32(c, d));   // per 128-bit lane: a b c d quarters
        p = _mm256_permutevar8x32_epi32(p, perm);
        vmx = _mm256_max_epu8(vmx, p);
        _mm256_storeu_si256((__m256i *)(dst + i), p);
    }
    uint64_t t[4]; uint8_t m8[32];
    _mm256_storeu_si256((__m256i *)t, acc); _mm256_storeu_si256((__m256i *)m8, vmx);
    const uint64_t o = t[0] | t[1] | t[2] | t[3];
    *ored |= (o | (o >> 32)) & 0xFFFFFFFFull;
    for (int k = 0; k < 32; ++k) *mx = m8[k] > *mx ? m8[k] : *mx;
    return i;
}
__attribute__((target("avx2"))) static int64_t stage_actions64_avx2(const int64_t *src, uint8_t *dst, int64_t n, uint64_t *ored, uint32_t *mx) {
    __m256i acc = _mm256_setzero_si256(), vmx = _mm256_setzero_si256();
    const __m256i lo = _mm256_setr_epi32(0, 2, 4, 6, 0, 2, 4, 6), perm = _mm256_setr_epi32(0, 4, 1, 5, 2, 6, 3, 7);
    int64_t i = 0;
    for (; i + 32 <= n; i += 32) {
        __m256i w[4];
        for (int k = 0; k < 4; ++k) {
            const __m256i x = _mm256_loadu_si256((const __m256i *)(src + i + 8 * k)), y = _mm256_loadu_si256((const __m256i *)(src + i + 8 * k + 4));
            acc = _mm256_or_si256(acc, _mm256_or_si256(x, y));
            const __m256i xl = _mm256_permutevar8x32_epi32(x, lo), yl = _mm256_permutevar8x32_epi32(y, lo);   // low dwords -> low half
            w[k] = _mm256_inserti128_si256(xl, _mm256_castsi256_si128(yl), 1);
        }
        __m256i p = _mm256_packus_epi16(_mm256_packs_epi32(w[0], w[1]), _mm256_packs_epi32(w[2], w[3]));
        p = _mm256_permutevar8x32_epi32(p, perm);
        vmx = _mm256_max_epu8(vmx, p);
        _mm256_storeu_si256((__m256i *)(dst + i), p);
    }
    uint64_t t[4]; uint8_t m8[32];
    _mm256_storeu_si256((__m256i *)t, acc); _mm256_storeu_si256((__m256i *)m8, vmx);
    const uint64_t o = t[0] | t[1] | t[2] | t[3];
    *ored |= (o & ~7ull) ? 0xFFFFFFFFull : (o & 7ull);
    for (int k = 0; k < 32; ++k) *mx = m8[k] > *mx ? m8[k] : *mx;
    return i;
}
#endif

extern "C" {

int tmla_task_from_name(const char *name) {
    if (!name) { tmla_set_error("task name is NULL"); return TMLA_EINVAL; }
    if (!strcmp(name, "basic")) return TMLA_BASIC;
    if (!strcmp(name, "ball3d")) return TMLA_BALL3D;
    if (!strcmp(name, "gridworld")) return TMLA_GRIDWORLD;
    if (!strcmp(name, "push")) return TMLA_PUSH;
    if (!strcmp(name, "walljump")) return TMLA_WALLJUMP;
    if (!strcmp(name, "brickbreak")) return TMLA_BRICKBREAK;
    if (!strcmp(name, "bicycle")) return TMLA_BICYCLE;
    if (!strcmp(name, "glider")) return TMLA_GLIDER;
    tmla_set_error("no CUDA backend for task '%s' (have: basic, ball3d, gridworld, push, walljump, brickbreak, bicycle, glider)", name);
    return TMLA_EINVAL;
}
#define TASK_META(fn, table)                                                                   \
    int fn(int task) {                                                                         \
        if (task < 0 || task >= TMLA_NUM_TASKS) { tmla_set_error(#fn ": unknown task %d", task); return TMLA_EINVAL; } \
        return table[task];                                                                    \
    }
TASK_META(tmla_task_obs_dim, kObsDim)
TASK_META(tmla_task_num_actions, kNumActions)
TASK_META(tmla_task_max_steps, kMaxSteps)
TASK_META(tmla_task_state_size, kStateSize)

int tmla_create(int task, int64_t n_envs, uint64_t seed, uint64_t env_id_base, int device, tmla_env **out) {
    TMLA_REQUIRE(out != nullptr, "out is NULL");
    TMLA_REQUIRE(task >= 0 && task < TMLA_NUM_TASKS, "unknown task");
    TMLA_REQUIRE(n_envs > 0 && n_envs < (int64_t)1 << 31, "n_envs must be in (0, 2^31)");
    int ndev = 0;
    TMLA_CUDA(cudaGetDeviceCount(&ndev));
    TMLA_REQUIRE(device >= 0 && device < ndev, "no such CUDA device (this library has no CPU path)");
    DeviceGuard guard(device);
    tmla_env *h = new (std::nothrow) tmla_env();
    if (!h) { tmla_set_error("out of host memory"); return TMLA_ENOMEM; }
    memset(h, 0, sizeof(*h));
    h->task = task; h->n = n_envs; h->seed = seed; h->env_id_base = env_id_base; h->device = device;
    h->rec_hint = 256;
    int nbuf = 0;
    size_t pb[4] = {0, 0, 0, 0};
    TASK_SWITCH(task, nbuf = TaskT::NBUF; for (int b = 0; b < nbuf; ++b) pb[b] = TaskT::plane_bytes(b));
    for (int b = 0; b < nbuf; ++b) {
        cudaError_t e = cudaMalloc(&h->buf[b], pb[b] * (size_t)n_envs);
        if (e != cudaSuccess) { tmla_set_error("cudaMalloc(state plane %d): %s", b, cudaGetErrorString(e)); tmla_destroy(h); return TMLA_ENOMEM; }
    }
    const int D = kObsDim[task];
    // staging layout: actions i32 | obs | reward | terminal_obs | ep_return | ep_length | done | truncated
    h->stage_bytes = stage_layout(n_envs, D).end + 64;
    if (cudaMalloc(&h->d_stage, h->stage_bytes) != cudaSuccess || cudaMallocHost(&h->h_stage, h->stage_bytes) != cudaSuccess ||
        cudaMalloc((void **)&h->err_flag, sizeof(int)) != cudaSuccess || cudaMalloc((void **)&h->d_ndone, sizeof(int32_t)) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->dev_evt, cudaEventDisableTiming) != cudaSuccess) {
        tmla_set_error("allocating staging buffers: %s", cudaGetErrorString(cudaGetLastError()));
        tmla_destroy(h);
        return TMLA_ENOMEM;
    }
    TMLA_CUDA(cudaMemset(h->err_flag, 0, sizeof(int)));
    memset((char *)h->h_stage + stage_layout(n_envs, D).end, 0, 64);      // ready[] words of the chunked host step
    TMLA_CUDA(cudaMemset((char *)h->d_stage + stage_layout(n_envs, D).flags, 0, 16));
    TMLA_CUDA(cudaMemset((char *)h->d_stage + stage_layout(n_envs, D).end, 0, 64));      // device copies of the ready[] words
    TMLA_CUDA(cudaMemset(h->d_ndone, 0, sizeof(int32_t)));
    *out = h;
    int rc = tmla_reset(h, nullptr, nullptr);
    if (rc) return rc;
    TMLA_CUDA(cudaStreamSynchronize(nullptr));
    h->dev_dirty = false;
    return TMLA_OK;
}

int tmla_destroy(tmla_env *h) {
    if (!h) return TMLA_OK;
    DeviceGuard guard(h->device);
    for (int b = 0; b < 4; ++b) if (h->buf[b]) cudaFree(h->buf[b]);
    if (h->d_stage) cudaFree(h->d_stage);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->err_flag) cudaFree(h->err_flag);
    if (h->d_ndone) cudaFree(h->d_ndone);
    for (int b = 0; b < 4; ++b) if (h->shadow[b]) cudaFree(h->shadow[b]);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->dev_evt) cudaEventDestroy(h->dev_evt);
    if (h->rollout_plan && h->rollout_plan_free) h->rollout_plan_free(h->rollout_plan);
    delete h;
    return TMLA_OK;
}

int tmla_seed(tmla_env *h, uint64_t seed) { TMLA_REQUIRE(h, "handle is NULL"); h->seed = seed; return TMLA_OK; }
int64_t tmla_num_envs(const tmla_env *h) { return h ? h->n : 0; }
uint64_t tmla_step_count(const tmla_env *h) { return h ? h->step_count : 0; }
int tmla_advance_steps(tmla_env *h, uint64_t n) { TMLA_REQUIRE(h, "handle is NULL"); h->step_count += n; return TMLA_OK; }

int tmla_reset(tmla_env *h, float *obs, void *stream) {
    TMLA_REQUIRE(h, "handle is NULL");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (st != h->own_stream) mark_device_path(h, st);
    TASK_SWITCH(h->task, (reset_kernel<TaskT><<<grid_for(h->n), kBlock, 0, st>>>(
                             ptrs_of(h), h->n, h->seed, h->env_id_base, h->step_count, TMLA_TAG_RESET_ALL, obs)));
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int tmla_step(tmla_env *h, const int32_t *actions, float *obs, float *reward, uint8_t *done, uint8_t *truncated,
              float *terminal_obs, float *ep_return, int32_t *ep_length, void *stream) {
    TMLA_REQUIRE(h, "handle is NULL");
    TMLA_REQUIRE(actions && obs && reward && done && truncated, "actions/obs/reward/done/truncated must be non-NULL");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    mark_device_path(h, st);
    TASK_SWITCH(h->task, (step_kernel<TaskT><<<grid_for(h->n), kBlock, 0, st>>>(
                             ptrs_of(h), h->n, h->seed, h->env_id_base, h->step_count, actions, obs, reward, done,
                             truncated, terminal_obs, ep_return, ep_length, nullptr, h->err_flag, nullptr, nullptr, 0, 0, nullptr, nullptr, 1, EnvPtrs{})));
    TMLA_LAUNCH_CHECK();
    h->step_count += 1;
    return TMLA_OK;
}

// VecEnv.step with the actions already in the pinned stage: H2D actions -> kernel -> ONE D2H of obs..flags and the head of
// the record area straight into `block` (pinned, result-block layout), then a synchronise.  The head is sized from the
// previous step's count; only a step that finishes more episodes than that pays a second copy.
static bool host_step_mapped() {      // TMLA_HOST_STEP=copy selects the copy-engine path (default: zero-copy mapped writes)
    static const bool mapped = [] { const char *e = getenv("TMLA_HOST_STEP"); return !(e && !strcmp(e, "copy")); }();
    return mapped;
}
// Waits until the last CTA of a mapped host step has published {n_done, bad_action, seq} in the block's flag words: ONE launch
// (or one launch per chunk) per step and no stream synchronise — the host polls the sequence word, which the kernel writes
// after all results (cudaStreamQuery every 4096 polls catches a failed launch; the flag word of d_stage is zeroed at create).
static int wait_block_published(tmla_env *h, const char *block, int seq, int64_t *n_done) {
    const StageLayout L = stage_layout(h->n, kObsDim[h->task]);
    const int32_t *bflags = (const int32_t *)(block + (L.flags - L.obs));
    volatile const int32_t *hseq = (volatile const int32_t *)bflags + 2;
    cudaStream_t st = h->own_stream;
    static const bool poll = [] { const char *e = getenv("TMLA_HOST_STEP"); return !(e && !strcmp(e, "sync")); }();
    if (!poll) TMLA_CUDA(cudaStreamSynchronize(st));
    for (uint32_t spins = 1; *hseq != seq; ++spins) {
        if ((spins & 4095u) == 0) {
            const cudaError_t q = cudaStreamQuery(st);
            if (q != cudaErrorNotReady) { TMLA_CUDA(q); if (*hseq != seq) { tmla_set_error("step kernel finished without publishing its results"); return TMLA_ECUDA; } }
        }
    }
    __sync_synchronize();
    if (n_done) *n_done = bflags[0];
    if (bflags[1]) {
        tmla_set_error("an action outside [0,%d) was passed to step()", kNumActions[h->task]);
        return TMLA_EACTION;
    }
    return TMLA_OK;
}
static int step_into_block(tmla_env *h, char *block, int64_t *n_done) {
    DeviceGuard guard(h->device);
    { const int rc = order_after_device_path(h); if (rc) return rc; }
    const int act_u8 = h->act_u8;                          // set by tmla_stage_actions for exactly one step
    h->act_u8 = 0;
    const int64_t n = h->n;
    const int D = kObsDim[h->task];
    const StageLayout L = stage_layout(n, D);
    char *d = (char *)h->d_stage, *p = (char *)h->h_stage;
    cudaStream_t st = h->own_stream;
    int32_t *dflags = (int32_t *)(d + L.flags);
    const int32_t *bflags = (const int32_t *)(block + (L.flags - L.obs));
    if (host_step_mapped()) {
        // zero-copy: pinned memory is device-addressable under UVA.  The kernel reads the actions and writes obs / reward /
        // done / truncated / records over PCIe itself (coalesced 128-byte lines), overlapping the transfer with the step
        // arithmetic and saving the two copy-engine hand-offs; only the 16-byte flag word is copied afterwards.
        char *b = block - L.obs;      // block-relative addressing with stage offsets
        const int seq = (int)((h->step_count + 1) & 0x3FFFFFFF) | 0x40000000;
        volatile int32_t *hseq = (volatile int32_t *)(b + L.flags) + 2;
        *hseq = 0;
        TASK_SWITCH(h->task, (step_kernel<TaskT><<<grid_for(n), kBlock, 0, st>>>(
                                 ptrs_of(h), n, h->seed, h->env_id_base, h->step_count, (const int32_t *)(p + L.act),
                                 (float *)(b + L.obs), (float *)(b + L.rew), (uint8_t *)(b + L.done), (uint8_t *)(b + L.trunc),
                                 nullptr, nullptr, nullptr, dflags, dflags + 1, (float *)(b + L.crec), (int32_t *)(b + L.flags), seq, act_u8, nullptr, nullptr, 1, EnvPtrs{})));
        TMLA_LAUNCH_CHECK();
        h->step_count += 1;
        // ONE launch per step, no stream synchronise: poll the sequence word the last CTA writes after all results
        // (cudaStreamQuery every 4096 polls catches a failed launch; the flag word of d_stage is zeroed at create)
        return wait_block_published(h, block, seq, n_done);
    }
    TMLA_CUDA(cudaMemcpyAsync(d + L.act, p + L.act, (act_u8 ? 1 : 4) * n, cudaMemcpyHostToDevice, st));
    TMLA_CUDA(cudaMemsetAsync(dflags, 0, 16, st));
    TASK_SWITCH(h->task, (step_kernel<TaskT><<<grid_for(n), kBlock, 0, st>>>(
                             ptrs_of(h), n, h->seed, h->env_id_base, h->step_count, (const int32_t *)(d + L.act),
                             (float *)(d + L.obs), (float *)(d + L.rew), (uint8_t *)(d + L.done), (uint8_t *)(d + L.trunc),
                             nullptr, nullptr, nullptr, dflags, dflags + 1, (float *)(d + L.crec), nullptr, 0, act_u8, nullptr, nullptr, 1, EnvPtrs{})));
    TMLA_LAUNCH_CHECK();
    h->step_count += 1;
    const size_t rec = (size_t)4 * record_words(D);
    const int64_t head = h->rec_hint < n ? h->rec_hint : n;
    TMLA_CUDA(cudaMemcpyAsync(block, d + L.obs, (L.crec - L.obs) + rec * head, cudaMemcpyDeviceToHost, st));
    TMLA_CUDA(cudaStreamSynchronize(st));
    const int32_t nd = bflags[0];
    if (nd > head) {
        TMLA_CUDA(cudaMemcpyAsync(block + (L.crec - L.obs) + rec * head, d + L.crec + rec * head, rec * (nd - head), cudaMemcpyDeviceToHost, st));
        TMLA_CUDA(cudaStreamSynchronize(st));
    }
    h->rec_hint = 256 + nd + nd / 2;
    if (n_done) *n_done = nd;
    if (bflags[1]) {
        tmla_set_error("an action outside [0,%d) was passed to step()", kNumActions[h->task]);
        return TMLA_EACTION;
    }
    return TMLA_OK;
}

// Actions of the next host step: range-checked and converted in ONE pass over the caller's array into the pinned action
// stage, as one byte per action (every task has <= 5 actions) — a quarter of the PCIe reads of int32, and an out-of-range
// action is reported BEFORE anything is launched, like the reference's ACTION_DELTAS[action] (ball3d.py:76) raising before
// any state change.  elem_bytes: 4 (int32) or 8 (int64, what SB3 hands to VecEnv.step).
// range [i0, i0 + m) of the caller's action array -> one byte per action in the pinned stage; accumulates the evidence of an
// out-of-range value (OR of the raw lanes: negatives and anything >= 8; running maximum of the narrowed bytes: A..7)
static void stage_action_range(tmla_env *h, const void *actions, int elem_bytes, int64_t i0, int64_t m, uint64_t *ored, uint32_t *mx) {
    uint8_t *dst = (uint8_t *)h->h_stage + stage_layout(h->n, kObsDim[h->task]).act + i0;
    const char *src = (const char *)actions + i0 * elem_bytes;
    int64_t i = 0;
#if defined(__x86_64__)
    static const bool has_avx2 = __builtin_cpu_supports("avx2");
    if (has_avx2)
        i = elem_bytes == 4 ? stage_actions32_avx2((const int32_t *)src, dst, m, ored, mx)
                            : stage_actions64_avx2((const int64_t *)src, dst, m, ored, mx);
#endif
    for (; i < m; ++i) {       // (a plain scalar loop costs ~0.5 ns per action)
        const uint64_t a = elem_bytes == 4 ? (uint64_t)(uint32_t)((const int32_t *)src)[i] : (uint64_t)((const int64_t *)src)[i];
        *ored |= (a | (a >> 32)) & 0xFFFFFFFFull;
        *mx = (uint32_t)(a & 7u) > *mx ? (uint32_t)(a & 7u) : *mx;
        dst[i] = (uint8_t)a;
    }
}
static inline bool staged_actions_bad(const tmla_env *h, uint64_t ored, uint32_t mx) {
    return (ored & ~7ull) != 0 || mx >= (uint32_t)kNumActions[h->task];        // every task has <= 8 actions
}

int tmla_stage_actions(tmla_env *h, const void *actions, int elem_bytes) {
    TMLA_REQUIRE(h && actions, "handle/actions is NULL");
    TMLA_REQUIRE(elem_bytes == 4 || elem_bytes == 8, "elem_bytes must be 4 (int32) or 8 (int64)");
    uint64_t ored = 0;
    uint32_t mx = 0;
    stage_action_range(h, actions, elem_bytes, 0, h->n, &ored, &mx);
    h->act_u8 = 1;
    if (staged_actions_bad(h, ored, mx)) {
        tmla_set_error("an action outside [0,%d) was passed to step()", kNumActions[h->task]);
        return TMLA_EACTION;
    }
    return TMLA_OK;
}

// Monitor rows for the policy-driven device path (tmla_step_policy / tmla_rollout): every finished episode appends
// {ep_return, ep_length} at slot atomicAdd(count); records beyond `capacity` are counted but dropped.  NULL detaches.
int tmla_set_episode_log(tmla_env *h, float *records, int32_t capacity, int32_t *count) {
    TMLA_REQUIRE(h, "handle is NULL");
    TMLA_REQUIRE((!records && !count) || (records && count && capacity > 0), "records/count must both be set (capacity > 0) or both NULL");
    h->ep_log = reinterpret_cast<float2 *>(records);
    h->ep_log_cap = records ? capacity : 0;
    h->ep_log_count = count;
    return TMLA_OK;
}

int tmla_step_block(tmla_env *h, void *block, int64_t *n_done) {
    TMLA_REQUIRE(h && block, "handle/block is NULL");
    return step_into_block(h, (char *)block, n_done);
}

// VecEnv.step_async / step_wait on the caller's own action array.  For int64 actions above 16 384 envs (what SB3 passes) the
// step kernel is launched FIRST and the batch is cut into chunks (TMLA_HOST_CHUNKS; default 4 for int64, 1 for int32): the host
// range-checks and narrows chunk c, then publishes ready[c] in mapped pinned memory; the CTAs of that chunk, already resident,
// step their envs and write the results into the block while the host stages chunk c+1, so that the staging pass hides behind
// the launch latency and the first chunks' PCIe traffic.  Measured on B200 at 65 536 ball3d envs (profiles/e2e_chunks.py, C
// level, begin + end): int64 89.5 us unchunked -> 82.6 (4 chunks) / 85.2 (8); int32 70.7 -> 73.5 / 75.1 — the GPU side of a step
// is 17 us of fixed latency + 0.65 ns per env of PCIe (46 GB/s), and only the staging of int64 (29.8 us for 512 KB of cache-cold
// actions against 11.1 us for int32) is long enough to be worth hiding; staging beside the incoming PCIe writes is itself
// ~50 % slower.  (One launch PER chunk was measured first: every extra launch costs ~7 us on the stream — 80 / 88 / 93 / 124 /
// 185 us per step with 1 / 2 / 4 / 8 / 16 launches; and letting every CTA poll the host word saturated the non-posted PCIe
// reads: 400-540 us per step.)
// "A rejected step changes nothing" still holds: the kernel keeps the pre-step state in shadow planes, and when a later chunk
// holds an out-of-range action the remaining chunks are told to leave and the envs already stepped are put back before the
// error returns.
static int host_chunks(const tmla_env *h, int elem_bytes) {
    static const int env_req = [] { const char *e = getenv("TMLA_HOST_CHUNKS"); const int v = e ? atoi(e) : 0; return v < 0 ? 0 : (v > 16 ? 16 : v); }();
    const int req = env_req ? env_req : (elem_bytes == 8 ? 4 : 1);
    if (h->n < 16384 || req == 1) return 1;
    // every CTA must be resident at once (a waiting CTA never yields its slot)
    static int resident[TMLA_NUM_TASKS];
    static int sms = 0;
    if (!sms) { cudaDeviceProp pr; if (cudaGetDeviceProperties(&pr, h->device) != cudaSuccess) return 1; sms = pr.multiProcessorCount; }
    if (!resident[h->task]) {
        int per_sm = 0;
        TASK_SWITCH(h->task, if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, step_kernel<TaskT>, kBlock, 0) != cudaSuccess) per_sm = 0);
        resident[h->task] = per_sm > 0 ? per_sm : -1;
    }
    if (resident[h->task] < 0 || (int64_t)grid_for(h->n) > (int64_t)resident[h->task] * sms) return 1;
    return req;
}
int tmla_step_block_begin(tmla_env *h, const void *actions, int elem_bytes, void *block) {
    TMLA_REQUIRE(h && actions && block, "handle/actions/block is NULL");
    TMLA_REQUIRE(elem_bytes == 4 || elem_bytes == 8, "elem_bytes must be 4 (int32) or 8 (int64)");
    TMLA_REQUIRE(h->pend_seq == 0, "a host step is already in flight (call tmla_step_block_end first)");
    DeviceGuard guard(h->device);
    const int nchunks = host_step_mapped() ? host_chunks(h, elem_bytes) : 1;
    if (nchunks == 1) {                                      // small batches / copy-engine variant: stage now, run the step in _end
        const int rc = tmla_stage_actions(h, actions, elem_bytes);
        if (rc == TMLA_OK) h->pend_seq = -1;
        return rc;
    }
    { const int rc = order_after_device_path(h); if (rc) return rc; }
    const int64_t n = h->n;
    const int D = kObsDim[h->task];
    const StageLayout L = stage_layout(n, D);
    const int chunk_ctas = (int)ceil_div64(grid_for(n), nchunks);
    const int64_t chunk = (int64_t)chunk_ctas * kBlock;
    int nbuf = 0;
    size_t pb[4] = {0, 0, 0, 0};
    TASK_SWITCH(h->task, nbuf = TaskT::NBUF; for (int b = 0; b < nbuf; ++b) pb[b] = TaskT::plane_bytes(b));
    EnvPtrs shadow{};
    for (int b = 0; b < nbuf; ++b) {
        if (!h->shadow[b] && cudaMalloc(&h->shadow[b], pb[b] * (size_t)n) != cudaSuccess) {
            tmla_set_error("cudaMalloc(shadow state plane %d): %s", b, cudaGetErrorString(cudaGetLastError()));
            return TMLA_ENOMEM;
        }
        shadow.buf[b] = h->shadow[b];
    }
    char *d = (char *)h->d_stage, *p = (char *)h->h_stage, *b = (char *)block - L.obs;
    cudaStream_t st = h->own_stream;
    int32_t *dflags = (int32_t *)(d + L.flags);
    volatile int32_t *ready = (volatile int32_t *)(p + L.end);          // 16 words after the layout (stage_bytes = end + 64)
    const int seq = (int)((h->step_count + 1) & 0x3FFFFFFF) | 0x40000000;
    *((volatile int32_t *)(b + L.flags) + 2) = 0;
    TASK_SWITCH(h->task, (step_kernel<TaskT><<<grid_for(n), kBlock, 0, st>>>(
                             ptrs_of(h), n, h->seed, h->env_id_base, h->step_count, (const int32_t *)(p + L.act),
                             (float *)(b + L.obs), (float *)(b + L.rew), (uint8_t *)(b + L.done), (uint8_t *)(b + L.trunc),
                             nullptr, nullptr, nullptr, dflags, dflags + 1, (float *)(b + L.crec), (int32_t *)(b + L.flags), seq, 1,
                             (const int32_t *)ready, (int32_t *)(d + L.end), chunk_ctas, shadow)));
    TMLA_LAUNCH_CHECK();
    uint64_t ored = 0;
    uint32_t mx = 0;
    int c = 0;
    for (int64_t i0 = 0; i0 < n; i0 += chunk, ++c) {
        const int64_t m = n - i0 < chunk ? n - i0 : chunk;
        stage_action_range(h, actions, elem_bytes, i0, m, &ored, &mx);
        if (staged_actions_bad(h, ored, mx)) {
            // tell the chunks not yet released to leave, wait, and put the envs already stepped back: state planes, device counters
            for (int q = c; q < nchunks; ++q) ready[q] = ~seq;
            __sync_synchronize();
            TMLA_CUDA(cudaStreamSynchronize(st));
            for (int q = 0; q < nbuf && i0 > 0; ++q) TMLA_CUDA(cudaMemcpyAsync(h->buf[q], h->shadow[q], pb[q] * (size_t)i0, cudaMemcpyDeviceToDevice, st));
            TMLA_CUDA(cudaMemsetAsync(dflags, 0, 16, st));
            TMLA_CUDA(cudaMemsetAsync(d + L.end, 0, 64, st));
            TMLA_CUDA(cudaStreamSynchronize(st));
            for (int q = 0; q < 16; ++q) ready[q] = 0;       // the next attempt reuses this sequence number
            tmla_set_error("an action outside [0,%d) was passed to step()", kNumActions[h->task]);
            return TMLA_EACTION;
        }
        __sync_synchronize();                                // the narrowed actions are visible before the flag
        ready[c] = seq;
    }
    h->step_count += 1;
    h->pend_seq = seq;
    return TMLA_OK;
}

int tmla_step_block_end(tmla_env *h, void *block, int64_t *n_done) {
    TMLA_REQUIRE(h && block, "handle/block is NULL");
    TMLA_REQUIRE(h->pend_seq != 0, "no host step in flight (call tmla_step_block_begin first)");
    const int seq = h->pend_seq;
    h->pend_seq = 0;
    if (seq == -1) return step_into_block(h, (char *)block, n_done);
    return wait_block_published(h, (const char *)block, seq, n_done);
}

int tmla_step_pinned(tmla_env *h, int64_t *n_done) {
    TMLA_REQUIRE(h, "handle is NULL");
    const int D = kObsDim[h->task];
    const StageLayout L = stage_layout(h->n, D);
    char *p = (char *)h->h_stage;
    int64_t nd = 0;
    const int rc = step_into_block(h, p + L.obs, &nd);
    if (rc != TMLA_OK && rc != TMLA_EACTION) return rc;
    if (nd > 0) {   // episode-end payload: nd compact records, scattered into the dense host arrays
        const size_t rec = (size_t)4 * record_words(D);
        float *tobs = (float *)(p + L.tobs), *ret = (float *)(p + L.ret);
        int32_t *len = (int32_t *)(p + L.len);
        for (int64_t s = 0; s < nd; ++s) {
            const float *r = (const float *)(p + L.crec + rec * s);
            int32_t i, l;
            memcpy(&i, r, 4); memcpy(&l, r + 2, 4);
            ret[i] = r[1]; len[i] = l;
            memcpy(tobs + (size_t)i * D, r + 3, (size_t)4 * D);
        }
    }
    if (n_done) *n_done = nd;
    return rc;
}

int tmla_result_block_layout(tmla_env *h, int64_t offsets[6], int64_t *bytes) {
    TMLA_REQUIRE(h && offsets && bytes, "NULL argument");
    const StageLayout L = stage_layout(h->n, kObsDim[h->task]);
    const size_t o[6] = {L.obs, L.rew, L.done, L.trunc, L.flags, L.crec};
    for (int i = 0; i < 6; ++i) offsets[i] = (int64_t)(o[i] - L.obs);
    *bytes = (int64_t)(L.tobs - L.obs);
    return TMLA_OK;
}
int tmla_result_block_alloc(tmla_env *h, void **block) {
    TMLA_REQUIRE(h && block, "NULL argument");
    DeviceGuard guard(h->device);
    const StageLayout L = stage_layout(h->n, kObsDim[h->task]);
    if (cudaMallocHost(block, L.tobs - L.obs) != cudaSuccess) {
        tmla_set_error("cudaMallocHost(result block, %zu bytes): %s", L.tobs - L.obs, cudaGetErrorString(cudaGetLastError()));
        return TMLA_ENOMEM;
    }
    return TMLA_OK;
}
int tmla_result_block_free(void *block) {
    if (block) TMLA_CUDA(cudaFreeHost(block));
    return TMLA_OK;
}

int tmla_host_views(tmla_env *h, int32_t **actions, float **obs, float **reward, uint8_t **done, uint8_t **truncated,
                    float **terminal_obs, float **ep_return, int32_t **ep_length) {
    TMLA_REQUIRE(h, "handle is NULL");
    const StageLayout L = stage_layout(h->n, kObsDim[h->task]);
    char *p = (char *)h->h_stage;
    if (actions) *actions = (int32_t *)(p + L.act);
    if (obs) *obs = (float *)(p + L.obs);
    if (reward) *reward = (float *)(p + L.rew);
    if (done) *done = (uint8_t *)(p + L.done);
    if (truncated) *truncated = (uint8_t *)(p + L.trunc);
    if (terminal_obs) *terminal_obs = (float *)(p + L.tobs);
    if (ep_return) *ep_return = (float *)(p + L.ret);
    if (ep_length) *ep_length = (int32_t *)(p + L.len);
    return TMLA_OK;
}

int tmla_host_records(tmla_env *h, const float **records, int32_t *floats_per_record) {
    TMLA_REQUIRE(h && records && floats_per_record, "NULL argument");
    const StageLayout L = stage_layout(h->n, kObsDim[h->task]);
    *records = (const float *)((char *)h->h_stage + L.crec);
    *floats_per_record = record_words(kObsDim[h->task]);
    return TMLA_OK;
}

int tmla_step_host(tmla_env *h, const int32_t *actions, float *obs, float *reward, uint8_t *done, uint8_t *truncated,
                   float *terminal_obs, float *ep_return, int32_t *ep_length, int64_t *n_done) {
    TMLA_REQUIRE(h, "handle is NULL");
    TMLA_REQUIRE(actions && obs && reward && done && truncated, "actions/obs/reward/done/truncated must be non-NULL");
    const int64_t n = h->n;
    const int D = kObsDim[h->task];
    const StageLayout L = stage_layout(n, D);
    char *p = (char *)h->h_stage;
    { const int rc = tmla_stage_actions(h, actions, 4); if (rc) return rc; }     // range check first: a rejected step changes nothing
    int64_t nd = 0;
    const int rc = step_into_block(h, p + L.obs, &nd);
    if (rc != TMLA_OK && rc != TMLA_EACTION) return rc;
    memcpy(obs, p + L.obs, 4 * n * D);
    memcpy(reward, p + L.rew, 4 * n);
    memcpy(done, p + L.done, n);
    memcpy(truncated, p + L.trunc, n);
    const size_t rec = (size_t)4 * record_words(D);
    for (int64_t s = 0; s < nd; ++s) {   // "written only where done": the records of the finished envs, not three dense arrays
        const float *r = (const float *)(p + L.crec + rec * s);
        int32_t i, l;
        memcpy(&i, r, 4); memcpy(&l, r + 2, 4);
        if (terminal_obs) memcpy(terminal_obs + (size_t)i * D, r + 3, (size_t)4 * D);
        if (ep_return) ep_return[i] = r[1];
        if (ep_length) ep_length[i] = l;
    }
    if (n_done) *n_done = nd;
    return rc;
}

int tmla_reset_host(tmla_env *h, float *obs) {
    TMLA_REQUIRE(h && obs, "handle/obs is NULL");
    DeviceGuard guard(h->device);
    { const int rc = order_after_device_path(h); if (rc) return rc; }
    const size_t bytes = (size_t)4 * h->n * kObsDim[h->task];
    const StageLayout L = stage_layout(h->n, kObsDim[h->task]);
    char *d = (char *)h->d_stage, *p = (char *)h->h_stage;
    int rc = tmla_reset(h, (float *)(d + L.obs), h->own_stream);
    if (rc) return rc;
    TMLA_CUDA(cudaMemcpyAsync(p + L.obs, d + L.obs, bytes, cudaMemcpyDeviceToHost, h->own_stream));
    TMLA_CUDA(cudaStreamSynchronize(h->own_stream));
    if (obs != (float *)(p + L.obs)) memcpy(obs, p + L.obs, bytes);
    return TMLA_OK;
}

int tmla_get_state(tmla_env *h, void *aos, void *stream) {
    TMLA_REQUIRE(h && aos, "handle/aos is NULL");
    DeviceGuard guard(h->device);
    mark_device_path(h, (cudaStream_t)stream);
    TASK_SWITCH(h->task, (get_state_kernel<TaskT><<<grid_for(h->n), kBlock, 0, (cudaStream_t)stream>>>(
                             ptrs_of(h), h->n, (typename TaskT::Wire *)aos)));
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
int tmla_set_state(tmla_env *h, const void *aos, void *stream) {
    TMLA_REQUIRE(h && aos, "handle/aos is NULL");
    DeviceGuard guard(h->device);
    mark_device_path(h, (cudaStream_t)stream);
    TASK_SWITCH(h->task, (set_state_kernel<TaskT><<<grid_for(h->n), kBlock, 0, (cudaStream_t)stream>>>(
                             ptrs_of(h), h->n, (const typename TaskT::Wire *)aos)));
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}
int tmla_check_actions(tmla_env *h, void *stream) {
    TMLA_REQUIRE(h, "handle is NULL");
    DeviceGuard guard(h->device);
    int err = 0;
    TMLA_CUDA(cudaMemcpyAsync(&err, h->err_flag, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    TMLA_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (err) {
        TMLA_CUDA(cudaMemsetAsync(h->err_flag, 0, sizeof(int), (cudaStream_t)stream));
        tmla_set_error("an action outside [0,%d) was passed to step()", kNumActions[h->task]);
        return TMLA_EACTION;
    }
    return TMLA_OK;
}

int tmla_rollout_random(tmla_env *h, int T, float *obs_buf, int32_t *act_buf, float *rew_buf, uint8_t *done_buf, void *stream) {
    TMLA_REQUIRE(h, "handle is NULL");
    TMLA_REQUIRE(T > 0, "T must be positive");
    DeviceGuard guard(h->device);
    mark_device_path(h, (cudaStream_t)stream);
    const int D = kObsDim[h->task];
    const bool fast = obs_buf && act_buf && rew_buf && done_buf && (h->n % kRollBlock == 0) &&
                      ((reinterpret_cast<uintptr_t>(obs_buf) & 15u) == 0) && ((int64_t)T * h->n * D / 4 < ((int64_t)1 << 31));
    const unsigned grid = (unsigned)ceil_div64(h->n, kRollBlock);
    if (fast) {
        TASK_SWITCH(h->task, (rollout_fast_kernel<TaskT><<<grid, kRollBlock, 0, (cudaStream_t)stream>>>(
                                 ptrs_of(h), (uint32_t)h->n, h->seed, h->env_id_base, h->step_count, T,
                                 reinterpret_cast<float4 *>(obs_buf), act_buf, rew_buf, done_buf)));
    } else {
        TASK_SWITCH(h->task, (rollout_random_kernel<TaskT><<<grid, kRollBlock, 0, (cudaStream_t)stream>>>(
                                 ptrs_of(h), h->n, h->seed, h->env_id_base, h->step_count, T, obs_buf, act_buf, rew_buf, done_buf)));
    }
    TMLA_LAUNCH_CHECK();
    h->step_count += (uint64_t)T;
    return TMLA_OK;
}

int tmla_step_policy(tmla_env *h, const float *logits, int deterministic, int32_t row_index, float *obs_next,
                     int32_t *act, float *logp, float *rew, uint8_t *done, int32_t *trunc_count, int32_t *trunc_index,
                     float *trunc_obs, int32_t trunc_capacity, float *ep_stats, const uint64_t *step_base, void *stream) {
    TMLA_REQUIRE(h, "handle is NULL");
    TMLA_REQUIRE(logits && obs_next && rew && done, "logits/obs_next/rew/done must be non-NULL");
    TMLA_REQUIRE(!trunc_count || (trunc_index && trunc_obs && trunc_capacity > 0), "truncation list is incomplete");
    DeviceGuard guard(h->device);
    mark_device_path(h, (cudaStream_t)stream);
    TASK_SWITCH(h->task, (step_policy_kernel<TaskT><<<grid_for(h->n), kBlock, 0, (cudaStream_t)stream>>>(
                             ptrs_of(h), h->n, h->seed, h->env_id_base, h->step_count, step_base, logits, deterministic,
                             (int64_t)row_index, obs_next, act, logp, rew, done, trunc_count, trunc_index, trunc_obs,
                             trunc_capacity, ep_stats, h->ep_log, h->ep_log_cap, h->ep_log_count)));
    TMLA_LAUNCH_CHECK();
    if (!step_base) h->step_count += 1;
    return TMLA_OK;
}

int tmla_selftest_arith(uint64_t *out3, void *stream) {
    TMLA_REQUIRE(out3, "out3 is NULL");
    TMLA_CUDA(cudaMemsetAsync(out3, 0, 3 * sizeof(uint64_t), (cudaStream_t)stream));
    selftest_arith_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>((unsigned long long *)out3);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

int tmla_counter_add(uint64_t *counter, uint64_t n, void *stream) {
    TMLA_REQUIRE(counter, "counter is NULL");
    counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter, n);
    TMLA_LAUNCH_CHECK();
    return TMLA_OK;
}

}  // extern "C"
