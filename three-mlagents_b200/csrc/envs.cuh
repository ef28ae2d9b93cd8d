// envs.cuh — device-side dynamics of the four tasks, one environment per thread, state in registers.
//
// Each task is a struct with the same static interface so the kernels in env_kernels.cu are
// written once and instantiated four times:
//     D, A, MAX_STEPS, NBUF                 observation width, #actions, adapter time limit, #SoA planes
//     State                                 register-resident episode state (+ Monitor accumulator)
//     load / store                          packed structure-of-arrays planes in HBM <-> State
//     from_wire / to_wire                   tmla_<task>_state (include/tmla.h) <-> State
//     observe(State, float o[D])            the task's _get_obs
//     step(State&, a, reward, term, trunc)  env.step + LegacySingleAgentGymAdapter.step flags
//     reset(State&, seed, env_id, k, tag)   env.reset with this repo's Philox streams
//
// Reference being restated (relative to /root/reference/backend), all checked bit-for-bit on the
// CPU side by oracle/envs_oracle.py against reference-made golden traces:
//     basic      mlagents/envs.py:17-84        ball3d     examples/ball3d.py:10-113
//     gridworld  examples/gridworld.py:14-95   push       examples/push.py:10-125
//     walljump   examples/walljump.py:14-98    brickbreak examples/brick_break.py:11-133
//     adapter    mlagents/envs.py:125-152 (steps>=limit -> truncated; terminated = done && !truncated)
#pragma once
#include "common.cuh"
#include "philox.cuh"

// ------------------------------------------------------------------------------------------------
// packed word shared by the three integer tasks: 3-bit cell coordinates, flags, 8-bit step counter
//   bits  0..17 : up to six 3-bit coordinates        bit 18 : goal type (gridworld)
//   bits 19..26 : steps (<= 120)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cell3(uint32_t w, int slot) { return (int)((w >> (3 * slot)) & 7u); }
__device__ __forceinline__ uint32_t put3(int v, int slot) { return ((uint32_t)v & 7u) << (3 * slot); }
__device__ __forceinline__ int iclamp(int v, int lo, int hi) { return min(max(v, lo), hi); }

// Correctly rounded x/3 and x/5 without the generic division sequence (Markstein: q = RN(x*r), e = x - c*q
// exactly by FMA, q' = RN(q + e*r), r = RN(1/c)).  Checked against __fdiv_rn over the whole input range the
// tasks can produce by tmla_selftest_arith (tests/test_envs_gpu.py::test_fast_arithmetic_is_exact).
__device__ __forceinline__ float div3_rn(float x) {
    const float r = 0.333333343267440796f;           // RN(1/3) = 0x3eaaaaab
    const float q = __fmul_rn(x, r);
    return __fmaf_rn(__fmaf_rn(-3.0f, q, x), r, q);
}
__device__ __forceinline__ float div5_rn(float x) {
    const float r = 0.200000002980232239f;           // RN(1/5) = 0x3e4ccccd
    const float q = __fmul_rn(x, r);
    return __fmaf_rn(__fmaf_rn(-5.0f, q, x), r, q);
}
struct NoConsts {};
struct NoSpare {};

// ---------------------------------------------------------------------------- basic (envs.py:17-84)
struct BasicTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 21, A = 3, MAX_STEPS = 50, NBUF = 1;
    typedef tmla_basic_state Wire;
    struct State { int pos, steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int) { return sizeof(uint2); }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        uint2 w = reinterpret_cast<const uint2 *>(buf[0])[i];
        return State{(int)(w.x & 31u), (int)((w.x >> 19) & 255u), __uint_as_float(w.y)};
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        reinterpret_cast<uint2 *>(buf[0])[i] =
            make_uint2((uint32_t)s.pos | ((uint32_t)s.steps << 19), __float_as_uint(s.ep_ret));
    }
    static __device__ State from_wire(const Wire &w) { return State{iclamp(w.pos, 0, 20), w.steps, w.ep_return}; }
    static __device__ Wire to_wire(const State &s) { return Wire{s.pos, s.steps, s.ep_ret}; }

    static __device__ __forceinline__ void observe(const State &s, float *o) {   // position_to_onehot, envs.py:24-27
#pragma unroll
        for (int j = 0; j < D; ++j) o[j] = (j == s.pos) ? 1.0f : 0.0f;
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        s.pos = iclamp(s.pos + a - 1, 0, 20);            // envs.py:61-62
        s.steps += 1;
        // envs.py:65-72: -0.01 (+0.1 | +1.0) evaluated in double, rounded once to f32
        const bool small = s.pos == 7, large = s.pos == 17;
        reward = __uint_as_float(small ? 0x3DB851ECu : (large ? 0x3F7D70A4u : 0xBC23D70Au));
        term = small || large;
        trunc = (s.steps >= MAX_STEPS) && !term;         // envs.py:74
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t, uint64_t, uint64_t, uint32_t) {
        s.pos = 10; s.steps = 0; s.ep_ret = 0.0f;        // envs.py:21,55-57 (no randomness)
    }
};

// ------------------------------------------------------------------ ball3d (examples/ball3d.py:10-113)
// Double-precision constants live in constant memory so that DFMA/DMUL/DADD take them as c[bank][offset]
// operands (64-bit literals cannot be encoded as immediates and would cost a UMOV pair each).
struct Ball3DConst {
    double max_tilt, tilt_delta, g, dt, half_lo;      // np.deg2rad(25), np.deg2rad(3), 9.81, 0.02, -max_tilt/2
    double s15, s13, s11, s9, s7, s5, s3;            // sin Taylor coefficients -1/15! ... -1/3!
    double inv32;                                    // 2^-32
};
#define TMLA_B3_INIT { \
    0x1.becde5da115a9p-2, 0x1.acee9f37bebd6p-5, 9.81, 0.02, -0x1.becde5da115a9p-3, \
    -7.6471637318198164759e-13, 1.6059043836821614599e-10, -2.5052108385441718775e-08, 2.7557319223985890653e-06, \
    -1.9841269841269841253e-04, 8.3333333333333332177e-03, -1.6666666666666665741e-01, 0x1p-32}
__device__ const Ball3DConst gB3 = TMLA_B3_INIT;      // same values in global memory (register-pinned loads)
__device__ __constant__ Ball3DConst kB3 = {
    0x1.becde5da115a9p-2, 0x1.acee9f37bebd6p-5, 9.81, 0.02, -0x1.becde5da115a9p-3,
    -7.6471637318198164759e-13, 1.6059043836821614599e-10, -2.5052108385441718775e-08, 2.7557319223985890653e-06,
    -1.9841269841269841253e-04, 8.3333333333333332177e-03, -1.6666666666666665741e-01,
    0x1p-32};

// sin on |x| <= MAX_TILT = 0.43633: odd Taylor/Horner through x^15, no range reduction.
// Truncation error < 2.2e-21 (x^17/17!), evaluation error ~0.6 ulp: agrees with libm's double sin to
// the last bit in the vast majority of cases; parity with the reference is tolerance-checked.
__device__ __forceinline__ double sin_small(double x) {
    const double z = x * x, z2 = z * z, z4 = z2 * z2;      // Estrin, identical to Ball3DTask::sin_small_c
    const double a = fma(kB3.s5, z, kB3.s3), b = fma(kB3.s9, z, kB3.s7), cc = fma(kB3.s13, z, kB3.s11);
    const double ab = fma(b, z2, a), cd = fma(kB3.s15, z2, cc);
    return fma(x * z, fma(cd, z4, ab), x);
}
// np.clip(x, -m, m) for finite x
__device__ __forceinline__ double clip_sym(double x, double m) { return fabs(x) > m ? copysign(m, x) : x; }
// uniform double in (0,1) with 32 random bits: (w + 0.5) * 2^-32 (exact)
__device__ __forceinline__ double u32_to_unit(uint32_t w) { return ((double)w + 0.5) * kB3.inv32; }

struct Ball3DTask {
    static constexpr int D = 6, A = 5, MAX_STEPS = 200, NBUF = 3;
    typedef tmla_ball3d_state Wire;
    // loop-invariant double constants pinned in registers (the asm barrier stops the compiler from
    // re-loading them from the constant bank on every iteration of the fused rollout loop)
    struct Consts { double max_tilt, tilt_delta, g, dt, s15, s13, s11, s9, s7, s5, s3; };
    static __device__ __forceinline__ double pinned(const double *p) {   // a load ptxas cannot rematerialise
        double v;
        asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ Consts load_consts() {
        const Ball3DConst *g = &gB3;
        return Consts{pinned(&g->max_tilt), pinned(&g->tilt_delta), pinned(&g->g), pinned(&g->dt), pinned(&g->s15),
                      pinned(&g->s13), pinned(&g->s11), pinned(&g->s9), pinned(&g->s7), pinned(&g->s5), pinned(&g->s3)};
    }
    static __device__ __forceinline__ double sin_small_c(const Consts &c, double x) {
        // Estrin evaluation of the same degree-15 odd polynomial: dependency depth 5 instead of 8
        const double z = x * x, z2 = z * z, z4 = z2 * z2;
        const double a = fma(c.s5, z, c.s3), b = fma(c.s9, z, c.s7), cc = fma(c.s13, z, c.s11);
        const double ab = fma(b, z2, a), cd = fma(c.s15, z2, cc);
        return fma(x * z, fma(cd, z4, ab), x);
    }
    // rx/rz change only when an action tilts THAT axis (at most one per step), so G*sin(rot)*DT and the f32 observation of
    // each axis are cached in the state and only the tilted axis is re-evaluated: one sin polynomial per step instead of two.
    // Bit-identical by construction (the cached value is what the reference recomputes from an unchanged rot).
    struct State { double rx, rz; float px, pz, vx, vz; int steps; float ep_ret; uint32_t episode; double axdt, azdt; float orx, orz; };
    static __device__ __forceinline__ void refresh(State &s) {              // caches from rx/rz (load, state injection, reset)
        s.axdt = __dmul_rn(__dmul_rn(kB3.g, sin_small(s.rx)), kB3.dt);       // ball3d.py:81-84: (G*sin(rot))*DT
        s.azdt = __dmul_rn(__dmul_rn(kB3.g, sin_small(s.rz)), kB3.dt);
        s.orx = __double2float_rn(s.rx); s.orz = __double2float_rn(s.rz);
    }
    static __host__ __device__ size_t plane_bytes(int b) { return b == 0 ? sizeof(double2) : (b == 1 ? sizeof(float4) : sizeof(int2)); }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        const double2 r = reinterpret_cast<const double2 *>(buf[0])[i];     // 128-bit
        const float4 pv = reinterpret_cast<const float4 *>(buf[1])[i];      // 128-bit
        const int2 m = reinterpret_cast<const int2 *>(buf[2])[i];
        State s{r.x, r.y, pv.x, pv.y, pv.z, pv.w, m.x & 255, __int_as_float(m.y), (uint32_t)m.x >> 8, 0.0, 0.0, 0.0f, 0.0f};   // steps | episode<<8
        refresh(s);
        return s;
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        reinterpret_cast<double2 *>(buf[0])[i] = make_double2(s.rx, s.rz);
        reinterpret_cast<float4 *>(buf[1])[i] = make_float4(s.px, s.pz, s.vx, s.vz);
        reinterpret_cast<int2 *>(buf[2])[i] = make_int2((int)((uint32_t)s.steps | (s.episode << 8)), __float_as_int(s.ep_ret));
    }
    static __device__ State from_wire(const Wire &w) {
        return State{w.rot[0], w.rot[1], w.pos[0], w.pos[1], w.vel[0], w.vel[1], w.steps, w.ep_return, (uint32_t)w.episode & 0xFFFFFFu,
                     0.0, 0.0, 0.0f, 0.0f};                                    // caches are rebuilt by load()
    }
    static __device__ Wire to_wire(const State &s) {
        Wire w; w.rot[0] = s.rx; w.rot[1] = s.rz; w.pos[0] = s.px; w.pos[1] = s.pz;
        w.vel[0] = s.vx; w.vel[1] = s.vz; w.steps = s.steps; w.ep_return = s.ep_ret; w.episode = (int32_t)s.episode; w.pad_ = 0; return w;
    }
    static __device__ __forceinline__ void observe(const State &s, float *o) {   // ball3d.py:61-72
        o[0] = s.orx; o[1] = s.orz;
        o[2] = s.px; o[3] = s.pz; o[4] = s.vx; o[5] = s.vz;
    }
    struct Pending { float sq; uint32_t flags; };
    // The tilt half of a step (ball3d.py:76-84): the new rotation of the ONE axis action `a` touches, with the products that
    // depend on it.  It reads only rx/rz (and, right after a reset, `steps == 0`), never pos/vel.
    struct Tilt { double rot, adt; float orot; bool x; };
    template <bool MAYBE_FIRST>
    static __device__ __forceinline__ Tilt plan(const Consts &c, const State &s, int a) {
        // ACTION_DELTAS (ball3d.py:31-37): 0:+x 1:-x 2:+z 3:-z 4:none, each +-np.deg2rad(3.0).  The sign is
        // XOR-ed into the high word; adding the 0.0 entries is the identity (rot is never -0.0) and is skipped.
        const int td_hi = __double2hiint(c.tilt_delta), td_lo = __double2loint(c.tilt_delta);
        // a odd -> -delta; action 4 adds (0, 0): it runs through the z axis with a zero delta (rot + 0, the clip and the f32
        // round trip of an f32 value are identities, the cached products are recomputed to the same bits) — no divergent branch
        const double sd = __hiloint2double(a < 4 ? td_hi ^ (int)((unsigned)a << 31) : 0, a < 4 ? td_lo : 0);
        Tilt tl;
        tl.x = a < 2;
        double rot = __dadd_rn(tl.x ? s.rx : s.rz, sd);                              // ball3d.py:77
        if (MAYBE_FIRST && s.steps == 0) {   // first step after reset(): rot is still the float32 array, `+=` casts back (the
            asm volatile("");     // untouched axis is already an f32 value); kept a branch: conversions for <1 % of the lanes
            rot = (double)__double2float_rn(rot);
        }
        rot = clip_sym(rot, c.max_tilt);                                             // ball3d.py:78 (float64 from here)
        tl.rot = rot;
        tl.adt = __dmul_rn(__dmul_rn(c.g, sin_small_c(c, rot)), c.dt);               // ball3d.py:81-84
        tl.orot = __double2float_rn(rot);
        return tl;
    }
    // the rest of the step: apply the planned tilt, integrate velocity and position, flags
    static __device__ __forceinline__ void advance_planned(const Consts &, State &s, const Tilt &tl, Pending &pend, bool &term, bool &trunc) {
        if (tl.x) { s.rx = tl.rot; s.axdt = tl.adt; s.orx = tl.orot; } else { s.rz = tl.rot; s.azdt = tl.adt; s.orz = tl.orot; }
        float vx = __double2float_rn(__dadd_rn((double)s.vx, s.axdt));              // ball3d.py:83-84
        float vz = __double2float_rn(__dadd_rn((double)s.vz, s.azdt));
        vx = __fmul_rn(vx, 0.98f);                                                  // ball3d.py:87
        vz = __fmul_rn(vz, 0.98f);
        const float px = __fadd_rn(s.px, __fmul_rn(vx, 0.02f));                     // ball3d.py:90
        const float pz = __fadd_rn(s.pz, __fmul_rn(vz, 0.02f));
        s.vx = vx; s.vz = vz; s.px = px; s.pz = pz;
        s.steps += 1;
        const bool off = (fabsf(px) > 3.0f) || (fabsf(pz) > 3.0f);                  // ball3d.py:96-98
        const bool timeout = s.steps >= 200;                                        // ball3d.py:99
        const bool done = off || timeout;
        pend.sq = __fadd_rn(__fmul_rn(px, px), __fmul_rn(pz, pz));                  // np.linalg.norm: x.dot(x) in f32
        pend.flags = (done ? 1u : 0u) | ((timeout && !off) ? 2u : 0u);
        trunc = s.steps >= MAX_STEPS;                                               // envs.py:141-145
        term = done && !trunc;
    }
    // NumPy-2 promotion makes this a mixed f64/f32 computation (SURVEY.md A2); every rounding is explicit (`__*_rn` never
    // contracts into FMA) so the result does not depend on compiler flags.
    static __device__ __forceinline__ void advance(const Consts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        const Tilt tl = plan<true>(c, s, a);
        advance_planned(c, s, tl, pend, term, trunc);
    }
    // second half of step(): the reward (ball3d.py:103-111).  It depends only on `Pending`, so the fused rollout
    // kernel evaluates it one iteration late, interleaved with the next step's physics (more ILP per warp).
    static __device__ __forceinline__ float finish(const Pending &pend) {
        const float d = __fsqrt_rn(pend.sq);
        float r = __fsub_rn(1.0f, div3_rn(d));                                      // ball3d.py:104 (IEEE d/3)
        if (pend.flags & 1u) r = (pend.flags & 2u) ? 1.0f : -1.0f;                  // ball3d.py:105-108
        return __fadd_rn(r, __fmul_rn(-0.02f, d));                                  // ball3d.py:110-111
    }
    static __device__ __forceinline__ void step(const Consts &c, State &s, int a, float &reward, bool &term, bool &trunc) {
        Pending pend;
        advance(c, s, a, pend, term, trunc);
        reward = finish(pend);
    }
    // Initial state of an episode.  np.random.uniform(lo, hi) = lo + (hi-lo)*u (ball3d.py:49-57) then
    // `.astype(np.float32)`; u carries 32 random bits (the reference's 53-bit double is rounded to 24 bits
    // anyway).  AUTO-RESET draws are indexed by the env's own episode counter (ctr = episode index, tag
    // TAG_RESET), not by the global step, so the fused rollout kernel can draw the next initial state ahead
    // of time, off the critical path (`Spare`); VecEnv.reset() draws use (global step, TAG_RESET_ALL).
    // A spare also carries the cached products of its rotation (G*sin(rot)*DT per axis): they are evaluated when the spare is
    // DRAWN — off the critical path, every kSpareEvery steps — so that the reset branch, which ~23 % of the warps of the fused
    // rollout enter on every step, is a handful of register moves instead of two sin polynomials.  Same expressions as refresh().
    struct Spare { float rx, rz, px, pz, vx, vz; double axdt, azdt; };
    static constexpr bool HAS_SPARE = true;
    static __device__ __forceinline__ Spare draw(uint64_t seed, uint64_t env_id, uint64_t counter, uint32_t tag) {
        const uint4 b0 = tmla_stream_block(seed, env_id, counter, tag, 0);
        const uint4 b1 = tmla_stream_block(seed, env_id, counter, tag, 1);
        const double mt = kB3.max_tilt, lo = kB3.half_lo;
        Spare sp;
        sp.rx = __double2float_rn(__dadd_rn(lo, __dmul_rn(mt, u32_to_unit(b0.x))));
        sp.rz = __double2float_rn(__dadd_rn(lo, __dmul_rn(mt, u32_to_unit(b0.y))));
        sp.px = __double2float_rn(__dadd_rn(-1.5, __dmul_rn(3.0, u32_to_unit(b0.z))));
        sp.pz = __double2float_rn(__dadd_rn(-1.5, __dmul_rn(3.0, u32_to_unit(b0.w))));
        sp.vx = __double2float_rn(__dadd_rn(-1.0, __dmul_rn(2.0, u32_to_unit(b1.x))));
        sp.vz = __double2float_rn(__dadd_rn(-1.0, __dmul_rn(2.0, u32_to_unit(b1.y))));
        sp.axdt = __dmul_rn(__dmul_rn(kB3.g, sin_small((double)sp.rx)), kB3.dt);      // = refresh() on the state begin_episode builds
        sp.azdt = __dmul_rn(__dmul_rn(kB3.g, sin_small((double)sp.rz)), kB3.dt);
        return sp;
    }
    static __device__ __forceinline__ void begin_episode(State &s, const Spare &sp, uint32_t episode) {
        s.rx = (double)sp.rx; s.rz = (double)sp.rz; s.px = sp.px; s.pz = sp.pz; s.vx = sp.vx; s.vz = sp.vz;
        s.steps = 0; s.ep_ret = 0.0f; s.episode = episode;
        s.axdt = sp.axdt; s.azdt = sp.azdt;                 // refresh(s), with the products taken from the spare:
        s.orx = sp.rx; s.orz = sp.rz;                       // f32(f64(f32 x)) == x
    }
    static __device__ __forceinline__ uint32_t next_episode(const State &s) { return (s.episode + 1u) & 0xFFFFFFu; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        if (tag == TMLA_TAG_RESET) {
            const uint32_t e = next_episode(s);
            begin_episode(s, draw(seed, env_id, e, TMLA_TAG_RESET), e);
        } else {
            begin_episode(s, draw(seed, env_id, k, tag), 0u);
        }
    }
};

// shared move table of gridworld.py:19-25 and push.py:14-20: 0 stay, 1 (0,+1), 2 (0,-1), 3 (-1,0), 4 (+1,0)
__device__ __forceinline__ void grid_delta(int a, int &dx, int &dy) {
    dx = (a == 4) - (a == 3);
    dy = (a == 1) - (a == 2);
}

// ------------------------------------------------------------- gridworld (examples/gridworld.py:14-95)
struct GridWorldTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 4, A = 5, MAX_STEPS = 100, NBUF = 1;
    typedef tmla_gridworld_state Wire;
    struct State { int ax, ay, gx, gy, rx, ry, type, steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int) { return sizeof(uint2); }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        const uint2 w = reinterpret_cast<const uint2 *>(buf[0])[i];
        return State{cell3(w.x, 0), cell3(w.x, 1), cell3(w.x, 2), cell3(w.x, 3), cell3(w.x, 4), cell3(w.x, 5),
                     (int)((w.x >> 18) & 1u), (int)((w.x >> 19) & 255u), __uint_as_float(w.y)};
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        const uint32_t w = put3(s.ax, 0) | put3(s.ay, 1) | put3(s.gx, 2) | put3(s.gy, 3) | put3(s.rx, 4) |
                           put3(s.ry, 5) | ((uint32_t)s.type << 18) | ((uint32_t)s.steps << 19);
        reinterpret_cast<uint2 *>(buf[0])[i] = make_uint2(w, __float_as_uint(s.ep_ret));
    }
    static __device__ State from_wire(const Wire &w) {
        return State{w.agent[0], w.agent[1], w.green[0], w.green[1], w.red[0], w.red[1], w.goal_type & 1, w.steps, w.ep_return};
    }
    static __device__ Wire to_wire(const State &s) {
        Wire w; w.agent[0] = s.ax; w.agent[1] = s.ay; w.green[0] = s.gx; w.green[1] = s.gy;
        w.red[0] = s.rx; w.red[1] = s.ry; w.goal_type = s.type; w.steps = s.steps; w.ep_return = s.ep_ret; return w;
    }
    static __device__ __forceinline__ void observe(const State &s, float *o) {   // gridworld.py:55-64
        const int tx = s.type ? s.rx : s.gx, ty = s.type ? s.ry : s.gy;
        o[0] = (float)(tx - s.ax) * 0.25f;      // k/4 is exact in f32
        o[1] = (float)(ty - s.ay) * 0.25f;
        o[2] = s.type ? 0.0f : 1.0f;
        o[3] = s.type ? 1.0f : 0.0f;
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        int dx, dy; grid_delta(a, dx, dy);
        s.ax = iclamp(s.ax + dx, 0, 4);                                  // gridworld.py:68-71
        s.ay = iclamp(s.ay + dy, 0, 4);
        s.steps += 1;
        const bool on_green = (s.ax == s.gx) && (s.ay == s.gy);          // gridworld.py:79-90 (if / elif)
        const bool on_red = !on_green && (s.ax == s.rx) && (s.ay == s.ry);
        reward = __uint_as_float(0xBC23D70Au);                           // f32(-0.01)
        if (on_green) reward = (s.type == 0) ? 1.0f : -1.0f;
        if (on_red) reward = (s.type == 1) ? 1.0f : -1.0f;
        const bool done = on_green || on_red || (s.steps >= 100);        // gridworld.py:92-93
        trunc = s.steps >= MAX_STEPS;                                    // envs.py:141-145
        term = done && !trunc;
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        // np.random.shuffle(cells)[:3] = uniform ordered triple of distinct cells; np.random.choice([0,1])
        const uint4 b = tmla_stream_block(seed, env_id, k, tag, 0);      // gridworld.py:42-50
        const int a = tmla_bounded(b.x, 25);
        int g = tmla_bounded(b.y, 24); g += (g >= a);
        int r = tmla_bounded(b.z, 23);
        const int lo = min(a, g), hi = max(a, g);
        r += (r >= lo); r += (r >= hi);
        s.ax = a / 5; s.ay = a % 5; s.gx = g / 5; s.gy = g % 5; s.rx = r / 5; s.ry = r % 5;
        s.type = (int)(b.w >> 31);
        s.steps = 0; s.ep_ret = 0.0f;
    }
};

// ---------------------------------------------------------------------- push (examples/push.py:10-125)
// 18-entry reward table [(d_ab+1)*6 + (d_bg+1)*2 + invalid]: the reference evaluates
// -0.01 + 0.05*d_ab + 0.3*d_bg (- 0.05) in Python doubles (push.py:77,111-115) and SB3 stores f32;
// float32 arithmetic is 1-2 ulp off in 10 of 18 cases, so the f32(double) values are tabulated
// (same table built at run time by oracle/envs_oracle.py:push_reward_lut and compared in tests).
__device__ __constant__ uint32_t kPushRewardBits[18] = {
    0xbeb851ecu, 0xbed1eb85u, 0xbd75c28fu, 0xbde147aeu, 0x3e75c28fu, 0x3e428f5cu,
    0xbe9eb852u, 0xbeb851ecu, 0xbc23d70au, 0xbd75c28fu, 0x3e947ae1u, 0x3e75c28fu,
    0xbe851eb8u, 0xbe9eb852u, 0x3d23d70au, 0xbc23d70au, 0x3eae147bu, 0x3e947ae1u};

struct PushTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 4, A = 5, MAX_STEPS = 120, NBUF = 1;
    typedef tmla_push_state Wire;
    struct State { int ax, ay, bx, by, goal_x, steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int) { return sizeof(uint2); }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        const uint2 w = reinterpret_cast<const uint2 *>(buf[0])[i];
        return State{cell3(w.x, 0), cell3(w.x, 1), cell3(w.x, 2), cell3(w.x, 3), cell3(w.x, 4),
                     (int)((w.x >> 19) & 255u), __uint_as_float(w.y)};
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        const uint32_t w = put3(s.ax, 0) | put3(s.ay, 1) | put3(s.bx, 2) | put3(s.by, 3) | put3(s.goal_x, 4) |
                           ((uint32_t)s.steps << 19);
        reinterpret_cast<uint2 *>(buf[0])[i] = make_uint2(w, __float_as_uint(s.ep_ret));
    }
    static __device__ State from_wire(const Wire &w) {
        return State{w.agent[0], w.agent[1], w.box[0], w.box[1], w.goal_x, w.steps, w.ep_return};
    }
    static __device__ Wire to_wire(const State &s) {
        Wire w; w.agent[0] = s.ax; w.agent[1] = s.ay; w.box[0] = s.bx; w.box[1] = s.by;
        w.goal_x = s.goal_x; w.steps = s.steps; w.ep_return = s.ep_ret; return w;
    }
    static __device__ __forceinline__ void observe(const State &s, float *o) {   // push.py:53-59
        // f32(k/5.0) == f32(k)/f32(5) for |k| <= 5 (checked in tests); correctly rounded division
        o[0] = div5_rn((float)(s.bx - s.ax));
        o[1] = div5_rn((float)(s.by - s.ay));
        o[2] = div5_rn((float)(s.goal_x - s.bx));
        o[3] = div5_rn((float)(5 - s.by));
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        int dx, dy; grid_delta(a, dx, dy);
        int nax = iclamp(s.ax + dx, 0, 5), nay = iclamp(s.ay + dy, 0, 5);          // push.py:63-65
        const int prev_bg = abs(s.goal_x - s.bx) + abs(5 - s.by);                  // push.py:70-75
        const int prev_ab = abs(s.bx - s.ax) + abs(s.by - s.ay);
        int nbx = s.bx, nby = s.by;
        bool invalid = false;
        if (nax == s.bx && nay == s.by) {                                          // push.py:83-95
            const int tx = s.bx + dx, ty = s.by + dy;
            if (tx >= 0 && tx < 6 && ty >= 0 && ty < 6) { nbx = tx; nby = ty; }
            else { nax = s.ax; nay = s.ay; invalid = true; }
        }
        s.ax = nax; s.ay = nay; s.bx = nbx; s.by = nby;
        s.steps += 1;
        const int dist_bg = abs(s.goal_x - nbx) + abs(5 - nby);                    // push.py:103-108
        const int dist_ab = abs(nbx - nax) + abs(nby - nay);
        const int idx = (prev_ab - dist_ab + 1) * 6 + (prev_bg - dist_bg + 1) * 2 + (invalid ? 1 : 0);
        reward = __uint_as_float(kPushRewardBits[idx]);                            // push.py:77,111-115
        const bool top = nby == 5;                                                 // push.py:118-120
        if (top) reward = 1.0f;
        const bool done = top || (s.steps >= 120);                                 // push.py:122-123
        trunc = s.steps >= MAX_STEPS;                                              // envs.py:141-145
        term = done && !trunc;
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        const uint4 b = tmla_stream_block(seed, env_id, k, tag, 0);                // push.py:40-47
        const int a = tmla_bounded(b.x, 36);
        int bx = tmla_bounded(b.y, 35); bx += (bx >= a);
        s.ax = a / 6; s.ay = a % 6; s.bx = bx / 6; s.by = bx % 6;
        s.goal_x = tmla_bounded(b.z, 6);
        s.steps = 0; s.ep_ret = 0.0f;
    }
};

// ------------------------------------------------------------ walljump (examples/walljump.py:14-98)
// 1-D track of 20 cells, a wall at x = 10 present with probability 0.7, a jump lasts 3 steps.  Integer state;
// the rewards are the Python doubles -0.01, -0.01-0.02, -0.01-0.03 and 1.0 rounded once to f32
// (0xbc23d70a, 0xbcf5c28f, 0xbd23d70a; the golden traces hold exactly these four values).
struct WallJumpTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 4, A = 4, MAX_STEPS = 150, NBUF = 1, WIDTH = 20, WALL_X = 10, JUMP = 3;
    typedef tmla_walljump_state Wire;
    struct State { int x, in_air, wall, steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int) { return sizeof(uint2); }

    // packed word: x bits 0..4 | in_air bits 5..6 | wall bit 7 | steps bits 19..26
    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        const uint2 w = reinterpret_cast<const uint2 *>(buf[0])[i];
        return State{(int)(w.x & 31u), (int)((w.x >> 5) & 3u), (int)((w.x >> 7) & 1u), (int)((w.x >> 19) & 255u), __uint_as_float(w.y)};
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        const uint32_t w = (uint32_t)s.x | ((uint32_t)s.in_air << 5) | ((uint32_t)s.wall << 7) | ((uint32_t)s.steps << 19);
        reinterpret_cast<uint2 *>(buf[0])[i] = make_uint2(w, __float_as_uint(s.ep_ret));
    }
    static __device__ State from_wire(const Wire &w) {
        return State{iclamp(w.agent_x, 0, WIDTH - 1), iclamp(w.in_air, 0, JUMP), w.wall & 1, w.steps, w.ep_return};
    }
    static __device__ Wire to_wire(const State &s) { return Wire{s.x, s.in_air, s.wall, s.steps, s.ep_ret}; }

    static __device__ __forceinline__ void observe(const State &s, float *o) {   // walljump.py:48-53
        // f32(k/19.0) == f32(k)/f32(19) for every reachable k in [-9,19] (tests/test_oracle_cpu.py); IEEE f32 division
        o[0] = __fdiv_rn((float)(WIDTH - 1 - s.x), 19.0f);
        o[1] = __fdiv_rn((float)(WALL_X - s.x), 19.0f);
        o[2] = (float)s.wall;
        o[3] = s.in_air == 0 ? 1.0f : 0.0f;
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        bool just_jumped = false;
        if (a == 3 && s.in_air == 0) { s.in_air = JUMP; just_jumped = true; }       // walljump.py:62-65
        const int dx = (a == 1 || a == 3) ? 1 : (a == 2 ? -1 : 0);                  // ACTION_DELTAS, walljump.py:18
        int px = iclamp(s.x + dx, 0, WIDTH - 1);                                    // walljump.py:68-69
        const bool crossing = (s.x < WALL_X && WALL_X <= px) || (px < WALL_X && WALL_X <= s.x);   // walljump.py:72-74
        uint32_t rbits = 0xBC23D70Au;                                               // f32(-0.01)
        if (crossing && s.wall == 1 && s.in_air == 0) { px = s.x; rbits = 0xBCF5C28Fu; }          // walljump.py:75-77: -0.01 - 0.02
        if (just_jumped && !crossing && abs(WALL_X - s.x) > 1) rbits = 0xBD23D70Au;                // walljump.py:80-81: -0.01 - 0.03
        s.x = px;
        if (s.in_air > 0) s.in_air -= 1;                                            // walljump.py:86-87
        bool done = false;
        if (s.x == WIDTH - 1) { rbits = 0x3F800000u; done = true; }                 // walljump.py:90-92
        s.steps += 1;
        done = done || (s.steps >= 150);                                            // walljump.py:94-96
        reward = __uint_as_float(rbits);
        trunc = s.steps >= MAX_STEPS;                                               // envs.py:141-145
        term = done && !trunc;
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        const uint4 b = tmla_stream_block(seed, env_id, k, tag, 0);                 // walljump.py:39-45
        s.x = 0; s.in_air = 0;
        s.wall = tmla_u24(b.x) < 0.7f ? 1 : 0;                                      // int(np.random.rand() < 0.7)
        s.steps = 0; s.ep_ret = 0.0f;
    }
};

// ------------------------------------------------------- brickbreak (examples/brick_break.py:11-133)
// 40x40 court, 8-wide paddle, 5x8 bricks of 5x2 at y = 20..30; the whole state is float64 in the reference (NumPy arrays and
// Python floats), so every operation below is an explicit f64 add/mul/div in the reference's order (no FMA contraction).
// The serve angle uses a fixed Horner polynomial for sin/cos (plain mul/add), the same sequence as
// oracle/envs_oracle.py:sin_cos_quarter, so that oracle and device resets agree bit for bit.
// sin/cos on [-pi/4, pi/4] as fixed Horner polynomials in plain f64 mul/add (no fma, no libm): reset draws that need an
// angle use this on the device and in the oracle (oracle/envs_oracle.py:sin_cos_quarter), so the two agree bit for bit.
static __device__ __forceinline__ void sin_cos_quarter(double y, double &sn, double &cs) {
    const double z = __dmul_rn(y, y);
    double ps = -1.0 / 1307674368000.0, pc = 1.0 / 20922789888000.0;
    const double sc[6] = {1.0 / 6227020800.0, -1.0 / 39916800.0, 1.0 / 362880.0, -1.0 / 5040.0, 1.0 / 120.0, -1.0 / 6.0};
    const double cc[7] = {-1.0 / 87178291200.0, 1.0 / 479001600.0, -1.0 / 3628800.0, 1.0 / 40320.0, -1.0 / 720.0, 1.0 / 24.0, -1.0 / 2.0};
#pragma unroll
    for (int j = 0; j < 6; ++j) ps = __dadd_rn(__dmul_rn(ps, z), sc[j]);
#pragma unroll
    for (int j = 0; j < 7; ++j) pc = __dadd_rn(__dmul_rn(pc, z), cc[j]);
    sn = __dadd_rn(y, __dmul_rn(__dmul_rn(y, z), ps));
    cs = __dadd_rn(1.0, __dmul_rn(z, pc));
}

struct BrickBreakTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 45, A = 3, MAX_STEPS = 2000, NBUF = 4;
    typedef tmla_brickbreak_state Wire;
    struct State { double px, py, vx, vy, paddle; unsigned long long bricks; int steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int b) { return b < 3 ? 16 : sizeof(int2); }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        const double2 p = reinterpret_cast<const double2 *>(buf[0])[i], v = reinterpret_cast<const double2 *>(buf[1])[i];
        const double2 pb = reinterpret_cast<const double2 *>(buf[2])[i];      // paddle | bricks bit mask
        const int2 m = reinterpret_cast<const int2 *>(buf[3])[i];
        return State{p.x, p.y, v.x, v.y, pb.x, (unsigned long long)__double_as_longlong(pb.y), m.x, __int_as_float(m.y)};
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        reinterpret_cast<double2 *>(buf[0])[i] = make_double2(s.px, s.py);
        reinterpret_cast<double2 *>(buf[1])[i] = make_double2(s.vx, s.vy);
        reinterpret_cast<double2 *>(buf[2])[i] = make_double2(s.paddle, __longlong_as_double((long long)s.bricks));
        reinterpret_cast<int2 *>(buf[3])[i] = make_int2(s.steps, __float_as_int(s.ep_ret));
    }
    static __device__ State from_wire(const Wire &w) {
        unsigned long long m = 0;
        for (int b = 0; b < 40; ++b) m |= (unsigned long long)(w.bricks[b] ? 1 : 0) << b;
        return State{w.pos[0], w.pos[1], w.vel[0], w.vel[1], w.paddle, m, w.steps, w.ep_return};
    }
    static __device__ Wire to_wire(const State &s) {
        Wire w; w.pos[0] = s.px; w.pos[1] = s.py; w.vel[0] = s.vx; w.vel[1] = s.vy; w.paddle = s.paddle;
        for (int b = 0; b < 40; ++b) w.bricks[b] = (uint8_t)((s.bricks >> b) & 1ull);
        w.steps = s.steps; w.ep_return = s.ep_ret; return w;
    }
    static __device__ __forceinline__ void observe(const State &s, float *o) {   // brick_break.py:118-126, cast envs.py:150
        o[0] = __double2float_rn(__ddiv_rn(s.px, 40.0));
        o[1] = __double2float_rn(__ddiv_rn(s.py, 40.0));
        o[2] = __double2float_rn(s.vx);
        o[3] = __double2float_rn(s.vy);
        o[4] = __double2float_rn(__ddiv_rn(s.paddle, 40.0));
#pragma unroll
        for (int b = 0; b < 40; ++b) o[5 + b] = (float)((s.bricks >> b) & 1ull);
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        double paddle = __dadd_rn(s.paddle, a == 0 ? -3.0 : (a == 2 ? 3.0 : 0.0));        // brick_break.py:51-54
        paddle = fmin(fmax(paddle, 4.0), 36.0);                                            // :56-58
        const double px = __dadd_rn(s.px, s.vx), py = __dadd_rn(s.py, s.vy);               // :61
        double vx = s.vx, vy = s.vy;
        if (px <= 1.0 || px >= 39.0) vx = -vx;                                             // :67-73
        if (py >= 39.0) vy = -vy;
        double r = 0.0;
        if (vy < 0.0 && __dsub_rn(py, 1.0) <= 2.0 && px >= __dsub_rn(paddle, 4.0) && px <= __dadd_rn(paddle, 4.0)) {   // :76-86
            vy = -vy;
            const double offset = __ddiv_rn(__dsub_rn(px, paddle), 4.0);
            vx = __dadd_rn(vx, __dmul_rn(offset, 0.5));
            r = 0.1;
        }
        unsigned long long bricks = s.bricks;
        if (py >= 20.0 && py <= 30.0) {                                                    // :88-105 (rows span y = 20 .. 30)
            bool found = false;
#pragma unroll 1
            for (int row = 0; row < 5 && !found; ++row) {
                const double by = 20.0 + 2.0 * row;
                if (!(py >= by && py <= by + 2.0)) continue;
#pragma unroll 1
                for (int c = 0; c < 8; ++c) {
                    const double bx = 5.0 * c;
                    if (((bricks >> (row * 8 + c)) & 1ull) && px >= bx && px <= bx + 5.0) {
                        bricks &= ~(1ull << (row * 8 + c));
                        vy = -vy;
                        r = 1.0;
                        found = true;
                        break;
                    }
                }
            }
        }
        bool done = false;
        if (py < 1.0) { r = -1.0; done = true; }                                           // :109-111
        if (bricks == 0ull) { r = 10.0; done = true; }                                     // :113-115
        s.px = px; s.py = py; s.vx = vx; s.vy = vy; s.paddle = paddle; s.bricks = bricks;
        s.steps += 1;
        if (s.steps > 2000) done = true;                                                   // :117-118
        reward = __double2float_rn(r);
        trunc = s.steps >= MAX_STEPS;                                                      // envs.py:141-145
        term = done && !trunc;
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        const uint4 b = tmla_stream_block(seed, env_id, k, tag, 0);                        // brick_break.py:39-46
        const double angle = __dadd_rn(0.78539816339744830962, __dmul_rn(1.57079632679489661923, u32_to_unit(b.x)));
        double sn, cs;
        sin_cos_quarter(__dsub_rn(angle, 1.57079632679489661923), sn, cs);
        s.px = 20.0; s.py = 10.0;
        s.vx = __dmul_rn(-sn, 1.5); s.vy = __dmul_rn(cs, 1.5);                             // cos(angle) = -sin(y), sin(angle) = cos(y)
        s.paddle = 20.0;
        s.bricks = (1ull << 40) - 1ull;
        s.steps = 0; s.ep_ret = 0.0f;
    }
};

// ---------------------------------------------------------------------------------------- bicycle (SURVEY 8(f) #3)
// examples/bicycle.py:11-146 behind the legacy adapter (envs.py:230-241): float64 lean/steer dynamics with sin, cos, tan and a
// square root per step, in the reference's operation order.  The reference's own results depend on its host's libm / SVML /
// BLAS builds (np.tan, `** 0.5` = pow, ddot; see oracle/envs_oracle.py), so this task is held to a stated tolerance, not to
// bit equality: CUDA's f64 sin/cos/tan are within 2 ulp, `** 0.5` is __dsqrt_rn, the 2-vector dots round like the FMA ddot.
struct BicycleTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 7, A = 3, MAX_STEPS = 2000, NBUF = 4;
    typedef tmla_bicycle_state Wire;
    struct State { double x, z, theta, phi, phi_dot, delta, gx, gz, dist; int steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int b) { return b < 3 ? 16 : 32; }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        const double2 p = reinterpret_cast<const double2 *>(buf[0])[i], q = reinterpret_cast<const double2 *>(buf[1])[i];
        const double2 r = reinterpret_cast<const double2 *>(buf[2])[i];
        const double2 g = reinterpret_cast<const double2 *>(buf[3])[2 * i], m = reinterpret_cast<const double2 *>(buf[3])[2 * i + 1];
        const long long meta = __double_as_longlong(m.y);                       // steps | ep_return bits << 32
        return State{p.x, p.y, q.x, q.y, r.x, r.y, g.x, g.y, m.x, (int)(meta & 0xFFFFFFFFll), __int_as_float((int)(meta >> 32))};
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        reinterpret_cast<double2 *>(buf[0])[i] = make_double2(s.x, s.z);
        reinterpret_cast<double2 *>(buf[1])[i] = make_double2(s.theta, s.phi);
        reinterpret_cast<double2 *>(buf[2])[i] = make_double2(s.phi_dot, s.delta);
        const long long meta = (long long)(unsigned)s.steps | ((long long)__float_as_int(s.ep_ret) << 32);
        reinterpret_cast<double2 *>(buf[3])[2 * i] = make_double2(s.gx, s.gz);
        reinterpret_cast<double2 *>(buf[3])[2 * i + 1] = make_double2(s.dist, __longlong_as_double(meta));
    }
    static __device__ State from_wire(const Wire &w) {
        return State{w.x, w.z, w.theta, w.phi, w.phi_dot, w.delta, w.goal[0], w.goal[1], w.dist, w.steps, w.ep_return};
    }
    static __device__ Wire to_wire(const State &s) {
        Wire w; w.x = s.x; w.z = s.z; w.theta = s.theta; w.phi = s.phi; w.phi_dot = s.phi_dot; w.delta = s.delta;
        w.goal[0] = s.gx; w.goal[1] = s.gz; w.dist = s.dist; w.steps = s.steps; w.ep_return = s.ep_ret; return w;
    }
    // np.linalg.norm / np.dot on 2-vectors = BLAS ddot, which rounds as fma(a1, b1, a0*b0) on FMA hosts (oracle: dot2)
    static __device__ __forceinline__ double dot2(double a0, double a1, double b0, double b1) { return __fma_rn(a1, b1, __dmul_rn(a0, b0)); }
    static __device__ __forceinline__ void observe(const State &s, float *o) {   // bicycle.py:128-145, cast envs.py:150
        const double v0 = __dsub_rn(s.gx, s.x), v1 = __dsub_rn(s.gz, s.z);
        const double dist = __dsqrt_rn(dot2(v0, v1, v0, v1));
        double st, ct;
        sincos(s.theta, &st, &ct);
        o[0] = __double2float_rn(s.phi); o[1] = __double2float_rn(s.phi_dot); o[2] = __double2float_rn(s.delta);
        o[3] = __double2float_rn(ct); o[4] = __double2float_rn(st);
        o[5] = dist > 0.0 ? __double2float_rn(__ddiv_rn(v0, dist)) : 0.0f;
        o[6] = dist > 0.0 ? __double2float_rn(__ddiv_rn(v1, dist)) : 0.0f;
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        constexpr double DT = 0.02, GH = 9.8 / 0.8, VLH = 25.0 / (1.0 * 0.8), VL = 5.0 / 1.0;        // bicycle.py:15-20 as evaluated
        constexpr double MAX_PHI = 3.141592653589793 / 4, MAX_DELTA = 3.141592653589793 / 6;       // :29-30
        double delta = __dadd_rn(s.delta, a == 0 ? -0.05 : (a == 2 ? 0.05 : 0.0));                 // :63-69
        delta = fmin(fmax(delta, -MAX_DELTA), MAX_DELTA);                                          // :70
        double sp, cp;
        sincos(s.phi, &sp, &cp);
        const double phi_ddot = __dsub_rn(__dmul_rn(GH, sp), __dmul_rn(__dmul_rn(VLH, tan(delta)), cp));   // :74-76
        const double phi_dot = __dadd_rn(s.phi_dot, __dmul_rn(phi_ddot, DT));                      // :77
        const double phi = __dadd_rn(s.phi, __dmul_rn(phi_dot, DT));                               // :78
        delta = __dmul_rn(delta, 0.95);                                                            // :81
        const double theta = __dadd_rn(s.theta, __dmul_rn(__dmul_rn(VL, tan(delta)), DT));         // :84
        double st, ct;
        sincos(theta, &st, &ct);
        const double x = __dadd_rn(s.x, __dmul_rn(__dmul_rn(5.0, ct), DT));                        // :85
        const double z = __dadd_rn(s.z, __dmul_rn(__dmul_rn(5.0, st), DT));                        // :86
        const double g0 = __dsub_rn(s.gx, x), g1 = __dsub_rn(s.gz, z);
        const double nd = __dsqrt_rn(dot2(g0, g1, g0, g1));                                        // :91
        const double progress = __dmul_rn(__dsub_rn(s.dist, nd), 10.0);                            // :94
        const double upright = __dmul_rn(__dsub_rn(1.0, __dsqrt_rn(__ddiv_rn(fabs(phi), MAX_PHI))), 0.2);   // :98
        const double den = nd > 0.0 ? nd : 1.0;                                                    // :103-105
        const double heading = __dmul_rn(dot2(ct, st, __ddiv_rn(g0, den), __ddiv_rn(g1, den)), 0.3);   // :101-106
        const double steering = __dmul_rn(-__ddiv_rn(fabs(delta), MAX_DELTA), 0.1);                // :109
        double r = __dadd_rn(__dadd_rn(__dadd_rn(progress, upright), heading), steering);          // :111
        s.x = x; s.z = z; s.theta = theta; s.phi = phi; s.phi_dot = phi_dot; s.delta = delta; s.dist = nd;
        s.steps += 1;
        bool done = false;
        if (fabs(phi) > MAX_PHI) { r = -10.0; done = true; }                                       // :113-115
        if (s.steps > 2000) done = true;                                                           // :117-118
        if (nd < 2.0) { r = 50.0; done = true; }                                                   // :120-122
        reward = __double2float_rn(r);
        trunc = s.steps >= MAX_STEPS;                                                              // envs.py:141-145
        term = done && !trunc;
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        const uint4 b = tmla_stream_block(seed, env_id, k, tag, 0);                                // bicycle.py:40-58
        s.x = 0.0; s.z = 0.0; s.theta = 0.0; s.delta = 0.0;
        s.phi = __dadd_rn(-0.1, __dmul_rn(0.2, u32_to_unit(b.x)));                                 // uniform(lo, hi) = lo + (hi - lo) * u
        s.phi_dot = __dadd_rn(-0.1, __dmul_rn(0.2, u32_to_unit(b.y)));
        const double radius = __dadd_rn(15.0, __dmul_rn(10.0, u32_to_unit(b.z)));
        double sn, cs;
        sin_cos_quarter(__dadd_rn(-0.78539816339744830962, __dmul_rn(1.57079632679489661923, u32_to_unit(b.w))), sn, cs);
        s.gx = __dmul_rn(radius, cs); s.gz = __dmul_rn(radius, sn);
        s.dist = __dsqrt_rn(dot2(s.gx, s.gz, s.gx, s.gz));
        s.steps = 0; s.ep_ret = 0.0f;
    }
};

// ---------------------------------------------------------------------------------------- glider (SURVEY 8(f) #3)
// examples/glider.py:11-265 behind the legacy adapter (envs.py:244-255): float64 rigid-body glider in a sinusoidal thermal
// field, 16-float observation, 5 actions, 4000-step limit.  Reference operation order throughout; the BLAS calls of the
// reference (np.linalg.norm / np.dot on 3-vectors, the 3x3 `@` chain, R @ f) round as forward FMA chains on FMA hosts
// (measured, see oracle/envs_oracle.py) and are written out that way with the structural zeros and ones of the rotation
// matrices folded (an FMA with a zero factor is the identity).  Like bicycle the task is held to a stated tolerance:
// CUDA's f64 sin / cos / atan2 are within 2 ulp of the host's.
struct GliderTask {
    static constexpr bool HAS_SPARE = false;
    typedef NoSpare Spare;
    typedef NoConsts Consts;
    static __device__ __forceinline__ Consts load_consts() { return Consts{}; }
    static constexpr int D = 16, A = 5, MAX_STEPS = 4000, NBUF = 4;
    typedef tmla_glider_state Wire;
    struct State { double pos[3], vel[3], rot[3], av[3]; int wp, steps; float ep_ret; };
    static __host__ __device__ size_t plane_bytes(int b) { return b < 3 ? 32 : 16; }

    static __device__ __forceinline__ State load(void *const *buf, int64_t i) {
        State s;
        double v[12];
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const double2 lo = reinterpret_cast<const double2 *>(buf[b])[2 * i], hi = reinterpret_cast<const double2 *>(buf[b])[2 * i + 1];
            v[4 * b] = lo.x; v[4 * b + 1] = lo.y; v[4 * b + 2] = hi.x; v[4 * b + 3] = hi.y;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) { s.pos[k] = v[k]; s.vel[k] = v[3 + k]; s.rot[k] = v[6 + k]; s.av[k] = v[9 + k]; }
        const int4 m = reinterpret_cast<const int4 *>(buf[3])[i];
        s.wp = m.x; s.steps = m.y; s.ep_ret = __int_as_float(m.z);
        return s;
    }
    static __device__ __forceinline__ void store(void *const *buf, int64_t i, const State &s) {
        double v[12];
#pragma unroll
        for (int k = 0; k < 3; ++k) { v[k] = s.pos[k]; v[3 + k] = s.vel[k]; v[6 + k] = s.rot[k]; v[9 + k] = s.av[k]; }
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            reinterpret_cast<double2 *>(buf[b])[2 * i] = make_double2(v[4 * b], v[4 * b + 1]);
            reinterpret_cast<double2 *>(buf[b])[2 * i + 1] = make_double2(v[4 * b + 2], v[4 * b + 3]);
        }
        reinterpret_cast<int4 *>(buf[3])[i] = make_int4(s.wp, s.steps, __float_as_int(s.ep_ret), 0);
    }
    static __device__ State from_wire(const Wire &w) {
        State s;
        for (int k = 0; k < 3; ++k) { s.pos[k] = w.pos[k]; s.vel[k] = w.vel[k]; s.rot[k] = w.rot[k]; s.av[k] = w.ang_vel[k]; }
        s.wp = w.waypoint & 1; s.steps = w.steps; s.ep_ret = w.ep_return;
        return s;
    }
    static __device__ Wire to_wire(const State &s) {
        Wire w;
        for (int k = 0; k < 3; ++k) { w.pos[k] = s.pos[k]; w.vel[k] = s.vel[k]; w.rot[k] = s.rot[k]; w.ang_vel[k] = s.av[k]; }
        w.waypoint = s.wp; w.steps = s.steps; w.ep_return = s.ep_ret; w.pad_ = 0;
        return w;
    }
    // ddot / dgemm / dgemv on 3-vectors: forward FMA chain
    static __device__ __forceinline__ double dot3(const double *a, const double *b) {
        return __fma_rn(a[2], b[2], __fma_rn(a[1], b[1], __dmul_rn(a[0], b[0])));
    }
    static __device__ __forceinline__ void to_target(const State &s, double *vec, double &dist) {   // glider.py:173-175 / 243-245
        vec[0] = __dsub_rn(s.wp ? 160.0 : -160.0, s.pos[0]);
        vec[1] = __dsub_rn(0.0, s.pos[1]);
        vec[2] = __dsub_rn(70.0, s.pos[2]);
        dist = __dsqrt_rn(dot3(vec, vec));
    }
    static __device__ __forceinline__ void observe(const State &s, float *o) {   // glider.py:241-265, cast envs.py:150
        double vec[3], dist, sy, cy;
        to_target(s, vec, dist);
        sincos(s.rot[2], &sy, &cy);
        const double den = __dadd_rn(dist, 1e-8);
        o[0] = __double2float_rn(__ddiv_rn(s.vel[2], 10.0));
        o[1] = __double2float_rn(__ddiv_rn(__dsub_rn(s.pos[2], 50.0), 50.0));
        o[2] = __double2float_rn(s.rot[0]); o[3] = __double2float_rn(s.rot[1]);
        o[4] = __double2float_rn(sy); o[5] = __double2float_rn(cy);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            o[6 + k] = __double2float_rn(s.av[k]);
            o[9 + k] = __double2float_rn(__ddiv_rn(s.vel[k], 20.0));
            o[12 + k] = __double2float_rn(__ddiv_rn(vec[k], den));
        }
        o[15] = __double2float_rn(__ddiv_rn(dist, 100.0));
    }
    static __device__ __forceinline__ void step(const Consts &, State &s, int a, float &reward, bool &term, bool &trunc) {
        constexpr double PI = 3.141592653589793, DT = 0.02, MASS = 1.5, G = 9.81;
        constexpr double F1 = 1.0 / 250.0, F2 = 1.0 / 400.0, CL_ALPHA = 2 * PI, MAX_AOA = 0.2617993877991494;   // np.deg2rad(15)
        const double roll_t = a == 1 ? -15.0 : (a == 2 ? 15.0 : 0.0), pitch_t = a == 3 ? 10.0 : (a == 4 ? -10.0 : 0.0);   // glider.py:92-103
        const double yaw_t = a == 1 ? 4.0 : (a == 2 ? -4.0 : 0.0);
        s.av[0] = __dmul_rn(__dadd_rn(s.av[0], __dmul_rn(roll_t, DT)), 0.95);                      // :107-110
        s.av[1] = __dmul_rn(__dadd_rn(s.av[1], __dmul_rn(pitch_t, DT)), 0.95);
        s.av[2] = __dmul_rn(__dadd_rn(s.av[2], __dmul_rn(yaw_t, DT)), 0.95);
#pragma unroll
        for (int k = 0; k < 3; ++k) s.rot[k] = __dadd_rn(s.rot[k], __dmul_rn(s.av[k], DT));       // :111
        s.rot[0] = fmin(fmax(s.rot[0], -PI / 2), PI / 2);                                          // :114-115
        s.rot[1] = fmin(fmax(s.rot[1], -PI / 4), PI / 4);
        // wind at the position before integration (:55-77): ((x * f) * 2) * pi [/ 1.5]
        const double ax1 = __dmul_rn(__dmul_rn(__dmul_rn(s.pos[0], F1), 2.0), PI), ay1 = __dmul_rn(__dmul_rn(__dmul_rn(s.pos[1], F1), 2.0), PI);
        const double ax2 = __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(s.pos[0], F2), 2.0), PI), 1.5), ay2 = __ddiv_rn(ay1, 1.5);
        const double up1 = __dmul_rn(__dmul_rn(__dmul_rn(sin(ax1), cos(ay1)), 8.0), 1.0);
        const double up2 = __dmul_rn(__dmul_rn(__dmul_rn(sin(ax2), cos(ay2)), 8.0), 0.7);
        const double va[3] = {__dsub_rn(s.vel[0], 1.0), __dsub_rn(s.vel[1], 0.5), __dsub_rn(s.vel[2], __dadd_rn(up1, up2))};   // :118-119
        const double vam = __dsqrt_rn(dot3(va, va));                                               // :120
        double aoa = va[0] != 0.0 ? atan2(-va[2], va[0]) : 0.0;                                    // :123
        double aero[3] = {0.0, 0.0, 0.0};
        if (vam > 0.1) {                                                                           // :125-160
            const double CL = __dmul_rn(CL_ALPHA, aoa);
            const double CD = __dadd_rn(0.02, __dmul_rn(0.05, __dmul_rn(CL, CL)));
            const double q = __dmul_rn(__dmul_rn(0.5 * 1.225, __dmul_rn(vam, vam)), 0.5);          // ((0.5 * rho) * |v|^2) * S
            const double lift = __dmul_rn(q, CL), ndrag = -__dmul_rn(q, CD);
            double s0, c0, s1, c1, s2, c2;
            sincos(s.rot[0], &s0, &c0); sincos(s.rot[1], &s1, &c1); sincos(s.rot[2], &s2, &c2);
            // R = (R_yaw @ R_pitch) @ R_roll, columns 0 and 2 (the force [-drag, 0, lift] has no y component)
            const double r00 = __dmul_rn(c2, c1), r10 = __dmul_rn(s2, c1), r20 = -s1;
            const double r02 = __fma_rn(__dmul_rn(c2, s1), c0, __dmul_rn(-s2, -s0));
            const double r12 = __fma_rn(__dmul_rn(s2, s1), c0, __dmul_rn(c2, -s0));
            const double r22 = __dmul_rn(c1, c0);
            aero[0] = __fma_rn(r02, lift, __dmul_rn(r00, ndrag));                                  // dgemv: fma(R[i][2], f2, R[i][0] * f0)
            aero[1] = __fma_rn(r12, lift, __dmul_rn(r10, ndrag));
            aero[2] = __fma_rn(r22, lift, __dmul_rn(r20, ndrag));
        } else aoa = 0.0;
        aero[2] = __dadd_rn(aero[2], -(MASS * G));                                                 // :162-163 (adding 0 to x, y is exact)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            s.vel[k] = __dadd_rn(s.vel[k], __dmul_rn(__ddiv_rn(aero[k], MASS), DT));               // :166
            s.pos[k] = __dadd_rn(s.pos[k], __dmul_rn(s.vel[k], DT));                               // :167
        }
        double vec[3], dist;
        to_target(s, vec, dist);
        if (dist < 15.0) s.wp ^= 1;                                                                // :177-180
        const double vmag = __dsqrt_rn(dot3(s.vel, s.vel));
        const double dv = __dadd_rn(vmag, 1e-8), dt_ = __dadd_rn(dist, 1e-8);
        const double vd[3] = {__ddiv_rn(s.vel[0], dv), __ddiv_rn(s.vel[1], dv), __ddiv_rn(s.vel[2], dv)};   // :183-185
        const double td[3] = {__ddiv_rn(vec[0], dt_), __ddiv_rn(vec[1], dt_), __ddiv_rn(vec[2], dt_)};
        const double Hh = __ddiv_rn(__dadd_rn(dot3(vd, td), 1.0), 2.0);                            // :188
        const double E = fmin(fmax(__ddiv_rn(vmag, 30.0), 0.0), 2.0);                              // :190-192
        double r = __dmul_rn(E, __dadd_rn(__dsub_rn(Hh, E), 1.0));                                 // :196
        const double lateral = fabs(s.pos[1]);                                                     // :201-206
        if (lateral > 250.0) { const double pr = __ddiv_rn(__dsub_rn(lateral, 250.0), 100.0); r = __dsub_rn(r, __dmul_rn(2.0, __dmul_rn(pr, pr))); }
        if (s.pos[2] > 250.0) { const double pr = __ddiv_rn(__dsub_rn(s.pos[2], 250.0), 50.0); r = __dsub_rn(r, __dmul_rn(2.0, __dmul_rn(pr, pr))); }   // :209-215
        else if (s.pos[2] < 25.0) r = __dsub_rn(r, 0.5);
        bool done = false;
        if (s.pos[2] < 5.0) { r = -50.0; done = true; }                                            // :218-220
        if (fabs(aoa) > MAX_AOA) { r = -50.0; done = true; }                                       // :223-225
        if (dist > 500.0) { r = -50.0; done = true; }                                              // :228-230
        s.steps += 1;
        if (s.steps > 4000) done = true;                                                           // :233-234
        reward = __double2float_rn(r);
        trunc = s.steps >= MAX_STEPS;                                                              // envs.py:141-145
        term = done && !trunc;
    }
    struct Pending { float r; };
    static __device__ __forceinline__ void advance(const NoConsts &c, State &s, int a, Pending &pend, bool &term, bool &trunc) {
        step(c, s, a, pend.r, term, trunc);
    }
    static __device__ __forceinline__ float finish(const Pending &pend) { return pend.r; }
    static __device__ __forceinline__ void reset(State &s, uint64_t seed, uint64_t env_id, uint64_t k, uint32_t tag) {
        const uint4 b = tmla_stream_block(seed, env_id, k, tag, 0);                                // glider.py:79-86
        s.pos[0] = 0.0; s.pos[1] = 0.0; s.pos[2] = 60.0;
        s.vel[0] = 15.0; s.vel[1] = 0.0; s.vel[2] = -1.0;
        s.rot[0] = 0.0; s.rot[1] = 0.0; s.rot[2] = 0.0;
        s.av[0] = __dadd_rn(-0.1, __dmul_rn(0.2, u32_to_unit(b.x)));                               // np.random.uniform(-0.1, 0.1, 3)
        s.av[1] = __dadd_rn(-0.1, __dmul_rn(0.2, u32_to_unit(b.y)));
        s.av[2] = __dadd_rn(-0.1, __dmul_rn(0.2, u32_to_unit(b.z)));
        s.wp = (int)(b.w >> 31);                                                                   // np.random.randint(0, 2)
        s.steps = 0; s.ep_ret = 0.0f;
    }
};
