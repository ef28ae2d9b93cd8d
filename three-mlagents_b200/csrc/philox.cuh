// philox.cuh — Philox4x32-10 counter-based generator and this repo's stream layout.
// CPU twin: oracle/philox.py (bit-exact; pinned by Random123 known-answer vectors).
// Replaces the reference's global MT19937 draws (np.random.* in examples/ball3d.py:49-57,
// gridworld.py:42-50, push.py:40-47), which cannot be reproduced per-env (SURVEY.md §3.4).
#pragma once
#include <stdint.h>

#define TMLA_TAG_RESET 0u
#define TMLA_TAG_ACTION 1u
#define TMLA_TAG_SAMPLE 2u
#define TMLA_TAG_PERM 3u
#define TMLA_TAG_RESET_ALL 4u

__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c.x;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c.z;
        uint4 n;
        n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k.x;
        n.y = (uint32_t)p1;
        n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k.y;
        n.w = (uint32_t)p0;
        c = n;
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// ctr = (env_lo, env_hi, k_lo, k_hi<<8 | block<<4 | tag) ; key = (seed_lo, seed_hi)
__host__ __device__ __forceinline__ uint4 tmla_stream_block(uint64_t seed, uint64_t env_id, uint64_t k,
                                                            uint32_t tag, uint32_t block) {
    uint4 c;
    c.x = (uint32_t)env_id;
    c.y = (uint32_t)(env_id >> 32);
    c.z = (uint32_t)k;
    c.w = ((uint32_t)(k >> 32) << 8) | (block << 4) | tag;
    return philox4x32_10(c, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// Lemire multiply-shift: floor(x*n / 2^32)
__host__ __device__ __forceinline__ int tmla_bounded(uint32_t x, uint32_t n) {
    return (int)(((uint64_t)x * n) >> 32);
}
// 53-bit double in [0,1): ((a>>5)*2^26 + (b>>6)) / 2^53  (MT19937 genrand_res53 recipe)
__host__ __device__ __forceinline__ double tmla_u53(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}
__host__ __device__ __forceinline__ float tmla_u24(uint32_t a) { return (float)(a >> 8) * (1.0f / 16777216.0f); }

// Random-policy action stream (TAG_ACTION): one Philox block serves 16 consecutive steps.  Word w of the
// block is read as a 32-bit fraction and expanded into 4 base-A digits by repeated multiply-shift
// (digit = floor(frac*A), frac = frac*A mod 1); bias per digit <= A^4 / 2^32.
//   step k -> block k>>4, word (k&15)>>2, digit k&3
struct TmlaActionStream {
    uint4 blk;
    uint32_t frac;
    __device__ __forceinline__ static uint32_t word_of(const uint4 &b, uint32_t w) {
        return w == 0 ? b.x : (w == 1 ? b.y : (w == 2 ? b.z : b.w));
    }
    // position the stream so that the next call to next() yields the action of step k
    __device__ __forceinline__ void seek(uint64_t seed, uint64_t env_id, uint64_t k, uint32_t n_actions) {
        blk = tmla_stream_block(seed, env_id, k >> 4, TMLA_TAG_ACTION, 0);
        frac = word_of(blk, (uint32_t)(k & 15u) >> 2);
        for (uint32_t d = 0; d < (uint32_t)(k & 3u); ++d) frac = (uint32_t)((uint64_t)frac * n_actions);
    }
    // action of step k = step0 + t (t must advance by one per call after seek(step0)).  Only the low bits of
    // k are touched on the common path; the 64-bit counter is formed inside the 1-in-16 Philox branch.
    __device__ __forceinline__ int next(uint64_t seed, uint64_t env_id, uint64_t step0, uint32_t t, uint32_t n_actions) {
        const uint32_t j = ((uint32_t)step0 + t) & 15u;
        if ((j & 3u) == 0) {
            if (j == 0 && t != 0) blk = tmla_stream_block(seed, env_id, (step0 + t) >> 4, TMLA_TAG_ACTION, 0);
            frac = word_of(blk, j >> 2);
        }
        const uint64_t p = (uint64_t)frac * n_actions;
        frac = (uint32_t)p;
        return (int)(p >> 32);
    }
    // The 16 actions of Philox block `blk` (steps 16*blk .. 16*blk+15), expanded by the same multiply-shift sequence as
    // next() and packed as 4-bit digits: the action of step 16*blk + j is (digits >> 4*j) & 15.  Needs n_actions <= 16.
    __device__ __forceinline__ static uint64_t block_digits(uint64_t seed, uint64_t env_id, uint64_t blk, uint32_t n_actions) {
        const uint4 b = tmla_stream_block(seed, env_id, blk, TMLA_TAG_ACTION, 0);
        const uint32_t w[4] = {b.x, b.y, b.z, b.w};
        uint32_t half[2] = {0u, 0u};                      // digits 0-7 | digits 8-15
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t frac = w[q];
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const uint64_t p = (uint64_t)frac * n_actions;
                frac = (uint32_t)p;
                half[q >> 1] |= (uint32_t)(p >> 32) << (4 * (4 * (q & 1) + d));
            }
        }
        return ((uint64_t)half[1] << 32) | half[0];
    }
};
