// Counter-based reset RNG for the swarm env batch: Philox4x32-10 (Salmon et al., SC'11).
//
// Replaces the reference's global MT19937 stream (fed_gym/envs/multiagent.py:48-56) with a
// stateless generator keyed by (seed, GLOBAL env id, episode), so an env's draws do not
// depend on how the batch is sharded over GPUs, and any draw can be regenerated in place.
//
// Draw layout (restated for the tests in oracle/philox.py; rows past n_burn in tests/_fresh_noise.py):
//   key     = (seed & 0xffffffff, seed >> 32)
//   counter = (element index, row, global env id, (episode << 3) | stream)
//   stream 0: x0   1: xa0   2: burn-in actions (rows 0..n_burn-1)
//          3: agent noise (rows 0..n_burn + elapsed)   4: particle noise (rows 0..n_burn + elapsed)
//   (rows 0..n_burn-1 feed the burn-in, row n_burn the first step after the reset -- and every later step
//   in the frozen mode of the reference; with SWARM_STEP_FRESH_NOISE step `elapsed` uses row n_burn + elapsed)
//   stream 5: the physics row of SWARM_PHYSICS_RESAMPLE (uniform pairs 0..2, row 0: column c is pair c / 2, .x / .y)
#pragma once
#include <stdint.h>

namespace swarm {

enum : uint32_t { STREAM_X0 = 0, STREAM_XA0 = 1, STREAM_BURN = 2, STREAM_NOISE_A = 3, STREAM_NOISE_X = 4,
                  STREAM_PHYSICS = 5 };

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

struct DrawCtx {
    uint2 key;
    uint32_t env;      // global env id
    uint32_t episode;  // resets completed so far
};

__device__ __forceinline__ uint4 draw_words(const DrawCtx& c, uint32_t stream, uint32_t row, uint32_t idx) {
    return philox4x32_10(make_uint4(idx, row, c.env, (c.episode << 3) | stream), c.key);
}

// two doubles in [0,1) with 53 random bits each (numpy's legacy random_sample bit recipe)
__device__ __forceinline__ double2 draw_uniform2(const DrawCtx& c, uint32_t stream, uint32_t idx) {
    const uint4 o = draw_words(c, stream, 0u, idx);
    const double k = 1.0 / 9007199254740992.0;
    double2 u;
    u.x = ((double)(o.x >> 5) * 67108864.0 + (double)(o.y >> 6)) * k;
    u.y = ((double)(o.z >> 5) * 67108864.0 + (double)(o.w >> 6)) * k;
    return u;
}

// two independent N(0,1) (FP32 Box-Muller, returned as doubles)
__device__ __forceinline__ double2 draw_normal2(const DrawCtx& c, uint32_t stream, uint32_t row, uint32_t idx) {
    const uint4 o = draw_words(c, stream, row, idx);
    const float u1 = ((float)(o.x >> 8) + 1.0f) * 5.9604644775390625e-8f;  // (0,1]
    const float u2 = (float)(o.y >> 8) * 5.9604644775390625e-8f;           // [0,1)
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    return make_double2((double)(rad * cs), (double)(rad * sn));
}

}  // namespace swarm
