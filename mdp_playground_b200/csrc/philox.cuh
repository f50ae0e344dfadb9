// Philox4x32-10 counter-based RNG (Salmon et al., SC'11) and the draw
// conversions of the step path.  Stateless: every draw is a pure function of
// (seed, global env id, global step index, stream), so results do not depend
// on launch shape, rollout chunking or the number of GPUs.
// oracle/philox.py restates exactly these functions in numpy.
#pragma once
#include <stdint.h>

namespace mdpp {

enum PhiloxStream : uint32_t {
  // per-step streams: counter = (env, quad lo, quad hi, stream), quad = step>>2,
  // word j of the result belongs to step 4*quad + j
  STREAM_STEP = 0,       // 32-bit transition uniforms
  STREAM_RESET = 1,      // manual reset(): counter word 1 = episode, w0,w1 -> u53
  STREAM_ACTION = 2,     // counter = (env, step): w0 -> uniform policy action
  STREAM_IMAGE = 3,      // image transform draws
  STREAM_NORMAL = 4,     // (w0,w1),(w2,w3) -> two Box-Muller pairs (reward noise)
  STREAM_AUTORESET = 5,  // 32-bit uniforms of the same-step auto-reset
  STREAM_ZIG = 6,        // counter = step >> 1: (w0,w1) / (w2,w3) = the 64-bit
                         // first ziggurat word of the even / odd step
  STREAM_STATE_NOISE = 8,  // + pair index: continuous transition noise
  STREAM_IRR_STEP = 32,       // like STREAM_STEP / STREAM_AUTORESET, for the
  STREAM_IRR_AUTORESET = 33,  // irrelevant sub-MDP (irrelevant_features)
  // grid envs: GRID_STEP counter = (env, step >> 1): (w0, w1) / (w2, w3) =
  // noise decision + substitute action of the even / odd step; GRID_NORMAL
  // counter = (env, step >> 2): 4 reward normals; auto-reset (counter = step)
  // and reset() (counter word 1 = episode): one word per dimension
  STREAM_GRID_STEP = 40,
  STREAM_GRID_AUTORESET = 41,
  STREAM_GRID_RESET = 42,
  STREAM_GRID_NORMAL = 43,
  // grid Q-learning (mdpp_grid_qlearn), counter = (env, step >> 1): (w0, w1) /
  // (w2, w3) = explore decision + exploring action of the even / odd step
  STREAM_GRID_ACTION = 45,
  STREAM_RESET_BOX = 64,   // + attempt*16 + dim/4 (continuous reset sampling)
  STREAM_ZIG_RETRY = 0x100,  // + c, counter = step: ziggurat words after a
                             // rejected first attempt (ziggurat.cuh)
  // ziggurat normals of the continuous and grid kernels: the first word of
  // state-noise dimensions (2c, 2c+1) = (w0,w1) / (w2,w3) of STREAM_STATE_NOISE
  // + c, of the continuous reward normal = (w0,w1) of STREAM_NORMAL (counter =
  // step); of the grid reward normal = the STREAM_GRID_ZIG word pair of the
  // step's parity (counter = step >> 1).  Retries of draw j of a step (j =
  // dimension, 16 = continuous reward, 17 = grid reward): + 64 j + c
  STREAM_GRID_ZIG = 44,
  STREAM_ZIG_DRAW_RETRY = 0x1000,
  // ARS perturbations (ars.cu), counter = (global id of the pair's + member,
  // iteration lo, iteration hi): word c of delta is STREAM_ARS_DELTA + c, c <
  // 68.  No other stream range reaches it: 0x1000 + 64 j + c tops out near
  // 0x1450, and the wrapper tail's 0x10000 + pair stays below 0x16000.
  STREAM_ARS_DELTA = 0x20000,
};

struct U4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ U4 philox4x32_10(uint32_t c0, uint32_t c1,
                                                     uint32_t c2, uint32_t c3,
                                                     uint32_t k0, uint32_t k1) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)M0 * c0;
    uint64_t p1 = (uint64_t)M1 * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += W0;
    k1 += W1;
  }
  return U4{c0, c1, c2, c3};
}

// The 10 round keys depend only on the launch-constant seed: the host expands
// them once into the kernel parameters (constant bank), so the hot loop spends
// no instructions on the key schedule.
__host__ __device__ __forceinline__ void philox_round_keys(uint32_t k0, uint32_t k1,
                                                           uint32_t* rk) {
  for (int r = 0; r < 10; ++r) {
    rk[2 * r] = k0 + (uint32_t)r * 0x9E3779B9u;
    rk[2 * r + 1] = k1 + (uint32_t)r * 0xBB67AE85u;
  }
}
#ifdef MDPP_EXP_PHILOX_ROUNDS  // (timing experiment only: NOT the contract's generator)
constexpr int kPhiloxRounds = MDPP_EXP_PHILOX_ROUNDS;
#else
constexpr int kPhiloxRounds = 10;
#endif
__host__ __device__ __forceinline__ U4 philox4x32_10_rk(uint32_t c0, uint32_t c1,
                                                        uint32_t c2, uint32_t c3,
                                                        const uint32_t* rk) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < kPhiloxRounds; ++r) {
    uint64_t p0 = (uint64_t)M0 * c0;
    uint64_t p1 = (uint64_t)M1 * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ rk[2 * r];
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ rk[2 * r + 1];
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
  }
  return U4{c0, c1, c2, c3};
}

// 53-bit uniform in [0,1): same construction as numpy's PCG64 double
// ((x >> 11) * 2^-53) applied to the 64-bit word (hi:lo).
__host__ __device__ __forceinline__ double uniform53(uint32_t lo, uint32_t hi) {
  uint64_t x = ((uint64_t)hi << 32) | lo;
  return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}

// 32-bit uniform in (0,1): (w + 0.5) * 2^-32 (exact in fp64).
__host__ __device__ __forceinline__ double uniform32(uint32_t w) {
  return ((double)w + 0.5) * (1.0 / 4294967296.0);
}

#ifdef __CUDACC__
// Box-Muller pair, fp64: r = sqrt(-2 ln u1); (z0, z1) = r (cos, sin)(2 pi u2).
__device__ __forceinline__ void normal_pair_f64(uint32_t a, uint32_t b,
                                                double* z0, double* z1) {
  double r = sqrt(-2.0 * log(uniform32(a)));
  double s, c;
  sincospi(2.0 * uniform32(b), &s, &c);
  *z0 = r * c;
  *z1 = r * s;
}
// Box-Muller pair on the SFU (MUFU lg2 / sqrt / sin / cos, fp32): ~1e-6
// relative accuracy, |z| <= 6.7.  The distribution tests in
// tests/test_cuda_discrete.py apply to both variants.
__device__ __forceinline__ void normal_pair_fast(uint32_t a, uint32_t b,
                                                 double* z0, double* z1) {
  const float u1 = ((float)(a >> 8) + 0.5f) * (1.0f / 16777216.0f);
  const float u2 = ((float)(b >> 8) + 0.5f) * (1.0f / 16777216.0f);
  // -2 ln u = -2 ln2 * log2 u
  // u1 is in [2^-25, 1): no denormal handling needed, so the bare SFU forms
  float lg, r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u1));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg));
  float s, c;
  __sincosf(6.283185307179586f * u2, &s, &c);
  *z0 = (double)(r * c);
  *z1 = (double)(r * s);
}
#endif

}  // namespace mdpp
