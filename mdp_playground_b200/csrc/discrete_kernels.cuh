// Discrete RLToyEnv step path on sm_100a: K1/K2 `discrete_rollout` (T fused
// steps, T = 1 is the gym-style single step) and K6 `discrete_reset`.
//
// Restates (per env, per step) rl_toy_env.py
//   transition_function :1602-1622   s' = P[s,a]; noisy redraw via cdf search
//   step                :2050-2058   window shift, t += 1
//   reward_function     :1817-1846   custom R[s,a] | gated sequence lookup
//                       :1968-1990   delay FIFO, every-n gate, noise, scale, shift
//   step epilogue       :2098-2109   done = terminal(s'), += term reward * scale
//   reset               :2250-2278   s0 ~ init dist, window/FIFO/t cleared
//
// Work decomposition: one thread = one environment, state in registers for
// the whole launch.  A CTA serves one configuration group; the group's tables
// (P as u16, terminal mask, init / noise cdfs, sequence LUT or hash, reward
// values) are staged once into shared memory with 128-bit copies.  Global
// traffic is struct-of-arrays, time-major [T][N], so every warp access is one
// contiguous segment.  Steps are processed in chunks of U: the chunk's
// action loads and its state-independent Philox / Box-Muller work are issued
// up front (memory- and instruction-level parallelism), then the short
// state-dependent chain runs.
#pragma once
#include "device_types.h"
#include "philox.cuh"
#include "ziggurat.cuh"

namespace mdpp {

constexpr int kBlock = 64;
#ifdef MDPP_JIT_CHUNK  // tuning override of the NVRTC build
constexpr int kChunk = MDPP_JIT_CHUNK;
#else
constexpr int kChunk = 8;
#endif
// 65 536 envs / 148 SMs = 443 threads per SM: all of them must be resident at
// once (one wave), so cap registers at 65 536 / 512 = 128 per thread.  Small
// CTAs (64 threads) keep the per-SM load within one CTA of the average
// (7 vs 6.9 CTAs) -- the kernel is issue-bound, so imbalance is lost time.
#ifdef MDPP_JIT_MINBLOCKS
constexpr int kMinBlocksPerSM = MDPP_JIT_MINBLOCKS;
#else
constexpr int kMinBlocksPerSM = 8;
#endif


// Launch-wide scalars: literals in a runtime-specialised build (jit.cu).
__device__ __forceinline__ int64_t n_envs_of(const RolloutParams& p) {
#ifdef MDPP_JIT
  return MDPP_N_ENVS;
#else
  return p.st.n_envs;
#endif
}
__device__ __forceinline__ bool autoreset_of(const RolloutParams& p) {
#ifdef MDPP_JIT
  return MDPP_AUTORESET != 0;
#else
  return p.autoreset != 0;
#endif
}
__device__ __forceinline__ int horizon_of(const RolloutParams& p) {
#ifdef MDPP_JIT
  return MDPP_HORIZON;
#else
  return p.horizon;
#endif
}

// element type of obs / final_obs (the reference's dtype_o): launch-wide
__device__ __forceinline__ int obs_dtype_of(const RolloutParams& p) {
#ifdef MDPP_JIT
  return MDPP_OBS_DTYPE;
#else
  return p.io.obs_dtype;
#endif
}

// Ziggurat normals staged a window ahead (zig_fill) only when the launch
// covers at least one window; shorter launches draw them chunk by chunk.
__device__ __forceinline__ bool stage_of(const RolloutParams& p) {
#ifdef MDPP_EXP_NO_STAGE  // (timing experiment: draw chunk by chunk)
  return false;
#elif defined(MDPP_JIT)
  return MDPP_CFG_STAGE;
#else
  return p.T >= kZigWindow;
#endif
}

// irrelevant_features: launch-wide (all groups agree, context.cu).  The
// ahead-of-time FAST kernels never see it (discrete_launch.h routes such
// launches to the generic variants), a specialised build gets a literal.
template <typename C>
__device__ __forceinline__ bool irr_of(const RolloutParams& p) {
#ifdef MDPP_JIT
  return MDPP_IRR != 0;
#else
  return !C::FAST && p.irr != 0;
#endif
}

// cache hint of the output stores (tuning knob of the NVRTC build):
// default .cs (streaming / evict first)
#if defined(MDPP_ST_POLICY) && MDPP_ST_POLICY == 1
#define MDPP_ST_HINT ""
#elif defined(MDPP_ST_POLICY) && MDPP_ST_POLICY == 2
#define MDPP_ST_HINT ".wt"
#elif defined(MDPP_ST_POLICY) && MDPP_ST_POLICY == 3
#define MDPP_ST_HINT ".cg"
#else
#define MDPP_ST_HINT ".cs"
#endif

__device__ __forceinline__ int2 ld_stream_i32x2(const int32_t* p) {
  int2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.s32 {%0, %1}, [%2];"
               : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ double2 ld_stream_f64x2(const double* p) {
  double2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];"
               : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream_x2(int64_t* p, int64_t a, int64_t b) {
  asm volatile("st.global" MDPP_ST_HINT ".v2.s64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}

__device__ __forceinline__ int32_t ld_stream_i32(const int32_t* p) {
  int32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ld_stream_f64(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
#ifndef MDPP_EXP_SKIP  // timing experiments only: drop classes of memory ops
#define MDPP_EXP_SKIP 0
#endif
__device__ __forceinline__ void st_stream(int64_t* p, int64_t v) {
  if (MDPP_EXP_SKIP & 2) return;
  asm volatile("st.global" MDPP_ST_HINT ".s64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_stream(double* p, double v) {
  if (MDPP_EXP_SKIP & 2) return;
  asm volatile("st.global" MDPP_ST_HINT ".f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void st_stream(int32_t* p, int32_t v) {
  if (MDPP_EXP_SKIP & 2) return;
  asm volatile("st.global" MDPP_ST_HINT ".s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream(uint8_t* p, uint8_t v) {
  if (MDPP_EXP_SKIP & 1) return;
  asm volatile("st.global" MDPP_ST_HINT ".u8 [%0], %1;" ::"l"(p), "r"((uint32_t)v) : "memory");
}

// one observation (row of 2 with an irrelevant sub-state) in the caller's dtype_o
__device__ __forceinline__ void store_obs(const RolloutParams& p, int64_t* base,
                                          int64_t off, bool irr, int32_t s,
                                          int32_t s_irr) {
  const int dt = obs_dtype_of(p);
  if (dt == MDPP_OBS_I64) {
    if (irr) st_stream_x2(base + 2 * off, (int64_t)s, (int64_t)s_irr);
    else st_stream(base + off, (int64_t)s);
  } else if (dt == MDPP_OBS_I32) {
    int32_t* b = reinterpret_cast<int32_t*>(base);
    if (irr) { st_stream(b + 2 * off, s); st_stream(b + 2 * off + 1, s_irr); }
    else st_stream(b + off, s);
  } else {
    uint8_t* b = reinterpret_cast<uint8_t*>(base);
    if (irr) { st_stream(b + 2 * off, (uint8_t)s); st_stream(b + 2 * off + 1, (uint8_t)s_irr); }
    else st_stream(b + off, (uint8_t)s);
  }
}

// numpy searchsorted(cdf, u, side='right') = number of entries <= u, as a
// branch-free binary search over a row padded to 2^log2n entries with a
// sentinel larger than any u (context.cu).  LOG2 >= 0 fixes the trip count at
// compile time (fully unrolled); LOG2 < 0 reads it from the group.
template <int LOG2>
__device__ __forceinline__ int cdf_search(const double* cdf, int log2n, int n,
                                          double u) {
  int pos = 0;
  if (LOG2 >= 0) {
#pragma unroll
    for (int b = LOG2 - 1; b >= 0; --b)
      if (cdf[pos + (1 << b) - 1] <= u) pos += 1 << b;
  } else {
#pragma unroll 1
    for (int step = (1 << log2n) >> 1; step > 0; step >>= 1)
      if (cdf[pos + step - 1] <= u) pos += step;
  }
  return min(pos, n - 1);
}

// Philox-mode noisy transition: (nxt + kk) mod S with kk = 0 (keep P[s,a]) or
// the pre-drawn rotation 1..S-1 -- uniform over the S-1 other states.
__device__ __forceinline__ int32_t rotate_state(int32_t nxt, int32_t kk, int S) {
  const int32_t t = nxt + kk;
  if ((S & (S - 1)) == 0) return t & (S - 1);
  return t >= S ? t - S : t;
}

// Identities a specialised build may use (see chain_step).
#if defined(MDPP_SCALE) && defined(MDPP_SHIFT) && defined(MDPP_TERM_REWARD)
constexpr bool kScaleIsOne = (MDPP_SCALE) == 1.0;
constexpr bool kShiftIsZero = (MDPP_SHIFT) == 0.0 && !MDPP_SHIFT_NEGZERO;
constexpr bool kTermRewardIsZero =
    (MDPP_TERM_REWARD) == 0.0 && !MDPP_TERM_NEGZERO && !MDPP_SHIFT_NEGZERO;
#else
constexpr bool kScaleIsOne = false, kShiftIsZero = false, kTermRewardIsZero = false;
#endif

struct GroupView {  // per-thread copy of the scalars + table pointers
  int S, A, L, delay, every_n, lookup_kind, key_bits, hash_shift;
  int cdf_log2, cdf_stride;
  bool has_pnoise, has_rnoise, has_guide, p8;
  const uint8_t* guide;
  uint32_t hash_mask;
  uint64_t key_mask;
  uint64_t pn_T, term_mask;  // closed-form transition noise (device_types.h)
  uint32_t pn_M;
  int pn_shift;
  double r_std, scale, shift, term_reward_scaled;
  const uint16_t* P;
  const uint8_t* term;
  const double* init_cdf;
  const double* noise_cdf;
  const double* lut;
  const uint64_t* hash_keys;
  const uint32_t* hash_vals;
  const double* values;
  const double* R;
  // irrelevant sub-MDP
  int S1, A1, irr_cdf_log2, irr_cdf_stride, irr_pn_shift;
  uint32_t irr_pn_M;
  const uint16_t* P_irr;
  const double* init_cdf_irr;
  const double* noise_cdf_irr;
  const uint4* zig_kw;  // {wi, (double)ki}[256] of the ziggurat, in shared memory
};

__device__ __forceinline__ GroupView make_view(const DiscreteGroupDev& g,
                                               const uint8_t* tab,
                                               const uint4* zig_kw) {
  GroupView v;
  v.zig_kw = zig_kw;
  v.S = g.S; v.A = g.A; v.L = g.L; v.delay = g.delay; v.every_n = g.every_n;
  v.lookup_kind = g.lookup_kind; v.key_bits = g.key_bits;
  v.hash_shift = g.hash_shift; v.hash_mask = g.hash_mask;
  v.has_pnoise = g.has_pnoise != 0; v.has_rnoise = g.has_rnoise != 0;
  v.cdf_log2 = g.cdf_log2; v.cdf_stride = g.cdf_stride;
  v.has_guide = g.has_guide != 0;
  v.p8 = g.p_is_u8 != 0;
  v.guide = tab + g.off_guide;
  v.key_mask = g.key_mask;
  v.r_std = g.r_std; v.scale = g.scale; v.shift = g.shift;
  v.term_reward_scaled = g.term_reward_scaled;
  v.P = reinterpret_cast<const uint16_t*>(tab + g.off_P);
  v.term = tab + g.off_term;
  v.init_cdf = reinterpret_cast<const double*>(tab + g.off_init_cdf);
  v.noise_cdf = reinterpret_cast<const double*>(tab + g.off_noise_cdf);
  v.pn_T = g.pn_T; v.pn_M = g.pn_M; v.pn_shift = g.pn_shift;
  v.term_mask = g.term_mask;
  v.lut = reinterpret_cast<const double*>(tab + g.off_lut);
  v.hash_keys = reinterpret_cast<const uint64_t*>(tab + g.off_hash_keys);
  v.hash_vals = reinterpret_cast<const uint32_t*>(tab + g.off_hash_vals);
  v.values = reinterpret_cast<const double*>(tab + g.off_values);
  v.R = reinterpret_cast<const double*>(tab + g.off_R);
  v.S1 = g.S1; v.A1 = g.A1;
  v.irr_cdf_log2 = g.irr_cdf_log2; v.irr_cdf_stride = g.irr_cdf_stride;
  v.irr_pn_M = g.irr_pn_M; v.irr_pn_shift = g.irr_pn_shift;
  v.P_irr = reinterpret_cast<const uint16_t*>(tab + g.off_P_irr);
  v.init_cdf_irr = reinterpret_cast<const double*>(tab + g.off_init_cdf_irr);
  v.noise_cdf_irr = reinterpret_cast<const double*>(tab + g.off_noise_cdf_irr);
#ifdef MDPP_JIT
  // Runtime-compiled specialisation (jit.cu): every group scalar that is the
  // same for all groups of the launch arrives as a literal, so the compiler
  // folds the branches, unrolls the searches and drops the dead features.
  // Scalars that differ between groups stay run-time (read from the group
  // descriptor above).
#ifdef MDPP_S
  v.S = MDPP_S;
#endif
#ifdef MDPP_A
  v.A = MDPP_A;
#endif
#ifdef MDPP_L
  v.L = MDPP_L;
#endif
#ifdef MDPP_DELAY
  v.delay = MDPP_DELAY;
#endif
#ifdef MDPP_EVERY_N
  v.every_n = MDPP_EVERY_N;
#endif
#ifdef MDPP_LOOKUP
  v.lookup_kind = MDPP_LOOKUP;
#endif
#ifdef MDPP_KEY_BITS
  v.key_bits = MDPP_KEY_BITS;
#endif
#ifdef MDPP_HASH_SHIFT
  v.hash_shift = MDPP_HASH_SHIFT;
#endif
#ifdef MDPP_HASH_MASK
  v.hash_mask = MDPP_HASH_MASK;
#endif
#ifdef MDPP_KEY_MASK
  v.key_mask = MDPP_KEY_MASK;
#endif
#ifdef MDPP_PNOISE
  v.has_pnoise = MDPP_PNOISE;
#endif
#ifdef MDPP_RNOISE
  v.has_rnoise = MDPP_RNOISE;
#endif
#ifdef MDPP_CDF_LOG2
  v.cdf_log2 = MDPP_CDF_LOG2; v.cdf_stride = 1 << MDPP_CDF_LOG2;
#endif
#ifdef MDPP_HAS_GUIDE
  v.has_guide = MDPP_HAS_GUIDE;
#endif
#ifdef MDPP_P8
  v.p8 = MDPP_P8;
#endif
#ifdef MDPP_PN_T
  v.pn_T = MDPP_PN_T; v.pn_M = MDPP_PN_M; v.pn_shift = MDPP_PN_SHIFT;
#endif
#ifdef MDPP_R_STD
  v.r_std = MDPP_R_STD;
#endif
#ifdef MDPP_SCALE
  v.scale = MDPP_SCALE;
#endif
#ifdef MDPP_SHIFT
  v.shift = MDPP_SHIFT;
#endif
#ifdef MDPP_TERM_REWARD
  v.term_reward_scaled = MDPP_TERM_REWARD;
#endif
#endif
  return v;
}

// P[idx]: u8 entries when every group table has <= 256 states, else u16
__device__ __forceinline__ int32_t table_next(const GroupView& v,
                                              const uint16_t* P, int32_t idx) {
  return v.p8 ? (int32_t)reinterpret_cast<const uint8_t*>(P)[idx] : (int32_t)P[idx];
}

__device__ __forceinline__ double sequence_reward(const GroupView& v,
                                                  uint64_t key) {
  if (v.lookup_kind == LOOKUP_LUT) return v.lut[key];
  if (v.lookup_kind == LOOKUP_LUT8)
    return v.values[reinterpret_cast<const uint8_t*>(v.lut)[key]];
  uint32_t slot = (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> v.hash_shift) &
                  v.hash_mask;
  while (true) {
    uint64_t k = v.hash_keys[slot];
    if (k == key) return v.values[v.hash_vals[slot]];
    if (k == kHashEmpty) return 0.0;
    slot = (slot + 1) & v.hash_mask;
  }
}

constexpr int kMaxRingRegs = 4;

struct EnvRegs {
  int32_t s;
  int32_t s_irr;  // irrelevant sub-state (irrelevant_features)
  uint64_t key;
  int32_t tl;
  int32_t phase;  // tl % every_n, tracked incrementally (no division per step)
  uint32_t ep;
  int32_t ring_pos;  // step % delay
  int32_t hist_pos;  // (step + 1) % history_depth
  double fifo[kMaxRingRegs];  // Cfg::RING_REGS: the delay FIFO, newest first
  // statistics accumulated over the launch
  double sum_reward, sum_abs_rnoise;
  uint32_t n_noisy, n_episodes, n_terminated, n_steps;
};

// Philox-mode draws of a group of 4 consecutive steps (quad = step >> 2),
// all state-independent so they are produced ahead of the state chain:
//   STREAM_STEP   word j          -> 32-bit transition uniform of step 4q+j
//   STREAM_NORMAL words (0,1),(2,3) -> two Box-Muller pairs = 4 reward normals
//   STREAM_AUTORESET word j       -> 32-bit uniform of the auto-reset after
//                                    step 4q+j
template <int NORMAL>
__device__ __forceinline__ uint32_t philox_quad_draws(
    uint32_t gid, uint64_t quad, const uint32_t* rk, bool want_u,
    bool want_normal, bool want_reset, uint32_t* w_tr, double* z, uint32_t* w_rs,
    const uint4* zig_kw) {
  const uint32_t q0 = (uint32_t)quad, q1 = (uint32_t)(quad >> 32);
  uint32_t rejected = 0;  // NORMAL == 2: bit j = step 4q+j needs zig_slow()
#ifdef MDPP_EXP_NO_CHAIN_PHILOX  // (timing experiment: a multiplicative hash instead)
#define MDPP_CHAIN_WORDS(stream) \
  U4{(gid ^ q0) * 2654435761u + stream, (gid + q0) * 2246822519u, (gid ^ (q0 << 7)) * 3266489917u, (gid - q0) * 668265263u}
#else
#define MDPP_CHAIN_WORDS(stream) philox4x32_10_rk(gid, q0, q1, stream, rk)
#endif
  if (want_u) {
    U4 w = MDPP_CHAIN_WORDS(STREAM_STEP);
    w_tr[0] = w.x; w_tr[1] = w.y; w_tr[2] = w.z; w_tr[3] = w.w;
  }
  if (want_normal) {
    if (NORMAL == MDPP_NORMAL_ZIGGURAT) {
      // one 64-bit word per normal: pair counter = step >> 1 = 2 quad (+ 1)
      const uint64_t pair = quad << 1;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint64_t pr = pair + h;
        U4 w = philox4x32_10_rk(gid, (uint32_t)pr, (uint32_t)(pr >> 32), STREAM_ZIG, rk);
        bool ok0, ok1;
        z[2 * h] = zig_first(w.x, w.y, zig_kw, &ok0);
        z[2 * h + 1] = zig_first(w.z, w.w, zig_kw, &ok1);
        if (!ok0) rejected |= 1u << (2 * h);
        if (!ok1) rejected |= 2u << (2 * h);
      }
    } else {
      U4 w = philox4x32_10_rk(gid, q0, q1, STREAM_NORMAL, rk);
      if (NORMAL == MDPP_NORMAL_F64) {
        normal_pair_f64(w.x, w.y, &z[0], &z[1]);
        normal_pair_f64(w.z, w.w, &z[2], &z[3]);
      } else {
        normal_pair_fast(w.x, w.y, &z[0], &z[1]);
        normal_pair_fast(w.z, w.w, &z[2], &z[3]);
      }
    }
  }
  if (want_reset) {
    U4 w = MDPP_CHAIN_WORDS(STREAM_AUTORESET);
    w_rs[0] = w.x; w_rs[1] = w.y; w_rs[2] = w.z; w_rs[3] = w.w;
  }
  return rejected;
}

// Compile-time configuration of a rollout kernel.
//   FAST  the standard rollout signature -- actions given; obs, reward,
//         terminated, truncated all written; no final_obs, no history -- so
//         none of the per-step NULL tests survive in the hot loop; tables and
//         the delay ring are in shared memory.
//   CDF_LOG2 >= 0: cdf rows have exactly 2^CDF_LOG2 entries (unrolled search).
//   SINGLE the launch has one configuration group: its descriptor comes
//         from the kernel parameters instead of shared memory.
//   RING_REGS = d > 0: every group has delay d <= kMaxRingRegs and the FIFO
//         lives in registers as a shift register (in unrolled code the shift
//         is a renaming, i.e. free); 0: ring buffer in shared / global memory.
template <int NOISE_, int NORMAL_, bool SMEM_, bool RING_SMEM_, bool FAST_,
          int CDF_LOG2_, bool SINGLE_ = false, int RING_REGS_ = 0>
struct Cfg {
  static constexpr bool SINGLE = SINGLE_;
  static constexpr int RING_REGS = RING_REGS_;
  static constexpr int NOISE = NOISE_;
  static constexpr int NORMAL = NORMAL_;
  static constexpr bool SMEM = SMEM_;
  static constexpr bool RING_SMEM = RING_SMEM_;
  static constexpr bool FAST = FAST_;
  static constexpr int CDF_LOG2 = CDF_LOG2_;
};

// ---- agents riding along the chain ------------------------------------------
// rollout_body runs a policy-free rollout with NoAgent: every hook is empty and
// inlines to nothing.  qlearn.cu plugs a learner in through the same hooks:
// draw()   sees the STREAM_ACTION words of the random policy (phase A),
// act()    picks the action of a step from the random one and the env state,
// update() sees the step's outcome (StepOut) and the state after any reset,
// begin() / end() load and store per-env agent state around the launch.
struct NoAgent {
  static constexpr bool kStepOut = false;  // chain_step hands out no StepOut
  __device__ __forceinline__ void begin(const GroupView&, int64_t, int32_t) {}
  __device__ __forceinline__ void draw(int, const U4&) {}
  __device__ __forceinline__ int32_t act(int, int32_t a_rand, int32_t) { return a_rand; }
  __device__ __forceinline__ void update(const RolloutParams&, const GroupView&,
                                         const StepOut&, int32_t, int64_t, int64_t) {}
  __device__ __forceinline__ void end(int64_t) {}
};

// ---- phase A: loads and state-independent random draws -------------------
// Everything a chunk of U steps needs that does not depend on the env state:
// the actions, the transition uniforms, the (sigma-scaled) reward normals and
// the candidate initial states of a possible auto-reset.  `n_valid` < U only
// on the last chunk of a launch (guards the action / replay loads).
// PRELOADED: act[] already holds the chunk's actions (prefetched by the
// caller one chunk ahead, see rollout_body).

// The same quantities for the irrelevant sub-MDP (irrelevant_features): dead
// code, hence no registers, in builds without one.
template <int U>
struct IrrDraws {
  int32_t act[U];
  double u_tr[U];
  int32_t k_tr[U];
  int32_t s0[U];
};

template <typename C>
__device__ __forceinline__ void load_action(const RolloutParams& p, int64_t off,
                                            int32_t& a, int32_t& a_irr) {
  if (MDPP_EXP_SKIP & 4) { a = (int32_t)(off & 7); a_irr = 0; return; }  // (timing experiment)
  if (irr_of<C>(p)) {  // rows (relevant, irrelevant): one 8-byte load
    const int2 v = ld_stream_i32x2(p.io.actions + 2 * off);
    a = v.x; a_irr = v.y;
  } else {
    a = ld_stream_i32(p.io.actions + off); a_irr = 0;
  }
}

// `zs` (STAGED): this thread's column of staged ziggurat normals, sigma
// applied, zs[j * kBlock] = step t0 + j (zig_fill); else drawn here.
template <typename C, int U, bool PRELOADED = false, bool STAGED = false,
          typename AG = NoAgent>
__device__ __forceinline__ void phase_a(const RolloutParams& p, const GroupView& v,
                                        AG& ag, int64_t env, uint32_t gid,
                                        uint64_t step_base, int t0,
                                        int n_valid, int32_t* act, double* u_tr,
                                        int32_t* k_tr, double* n_rw, int32_t* s0,
                                        IrrDraws<U>& q, const double* zs = nullptr) {
  constexpr int NOISE = C::NOISE;
  constexpr int NORMAL = C::NORMAL;
  constexpr bool FAST = C::FAST;
  const int64_t N = n_envs_of(p);
  const bool autoreset = autoreset_of(p);
  const bool irr = irr_of<C>(p);
  double u_rs[U], u_rs_i[U];
  const int64_t off0 = (int64_t)t0 * N + env;
  const uint64_t step0 = step_base + (uint64_t)t0;
  const bool have_actions = FAST || p.io.actions != nullptr;
#pragma unroll
  for (int j = 0; j < U; ++j) {
    const int64_t off = off0 + (int64_t)j * N;
    const uint64_t step = step0 + (uint64_t)j;
    if (PRELOADED) {
    } else if (have_actions) {
      act[j] = 0; q.act[j] = 0;
      if (j < n_valid) load_action<C>(p, off, act[j], q.act[j]);
    } else {
      U4 w = philox4x32_10(gid, (uint32_t)step, (uint32_t)(step >> 32),
                           STREAM_ACTION, p.k0, p.k1);
      act[j] = (int32_t)__umulhi(w.x, (uint32_t)v.A);
      q.act[j] = irr ? (int32_t)__umulhi(w.y, (uint32_t)v.A1) : 0;
      ag.draw(j, w);
    }
    u_tr[j] = 0.0; k_tr[j] = 0; n_rw[j] = 0.0; u_rs[j] = 0.0; s0[j] = 0;
    q.u_tr[j] = 0.0; q.k_tr[j] = 0; q.s0[j] = 0; u_rs_i[j] = 0.0;
    if (NOISE == MDPP_NOISE_REPLAY && j < n_valid) {
      if (irr) {  // rows (relevant, irrelevant)
        if (v.has_pnoise) {
          const double2 u = ld_stream_f64x2(p.io.replay_transition_u + 2 * off);
          u_tr[j] = u.x; q.u_tr[j] = u.y;
        }
        if (autoreset) {
          const double2 u = ld_stream_f64x2(p.io.replay_reset_u + 2 * off);
          u_rs[j] = u.x; u_rs_i[j] = u.y;
        }
      } else {
        if (v.has_pnoise) u_tr[j] = ld_stream_f64(p.io.replay_transition_u + off);
        if (autoreset) u_rs[j] = ld_stream_f64(p.io.replay_reset_u + off);
      }
      if (v.has_rnoise) n_rw[j] = ld_stream_f64(p.io.replay_reward_noise + off);
    }
  }
  uint32_t w_rs[U], w_tr[U];
#pragma unroll
  for (int j = 0; j < U; ++j) w_rs[j] = w_tr[j] = 0;
  if (NOISE != MDPP_NOISE_REPLAY) {
    const bool want_u = NOISE == MDPP_NOISE_PHILOX && v.has_pnoise;
    const bool want_z = NOISE == MDPP_NOISE_PHILOX && v.has_rnoise && !STAGED;
    const bool want_r = autoreset;
    if (STAGED && v.has_rnoise) {
#pragma unroll
      for (int j = 0; j < U; ++j) n_rw[j] = zs[j * kBlock];
    }
    if (U == 1) {
      double z4[4] = {0, 0, 0, 0};
      uint32_t u4[4] = {0, 0, 0, 0}, r4[4] = {0, 0, 0, 0};
      constexpr bool ZIG1 = NORMAL == MDPP_NORMAL_ZIGGURAT;
      philox_quad_draws<NORMAL>(gid, step0 >> 2, p.rk, want_u, want_z && !ZIG1,
                                want_r, u4, z4, r4, v.zig_kw);
      const int q4 = (int)(step0 & 3);
      w_tr[0] = q4 == 0 ? u4[0] : q4 == 1 ? u4[1] : q4 == 2 ? u4[2] : u4[3];
      double z = q4 == 0 ? z4[0] : q4 == 1 ? z4[1] : q4 == 2 ? z4[2] : z4[3];
      w_rs[0] = q4 == 0 ? r4[0] : q4 == 1 ? r4[1] : q4 == 2 ? r4[2] : r4[3];
      if (ZIG1 && want_z) {  // a single step: only the pair word that holds it
        const uint64_t pr = step0 >> 1;
        const U4 w = philox4x32_10_rk(gid, (uint32_t)pr, (uint32_t)(pr >> 32),
                                      STREAM_ZIG, p.rk);
        bool ok;
        z = zig_first((step0 & 1) ? w.z : w.x, (step0 & 1) ? w.w : w.y, v.zig_kw, &ok);
        if (!ok)
          z = zig_slow(gid, step0, p.rk, reinterpret_cast<const uint8_t*>(v.zig_kw));
      }
      if (!STAGED) n_rw[0] = __dmul_rn(v.r_std, z);
    } else {  // chunks start on a multiple-of-4 step (see the callers)
      uint32_t rej = 0;
#pragma unroll
      for (int j = 0; j + 3 < U; j += 4) {
        double z4[4] = {0, 0, 0, 0};
        rej |= philox_quad_draws<NORMAL>(gid, (step0 + j) >> 2, p.rk, want_u,
                                         want_z, want_r, &w_tr[j], z4, &w_rs[j],
                                         v.zig_kw) << j;
        // numpy: normal(0, sigma) = 0 + sigma * z
        if (!STAGED) {
#pragma unroll
          for (int k = 0; k < 4; ++k) n_rw[j + k] = __dmul_rn(v.r_std, z4[k]);
        }
      }
#ifdef MDPP_EXP_NO_SLOW
      rej = 0;
#endif
      if (NORMAL == MDPP_NORMAL_ZIGGURAT && !STAGED) {
        // the 1.5 % of draws whose first ziggurat attempt was rejected: one
        // out-of-line call per draw, lanes without one wait
#pragma unroll 1
        while (rej) {
          const int jb = __ffs((int)rej) - 1;
          rej &= rej - 1;
          const double nz = __dmul_rn(v.r_std, zig_slow(gid, step0 + jb, p.rk,
                                       reinterpret_cast<const uint8_t*>(v.zig_kw)));
#pragma unroll
          for (int j = 0; j < U; ++j)
            if (j == jb) n_rw[j] = nz;
        }
      }
    }
  }
  if (NOISE == MDPP_NOISE_PHILOX && v.has_pnoise) {
    // closed-form noisy draw (device_types.h): 0 = keep P[s,a], else the
    // rotation 1..S-1 that picks one of the S-1 other states;
    // state-independent, so done here
#pragma unroll
    for (int j = 0; j < U; ++j) {
      const uint32_t k = __umulhi(w_tr[j], v.pn_M) >> v.pn_shift;
      k_tr[j] = ((uint64_t)w_tr[j] < v.pn_T) ? (int32_t)k + 1 : 0;
    }
  }
  if (autoreset) {  // candidate initial states, also state-independent
    if (NOISE != MDPP_NOISE_REPLAY && v.has_guide) {
      // guide lookups for the whole chunk, then ONE rarely taken branch for
      // the buckets that straddle a cdf boundary (keeps the chunk's code in
      // one basic block, so the scheduler can interleave it freely)
      int32_t worst = 0;
#pragma unroll
      for (int j = 0; j < U; ++j) {
        s0[j] = v.guide[w_rs[j] >> (32 - kGuideBits)];
        worst = max(worst, s0[j]);
      }
      if (worst == kGuideMiss) {
#pragma unroll  // (a rolled loop would index s0 / w_rs dynamically: local memory)
        for (int j = 0; j < U; ++j)
          if (s0[j] == kGuideMiss)
            s0[j] = cdf_search<C::CDF_LOG2>(v.init_cdf, v.cdf_log2, v.S,
                                            uniform32(w_rs[j]));
      }
    } else {
#pragma unroll
      for (int j = 0; j < U; ++j) {
        const double u = NOISE == MDPP_NOISE_REPLAY ? u_rs[j] : uniform32(w_rs[j]);
        s0[j] = cdf_search<C::CDF_LOG2>(v.init_cdf, v.cdf_log2, v.S, u);
      }
    }
  }
  if (irr) {
    // the irrelevant sub-MDP's own words: STREAM_IRR_STEP / _AUTORESET, word j
    // of quad (step >> 2) like the relevant streams
    if (NOISE != MDPP_NOISE_REPLAY) {
      const bool want_u = NOISE == MDPP_NOISE_PHILOX && v.has_pnoise;
      uint32_t wi_tr[U], wi_rs[U];
#pragma unroll
      for (int j = 0; j < U; ++j) wi_tr[j] = wi_rs[j] = 0;
      if (U == 1) {
        const uint64_t quad = step0 >> 2;
        const int q4 = (int)(step0 & 3);
        if (want_u) {
          U4 w = philox4x32_10_rk(gid, (uint32_t)quad, (uint32_t)(quad >> 32),
                                  STREAM_IRR_STEP, p.rk);
          wi_tr[0] = q4 == 0 ? w.x : q4 == 1 ? w.y : q4 == 2 ? w.z : w.w;
        }
        if (autoreset) {
          U4 w = philox4x32_10_rk(gid, (uint32_t)quad, (uint32_t)(quad >> 32),
                                  STREAM_IRR_AUTORESET, p.rk);
          wi_rs[0] = q4 == 0 ? w.x : q4 == 1 ? w.y : q4 == 2 ? w.z : w.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j + 3 < U; j += 4) {
          const uint64_t quad = (step0 + j) >> 2;
          if (want_u) {
            U4 w = philox4x32_10_rk(gid, (uint32_t)quad, (uint32_t)(quad >> 32),
                                    STREAM_IRR_STEP, p.rk);
            wi_tr[j] = w.x; wi_tr[j + 1] = w.y; wi_tr[j + 2] = w.z; wi_tr[j + 3] = w.w;
          }
          if (autoreset) {
            U4 w = philox4x32_10_rk(gid, (uint32_t)quad, (uint32_t)(quad >> 32),
                                    STREAM_IRR_AUTORESET, p.rk);
            wi_rs[j] = w.x; wi_rs[j + 1] = w.y; wi_rs[j + 2] = w.z; wi_rs[j + 3] = w.w;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < U; ++j) {
        if (want_u) {
          const uint32_t k = __umulhi(wi_tr[j], v.irr_pn_M) >> v.irr_pn_shift;
          q.k_tr[j] = ((uint64_t)wi_tr[j] < v.pn_T) ? (int32_t)k + 1 : 0;
        }
        u_rs_i[j] = uniform32(wi_rs[j]);
      }
    }
    if (autoreset) {
#pragma unroll
      for (int j = 0; j < U; ++j)
        q.s0[j] = cdf_search<-1>(v.init_cdf_irr, v.irr_cdf_log2, v.S1, u_rs_i[j]);
    }
  }
}

// ---- phase B: the state-dependent chain -----------------------------------
// One environment step given its pre-drawn randomness.
template <typename C>
__device__ __forceinline__ void chain_step(const RolloutParams& p, const GroupView& v,
                                           EnvRegs& e, double* ring_smem,
                                           int ring_stride, int64_t env, int64_t off,
                                           int32_t act, double u_tr, int32_t k_tr,
                                           double n_rw, int32_t s0,
                                           int32_t act_i, double u_tr_i,
                                           int32_t k_tr_i, int32_t s0_i,
                                           StepOut* so = nullptr) {
  constexpr int NOISE = C::NOISE;
  constexpr bool RING_SMEM = C::RING_SMEM;
  constexpr bool FAST = C::FAST;
  const int64_t N = n_envs_of(p);
  const bool autoreset = autoreset_of(p);
  const int horizon = horizon_of(p);
  const bool irr = irr_of<C>(p);
  if (irr) {
    // the irrelevant sub-MDP (rl_toy_env.py:2062-2082): same table walk and
    // noisy redraw, no reward, no terminal states
    uint32_t ai = (uint32_t)act_i;
    if (ai >= (uint32_t)v.A1) ai = (uint32_t)v.A1 - 1;  // memory safety only
    int32_t nxt_i = table_next(v, v.P_irr, e.s_irr * v.A1 + (int32_t)ai);
    if (NOISE == MDPP_NOISE_REPLAY && v.has_pnoise) {
      nxt_i = cdf_search<-1>(v.noise_cdf_irr + nxt_i * v.irr_cdf_stride,
                             v.irr_cdf_log2, v.S1, u_tr_i);
    } else if (NOISE == MDPP_NOISE_PHILOX && v.has_pnoise) {
      nxt_i = rotate_state(nxt_i, k_tr_i, v.S1);
    }
    e.s_irr = nxt_i;
  }
  uint32_t a = (uint32_t)act;
  if (a >= (uint32_t)v.A) a = (uint32_t)v.A - 1;  // memory safety only
  int32_t nxt = table_next(v, v.P, e.s * v.A + (int32_t)a);
  if (NOISE == MDPP_NOISE_REPLAY && v.has_pnoise) {
    // the recorded fp64 uniform against the fp64 cdf, like the reference
    const int32_t noisy = cdf_search<C::CDF_LOG2>(
        v.noise_cdf + nxt * v.cdf_stride, v.cdf_log2, v.S, u_tr);
    e.n_noisy += (noisy != nxt);
    nxt = noisy;
  } else if (NOISE == MDPP_NOISE_PHILOX && v.has_pnoise) {
    nxt = rotate_state(nxt, k_tr, v.S);  // one of the S-1 other states
#ifndef MDPP_EXP_NO_STATS  // (timing experiment)
    e.n_noisy += (k_tr != 0);
#endif
  }
  e.key = ((e.key << v.key_bits) | (uint64_t)nxt) & v.key_mask;
  e.tl += 1;
  e.phase = (e.phase + 1 == v.every_n) ? 0 : e.phase + 1;
  double r = 0.0;
  if (v.lookup_kind == LOOKUP_MATRIX) {
    r = v.R[e.s * v.A + (int32_t)a];
  } else if (e.tl >= v.L) {  // isnan(aug[delay]) gate <=> t < L
    r = sequence_reward(v, e.key);
  }
  if (C::RING_REGS > 0) {
    constexpr int D = C::RING_REGS > 0 ? C::RING_REGS : 1;
    const double delayed = (e.tl > D) ? e.fifo[D - 1] : 0.0;
#pragma unroll
    for (int k = D - 1; k > 0; --k) e.fifo[k] = e.fifo[k - 1];
    e.fifo[0] = r;
    r = delayed;
  } else if (v.delay > 0) {  // FIFO of depth d: pay out what was earned d steps ago
    double* slot = RING_SMEM
        ? ring_smem + e.ring_pos * ring_stride
        : p.st.ring + (int64_t)e.ring_pos * N + env;
    double delayed = (e.tl > v.delay) ? *slot : 0.0;
    *slot = r;
    r = delayed;
    e.ring_pos = (e.ring_pos + 1 == v.delay) ? 0 : e.ring_pos + 1;
  }
  if (e.phase != 0) r = 0.0;
#ifndef MDPP_EXP_NO_STATS
  e.sum_reward += r;
#endif
  if (NOISE != MDPP_NOISE_OFF && v.has_rnoise) {
#ifndef MDPP_EXP_NO_STATS
    e.sum_abs_rnoise += fabs(n_rw);
#endif
    r = __dadd_rn(r, n_rw);
  }
  // `* 1.0` is the identity; `+ 0.0` only turns -0.0 into +0.0, and no -0.0
  // can reach this point when scale == 1 (context.cu stores no negative
  // zero and x + y is -0.0 only if both are) -- so a specialised build whose
  // literals say so drops these operations, bit-exactly
  if (!kScaleIsOne) r = __dmul_rn(r, v.scale);
  if (!(kScaleIsOne && kShiftIsZero)) r = __dadd_rn(r, v.shift);
  const bool done = v.S <= 64 ? ((v.term_mask >> nxt) & 1ull) != 0
                              : v.term[nxt] != 0;
  if (!kTermRewardIsZero)
    if (done) r = __dadd_rn(r, v.term_reward_scaled);
  const bool trunc = horizon > 0 && e.tl >= horizon;
  if (so) { so->r = r; so->nxt = nxt; so->done = done; so->trunc = trunc; }
#ifndef MDPP_EXP_NO_STATS
  e.n_terminated += done;
#endif
  e.s = nxt;
  if (!FAST && p.io.final_obs) store_obs(p, p.io.final_obs, off, irr, nxt, e.s_irr);
  if (autoreset && (done || trunc)) {
    e.s = s0;
    if (irr) e.s_irr = s0_i;
    e.key = (uint64_t)e.s;
    e.tl = 0;
    e.phase = 0;
    e.n_episodes += 1;  // (the episode counter advances by the same amount)
  }
  if (!FAST && p.st.history) {
    p.st.history[(int64_t)e.hist_pos * N + env] = e.s;
    e.hist_pos = (e.hist_pos + 1 == p.st.history_depth) ? 0 : e.hist_pos + 1;
  }
  if (FAST || p.io.obs) store_obs(p, p.io.obs, off, irr, e.s, e.s_irr);
  if (FAST || p.io.reward) st_stream(p.io.reward + off, r);
  if (FAST || p.io.terminated) st_stream(p.io.terminated + off, (uint8_t)done);
  if (FAST || p.io.truncated) st_stream(p.io.truncated + off, (uint8_t)trunc);
}

template <typename C, int U, bool PARTIAL, typename AG>
__device__ __forceinline__ void phase_b(const RolloutParams& p, const GroupView& v,
                                        AG& ag, EnvRegs& e, double* ring_smem,
                                        int ring_stride,
                                        int64_t env, int t0, int n_valid,
                                        const int32_t* act, const double* u_tr,
                                        const int32_t* k_tr, const double* n_rw,
                                        const int32_t* s0, const IrrDraws<U>& q) {
  const int64_t N = n_envs_of(p);
  const int64_t off0 = (int64_t)t0 * N + env;
#pragma unroll
  for (int j = 0; j < U; ++j) {
    if (PARTIAL && j >= n_valid) break;
    const int64_t off = off0 + (int64_t)j * N;
    StepOut so;
    chain_step<C>(p, v, e, ring_smem, ring_stride, env, off,
                  ag.act(j, act[j], e.s), u_tr[j], k_tr[j], n_rw[j], s0[j],
                  q.act[j], q.u_tr[j], q.k_tr[j], q.s0[j],
                  AG::kStepOut ? &so : nullptr);
    ag.update(p, v, so, e.s, env, off);
  }
  e.n_steps += PARTIAL ? n_valid : U;
}

// A full chunk whose actions were prefetched into act[] (and act_i[]).
template <typename C, int U, bool STAGED, typename AG>
__device__ __forceinline__ void run_chunk_preloaded(
    const RolloutParams& p, const GroupView& v, AG& ag, EnvRegs& e, double* ring_smem,
    int64_t env, uint32_t gid, uint64_t step_base, int t0, int32_t* act,
    const int32_t* act_i, const double* zs = nullptr) {
  int32_t s0[U], k_tr[U];
  double u_tr[U], n_rw[U];
  IrrDraws<U> q;
#pragma unroll
  for (int j = 0; j < U; ++j) q.act[j] = act_i[j];
  phase_a<C, U, true, STAGED>(p, v, ag, env, gid, step_base, t0, U, act, u_tr,
                              k_tr, n_rw, s0, q, zs);
  phase_b<C, U, false>(p, v, ag, e, ring_smem, kBlock, env, t0, U, act, u_tr, k_tr,
                       n_rw, s0, q);
}

template <typename C, int U, bool STAGED, typename AG>
__device__ __forceinline__ void run_chunk(const RolloutParams& p,
                                          const GroupView& v, AG& ag, EnvRegs& e,
                                          double* ring_smem, int64_t env,
                                          uint32_t gid, uint64_t step_base, int t0,
                                          const double* zs = nullptr) {
  int32_t act[U], s0[U];
  int32_t k_tr[U];
  double u_tr[U], n_rw[U];
  IrrDraws<U> q;
  phase_a<C, U, false, STAGED>(p, v, ag, env, gid, step_base, t0, U, act, u_tr,
                               k_tr, n_rw, s0, q, zs);
  phase_b<C, U, false>(p, v, ag, e, ring_smem, kBlock, env, t0, U, act, u_tr, k_tr,
                       n_rw, s0, q);
}

// ---- staged ziggurat normals ------------------------------------------------
// The rejected first attempts (1.5 % of the draws) are what makes a ziggurat
// expensive on a SIMT machine: resolved where they occur, nearly every warp
// runs the ~170-instruction slow path for one or two lanes per chunk.  So the
// reward normals of kZigWindow steps are drawn AHEAD into shared memory
// (state-independent, like all draws of the Philox mode), the rejected ones of
// the whole warp (~15 of 1024) are pooled in a queue, and the warp resolves
// them side by side, one per lane: one pass per window.
#ifdef MDPP_ZIG_FILL_UNROLL
constexpr int kZigFillUnroll = MDPP_ZIG_FILL_UNROLL;
#else
constexpr int kZigFillUnroll = 4;  // pairs per unrolled body of zig_fill
#endif
struct ZigStage {
  double* zs;        // this thread's column: zs[k * kBlock] = window step k
  uint32_t* qcnt;    // per warp: number of queued items
  uint16_t* queue;   // per warp: items (owner lane << 8 | k)
  unsigned amask;    // the warp's lanes that own an environment
  int rank, n_act;   // this lane's rank among them, and their number
};

#ifdef MDPP_ZIG_FILL_NOINLINE
#define MDPP_ZIG_FILL_ATTR __noinline__
#else
#define MDPP_ZIG_FILL_ATTR __forceinline__
#endif
static __device__ MDPP_ZIG_FILL_ATTR void zig_fill(const RolloutParams& p, const GroupView& v,
                                         const ZigStage& zst, uint32_t gid,
                                         uint64_t g0,    // even global step
                                         int n_need) {   // steps the caller will read
  const int lane = threadIdx.x & 31;
  const uint8_t* zt = reinterpret_cast<const uint8_t*>(v.zig_kw);  // smem copy
  if (zst.rank == 0) *zst.qcnt = 0;
  __syncwarp(zst.amask);
  uint32_t rej = 0;
  const uint64_t pair0 = g0 >> 1;
  // (always a whole window: a compile-time trip count measured 9 % faster than
  // drawing only what the last window needs; launches shorter than a window
  // do not stage at all, see stage_of)
#ifdef MDPP_ZIG_FILL_DYN  // short launches: the last window only as far as it is read
  const int hb_end = min(kZigWindow / 2, (n_need + 1) / 2);
#else
  constexpr int hb_end = kZigWindow / 2;
#endif
#pragma unroll 1
  for (int hb = 0; hb < hb_end; hb += kZigFillUnroll) {
    uint32_t r8 = 0;
    double* zcol = zst.zs + 2 * hb * kBlock;
#pragma unroll
    for (int h = 0; h < kZigFillUnroll; ++h) {
      const uint64_t pr = pair0 + (uint64_t)(hb + h);
      const U4 w = philox4x32_10_rk(gid, (uint32_t)pr, (uint32_t)(pr >> 32),
                                    STREAM_ZIG, p.rk);
      bool ok0, ok1;
      const double z0 = zig_first(w.x, w.y, v.zig_kw, &ok0);
      const double z1 = zig_first(w.z, w.w, v.zig_kw, &ok1);
      // numpy: normal(0, sigma) = 0 + sigma * z
      zcol[(2 * h) * kBlock] = __dmul_rn(v.r_std, z0);
      zcol[(2 * h + 1) * kBlock] = __dmul_rn(v.r_std, z1);
      if (!ok0) r8 |= 1u << (2 * h);      // (immediates: one predicated LOP3)
      if (!ok1) r8 |= 2u << (2 * h);
    }
    rej |= r8 << (2 * hb);
  }
#ifdef MDPP_EXP_NO_SLOW  // (timing experiment: wrong normals, no slow path)
  rej = 0;
#endif
  uint32_t slot = 0;
  if (rej) slot = atomicAdd(zst.qcnt, (uint32_t)__popc(rej));
  while (rej) {
    const int k = __ffs((int)rej) - 1;
    rej &= rej - 1;
    if (slot < (uint32_t)kZigQueueCap)
      zst.queue[slot] = (uint16_t)((lane << 8) | k);
    else  // queue full (practically never): resolve it here
      zst.zs[k * kBlock] = __dmul_rn(v.r_std, zig_slow(gid, g0 + (uint64_t)k, p.rk, zt));
    ++slot;
  }
  __syncwarp(zst.amask);
  const int total = min((int)*zst.qcnt, kZigQueueCap);
  for (int i = zst.rank; i < total; i += zst.n_act) {
    const uint32_t item = zst.queue[i];
    const int owner = (int)(item >> 8), k = (int)(item & 0xffu);
    zst.zs[k * kBlock + owner - lane] = __dmul_rn(
        v.r_std, zig_slow(gid - (uint32_t)lane + (uint32_t)owner, g0 + (uint64_t)k,
                          p.rk, zt));
  }
  __syncwarp(zst.amask);
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

template <typename C, typename AG>
__device__ __forceinline__ void rollout_body(const RolloutParams& p, AG& ag) {
  // A kernel launched behind this one with programmatic stream serialisation
  // (the renderer, MDPP_LAUNCH_OVERLAP_PREVIOUS) may start its independent
  // prologue now; it still waits for this grid to finish before it reads the
  // states.  No effect otherwise.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  constexpr bool SMEM = C::SMEM;
  constexpr bool RING_SMEM = C::RING_SMEM;
  extern __shared__ __align__(16) uint8_t smem_dyn[];
  __shared__ DiscreteGroupDev grp;
  const CtaMapEntry me = p.cta_map[blockIdx.x];
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(p.groups + me.group);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&grp);
    for (int i = threadIdx.x; i < (int)(sizeof(DiscreteGroupDev) / 4); i += kBlock)
      dst[i] = src[i];
  }
  __syncthreads();
  const uint8_t* tab = p.blob + grp.blob_offset;
  // dynamic smem: [ring: p.ring_smem_bytes][tables]
  double* ring_smem = reinterpret_cast<double*>(smem_dyn) + threadIdx.x;
  if (SMEM) {
    uint8_t* smem_tab = smem_dyn + p.ring_smem_bytes;
    const uint4* src = reinterpret_cast<const uint4*>(tab);
    uint4* dst = reinterpret_cast<uint4*>(smem_tab);
    for (int i = threadIdx.x; i < grp.blob_bytes / 16; i += kBlock) dst[i] = src[i];
    __syncthreads();
    tab = smem_tab;
  }
  // ziggurat tables behind the ring and the group tables (SMEM builds; the
  // others -- short launches, oversized tables -- read them from global memory)
  const uint4* zig_kw = nullptr;
  if (C::NORMAL == MDPP_NORMAL_ZIGGURAT && C::NOISE == MDPP_NOISE_PHILOX) {
    if (SMEM) {
      uint4* dst = reinterpret_cast<uint4*>(smem_dyn + p.ring_smem_bytes +
                                            p.tab_smem_bytes);
      const uint4* src = reinterpret_cast<const uint4*>(p.zig);
      for (int i = threadIdx.x; i < kZigBytes / 16; i += kBlock) dst[i] = src[i];
      __syncthreads();
      zig_kw = dst;
    } else {
      zig_kw = reinterpret_cast<const uint4*>(p.zig);
    }
  }
  const GroupView v = make_view(C::SINGLE ? p.group0 : grp, tab, zig_kw);
  // Everything above read immutable tables only, so under a programmatic
  // dependent launch (discrete_launch.h, jit.cu) it overlapped the previous
  // kernel of the stream; wait for that kernel before touching the env state,
  // the actions, the device step counter or the outputs.  Returns at once in an
  // ordinary launch.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int64_t local = (int64_t)me.chunk * kBlock + threadIdx.x;
  const bool active = local < grp.env_count;
  constexpr bool ZIG = C::NORMAL == MDPP_NORMAL_ZIGGURAT && C::NOISE == MDPP_NOISE_PHILOX;
  ZigStage zst;
  if (ZIG && SMEM) {
    uint8_t* st = smem_dyn + p.ring_smem_bytes + p.tab_smem_bytes + kZigBytes;
    zst.zs = reinterpret_cast<double*>(st) + threadIdx.x;
    uint8_t* qb = st + kZigWindow * kBlock * 8 + (threadIdx.x >> 5) * kZigQueueBytes;
    zst.qcnt = reinterpret_cast<uint32_t*>(qb);
    zst.queue = reinterpret_cast<uint16_t*>(qb + 16);
    zst.amask = __ballot_sync(0xffffffffu, active);
    zst.rank = __popc(zst.amask & ((1u << (threadIdx.x & 31)) - 1u));
    zst.n_act = __popc(zst.amask);
  }
  const bool staged = ZIG && SMEM && v.has_rnoise && stage_of(p);
  const bool stage_path = ZIG && SMEM && stage_of(p);  // (group-independent)
  int zs_t0 = -kZigWindow;  // local step at which the staged window starts
  const int64_t env = grp.env_begin + (active ? local : 0);
  const int64_t N = n_envs_of(p);
  const DiscreteGroupDev& gsel = C::SINGLE ? p.group0 : grp;
  const uint32_t gid = (uint32_t)(p.env_id_offset + gsel.gid_base + (active ? local : 0));

  EnvRegs e;
  e.s = p.st.cur_state[env];
  e.key = p.st.seq_key[env];
  e.tl = p.st.t_episode[env];
  e.ep = p.st.episode[env];
  const bool irr = irr_of<C>(p);
  e.s_irr = irr ? p.st.cur_state_irr[env] : 0;
  e.phase = e.tl % v.every_n;
  // global index of the launch's first step (+ the optional device counter
  // that lets a captured CUDA graph advance between replays)
  const uint64_t step_base =
      p.step_index + (p.step_index_dev ? *p.step_index_dev : 0ull);
  e.ring_pos = v.delay > 0 ? (int32_t)(step_base % (uint64_t)v.delay) : 0;
  e.hist_pos = p.st.history
      ? (int32_t)((step_base + 1) % (uint64_t)p.st.history_depth) : 0;
  e.sum_reward = e.sum_abs_rnoise = 0.0;
  e.n_noisy = e.n_episodes = e.n_terminated = e.n_steps = 0;

  if (active) {
    ag.begin(v, env, e.s);
    // the value written j steps ago sits in ring slot (pos - j) mod d
    if (C::RING_REGS > 0) {
#pragma unroll
      for (int k = 0; k < C::RING_REGS; ++k) {
        const int slot = (e.ring_pos + 2 * C::RING_REGS - 1 - k) % C::RING_REGS;
        e.fifo[k] = p.st.ring[(int64_t)slot * N + env];
      }
    } else if (RING_SMEM) {
      for (int k = 0; k < v.delay; ++k)
        ring_smem[k * kBlock] = p.st.ring[(int64_t)k * N + env];
    }
    int t0 = 0;
    // chunks of kChunk steps start on a multiple-of-4 global step (the Philox
    // draws come in groups of 4 steps); peel single steps until aligned
    while (t0 < p.T && ((step_base + (uint64_t)t0) & 3)) {
      run_chunk<C, 1, false>(p, v, ag, e, ring_smem, env, gid, step_base, t0);
      ++t0;
    }
#ifdef MDPP_STAGGER
    // de-synchronise the warps of an SM: odd warps run a half chunk first
    if (kChunk > 4 && ((blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5)) & 1) &&
        t0 + 4 <= p.T) {
      run_chunk<C, 4, false>(p, v, ag, e, ring_smem, env, gid, step_base, t0);
      t0 += 4;
    }
#endif
    if (C::FAST) {
      // Action rows are fetched one chunk ahead: under a write-heavy DRAM
      // stream a read takes longer than phase A (ncu: 28 % of all stall
      // samples sat on the first use of an action), a whole chunk hides it.
      // The last prefetch re-reads the final chunk instead of branching.
      int32_t act_next[kChunk], act_next_i[kChunk];
      const int t_last = p.T - kChunk;  // start of the last possible chunk
#pragma unroll
      for (int j = 0; j < kChunk; ++j) act_next[j] = act_next_i[j] = 0;
      if (t0 <= t_last) {
#pragma unroll
        for (int j = 0; j < kChunk; ++j)
          load_action<C>(p, (int64_t)(t0 + j) * N + env, act_next[j], act_next_i[j]);
      }
      for (; t0 <= t_last; t0 += kChunk) {
        if (staged && t0 >= zs_t0 + kZigWindow) {
          zs_t0 = t0;
#ifndef MDPP_EXP_NO_FILL  // (timing experiment: stale normals)
          zig_fill(p, v, zst, gid, step_base + (uint64_t)t0,
                   (p.T - t0) / kChunk * kChunk);
#endif
        }
        int32_t act[kChunk], act_i[kChunk];
        const int tn = min(t0 + kChunk, t_last);
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
          act[j] = act_next[j];
          act_i[j] = act_next_i[j];
          load_action<C>(p, (int64_t)(tn + j) * N + env, act_next[j], act_next_i[j]);
        }
        if (stage_path)
          run_chunk_preloaded<C, kChunk, ZIG && SMEM>(p, v, ag, e, ring_smem, env, gid,
                                                      step_base, t0, act, act_i,
                                                      zst.zs + (t0 - zs_t0) * kBlock);
        else
          run_chunk_preloaded<C, kChunk, false>(p, v, ag, e, ring_smem, env, gid,
                                                step_base, t0, act, act_i);
      }
    } else {
      for (; t0 + kChunk <= p.T; t0 += kChunk) {
        if (staged && t0 >= zs_t0 + kZigWindow) {
          zs_t0 = t0;
          zig_fill(p, v, zst, gid, step_base + (uint64_t)t0,
                   (p.T - t0) / kChunk * kChunk);
        }
        if (stage_path)
          run_chunk<C, kChunk, ZIG && SMEM>(p, v, ag, e, ring_smem, env, gid, step_base, t0,
                                            zst.zs + (t0 - zs_t0) * kBlock);
        else
          run_chunk<C, kChunk, false>(p, v, ag, e, ring_smem, env, gid, step_base, t0);
      }
    }
    // remainder: a half chunk first (t0 is still quad-aligned here; single
    // steps pay a whole Philox quad each), then single steps
    if (kChunk > 4)
      for (; t0 + 4 <= p.T; t0 += 4)
        run_chunk<C, 4, false>(p, v, ag, e, ring_smem, env, gid, step_base, t0);
    for (; t0 < p.T; ++t0)
      run_chunk<C, 1, false>(p, v, ag, e, ring_smem, env, gid, step_base, t0);
    p.st.cur_state[env] = e.s;
    if (irr) p.st.cur_state_irr[env] = e.s_irr;
    p.st.seq_key[env] = e.key;
    p.st.t_episode[env] = e.tl;
    p.st.episode[env] = e.ep + e.n_episodes;
    ag.end(env);
    if (C::RING_REGS > 0) {
      const int pos_end = (int)((step_base + (uint64_t)p.T) % (uint64_t)C::RING_REGS);
#pragma unroll
      for (int k = 0; k < C::RING_REGS; ++k) {
        const int slot = (pos_end + 2 * C::RING_REGS - 1 - k) % C::RING_REGS;
        p.st.ring[(int64_t)slot * N + env] = e.fifo[k];
      }
    } else if (RING_SMEM) {
      for (int k = 0; k < v.delay; ++k)
        p.st.ring[(int64_t)k * N + env] = ring_smem[k * kBlock];
    }
  }
  if (p.st.stats) {
    double vals[MDPP_N_STATS];
    vals[MDPP_STAT_EPISODES] = (double)e.n_episodes;
    vals[MDPP_STAT_TRANSITIONS] = (double)e.n_steps;
    vals[MDPP_STAT_REWARD] = e.sum_reward;
    vals[MDPP_STAT_NOISY_TRANSITIONS] = (double)e.n_noisy;
    vals[MDPP_STAT_ABS_REWARD_NOISE] = e.sum_abs_rnoise;
    vals[MDPP_STAT_ABS_TRANSITION_NOISE] = 0.0;
    vals[MDPP_STAT_RESERVED] = 0.0;
    vals[MDPP_STAT_TERMINATED] = (double)e.n_terminated;
    // warps spread their atomics over the `stats_slots` copies of the rows
    const int n_slots = max(p.st.stats_slots, 1);
    const int slot = (int)((blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5)) % (unsigned)n_slots);
    double* row = p.st.stats + ((int64_t)slot * p.n_groups + me.group) * MDPP_N_STATS;
#pragma unroll
    for (int k = 0; k < MDPP_N_STATS; ++k) {
      if (k == MDPP_STAT_ABS_TRANSITION_NOISE || k == MDPP_STAT_RESERVED) continue;
      double s = warp_sum(active ? vals[k] : 0.0);
      if ((threadIdx.x & 31) == 0 && s != 0.0) atomicAdd(row + k, s);
    }
  }
}

template <typename C>
__device__ __forceinline__ void rollout_body(const RolloutParams& p) {
  NoAgent ag;
  rollout_body<C>(p, ag);
}

template <typename C>
__global__ void __launch_bounds__(kBlock, kMinBlocksPerSM)
discrete_rollout_kernel(const __grid_constant__ RolloutParams p) {
  rollout_body<C>(p);
}

}  // namespace mdpp
