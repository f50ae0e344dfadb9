// Continuous RLToyEnv step path ("move_to_a_point") on sm_100a: K3
// `continuous_rollout` (T fused steps; T = 1 is the gym-style step) and the
// continuous reset.  Device-only header, also compiled by NVRTC (jit.cu) with
// the configuration as literals (MDPP_JIT): dim / order / relevant indices
// become compile-time, every per-dimension loop unrolls and the whole state
// ((order+1) x dim derivatives + the emitted state) lives in registers.  The
// ahead-of-time build keeps them as run-time values (arrays in local memory):
// a correct but slow fallback for hosts without NVRTC.
//
// Restates (per env, per step) rl_toy_env.py
//   transition_function :1625-1725  Taylor update of state_derivatives in the
//        reference's exact dtype path: (f32 * f32(tu^k)) -> / f64 factorial
//        -> += rounds back to f32; frozen state on an out-of-range action;
//        noise added to the emitted state only; clip => all derivatives
//        zeroed; sticky reached_terminal inside target_radius
//   reward_function :1912-1945 dense / sparse move_to_a_point, action loss,
//        :1968-1990 delay FIFO, every-n gate, noise, scale, shift -- including
//        numpy's scalar typing: the reward is np.float32 except when it comes
//        from the zero-initialised FIFO or the every-n gate (python float),
//        in which case the tail runs in double
//   step epilogue :2098-2109, reset :2284-2323
//
// One thread = one environment.  State is struct-of-arrays ([component][N],
// coalesced); actions / observations use the gym layout ([N][dim] rows).
// No FMA contraction anywhere on the parity path (explicit _rn intrinsics).
#pragma once
#include "device_types.h"
#include "philox.cuh"
#include "ziggurat.cuh"

namespace mdpp {

constexpr int kCBlock = 128;

struct ContinuousParams {
  mdpp_continuous_config cfg;
  double tu_pow[MDPP_MAX_ORDER];  // time_unit ** (j + 1), computed by the host
  mdpp_continuous_state st;
  mdpp_continuous_io io;
  int32_t T, autoreset, horizon, noise_mode;
  int32_t normal_mode, reserved0;  // MDPP_NORMAL_*: ziggurat / Box-Muller in fp64 / on the SFU
  const uint8_t* zig;              // the context's ziggurat tables (ziggurat.cuh layout)
  uint32_t k0, k1;
  uint32_t rk[20];  // Philox round keys expanded from (k0, k1) by the host
  uint64_t step_index;
  const uint64_t* step_index_dev;
  int64_t env_id_offset;
  // reset kernel only
  const uint8_t* mask;
  const void* init_states;
  void* reset_obs;
  // heterogeneous launches (mdpp_set_continuous_groups): CTA -> (group, chunk
  // of kCBlock envs); every CTA reads its group's configuration from `groups`.
  // NULL / 0 for the single-configuration launch (cfg / tu_pow above).
  const struct ContinuousGroupDev* groups;
  const CtaMapEntry* cta_map;
  int32_t n_groups, reserved1;
};

// One configuration group of a heterogeneous continuous launch: the groups
// share dim / order / relevant indices / dtype (the state arrays' shape) and
// differ in their scalars.
struct ContinuousGroupDev {
  mdpp_continuous_config cfg;
  double tu_pow[MDPP_MAX_ORDER];
  int64_t env_begin, env_count, gid_base;
};

template <typename R> struct RealOps;
template <> struct RealOps<float> {
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
  static __device__ __forceinline__ float sqrt(float a) { return __fsqrt_rn(a); }
};
template <> struct RealOps<double> {
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
  static __device__ __forceinline__ double sqrt(double a) { return __dsqrt_rn(a); }
};

#ifdef MDPP_JIT
#define MDPP_C_CONST(name, runtime) (MDPP_C_##name)
// double constants travel as their bit pattern (exact, inf-safe)
#define MDPP_C_F64(name, runtime) (__longlong_as_double(MDPP_C_##name##_BITS))
#else
#define MDPP_C_CONST(name, runtime) (runtime)
#define MDPP_C_F64(name, runtime) (runtime)
#endif

// relevant_indices[k]: a literal table in the specialised build so that
// indexing the register-resident state with it stays static.
__device__ __forceinline__ int rel_index(const mdpp_continuous_config& cfg, int k) {
#ifdef MDPP_JIT
  constexpr int kRel[MDPP_MAX_DIM] = {
      MDPP_C_REL0, MDPP_C_REL1, MDPP_C_REL2, MDPP_C_REL3, MDPP_C_REL4, MDPP_C_REL5,
      MDPP_C_REL6, MDPP_C_REL7, MDPP_C_REL8, MDPP_C_REL9, MDPP_C_REL10,
      MDPP_C_REL11, MDPP_C_REL12, MDPP_C_REL13, MDPP_C_REL14, MDPP_C_REL15};
  return kRel[k];
#else
  return cfg.relevant_indices[k];
#endif
}

// a / inertia (:1655).  For inertia = 2^k the product with 2^-k is the same
// correctly rounded value as the quotient, without the IEEE division's ~15
// instructions and slow-path branch; a literal inertia folds the test away.
__device__ __forceinline__ float div_inertia(float a, float inertia) {
  const float inv = 1.0f / inertia;  // (plain operator: folds for a literal)
  const uint32_t bi = __float_as_uint(inertia), bv = __float_as_uint(inv);
  const bool pow2 = (bi & 0x7FFFFFu) == 0 && (bv & 0x7FFFFFu) == 0 &&
                    ((bi >> 23) & 0xFF) != 0 && ((bi >> 23) & 0xFF) != 0xFF &&
                    ((bv >> 23) & 0xFF) != 0 && ((bv >> 23) & 0xFF) != 0xFF;
  return pow2 ? __fmul_rn(a, inv) : __fdiv_rn(a, inertia);
}
__device__ __forceinline__ double div_inertia(double a, double inertia) {
  const double inv = 1.0 / inertia;
  const uint64_t bi = (uint64_t)__double_as_longlong(inertia);
  const uint64_t bv = (uint64_t)__double_as_longlong(inv);
  const uint64_t man = 0xFFFFFFFFFFFFFull;
  const bool pow2 = (bi & man) == 0 && (bv & man) == 0 &&
                    ((bi >> 52) & 0x7FF) != 0 && ((bi >> 52) & 0x7FF) != 0x7FF &&
                    ((bv >> 52) & 0x7FF) != 0 && ((bv >> 52) & 0x7FF) != 0x7FF;
  return pow2 ? __dmul_rn(a, inv) : __ddiv_rn(a, inertia);
}

// One [dim] row of the gym-layout action / observation arrays.  The
// specialised build knows dim, so rows move as 16- or 8-byte vectors when the
// row size allows (the C entry points require 16-byte aligned I/O buffers).
template <typename R>
__device__ __forceinline__ void load_row(const R* src, int D, R* out) {
#ifdef MDPP_JIT
  constexpr int kD = MDPP_C_DIM;
  constexpr int kVec = (kD * sizeof(R)) % 16 == 0 ? 16 / sizeof(R)
                     : (kD * sizeof(R)) % 8 == 0 ? 8 / sizeof(R) : 1;
  if (kVec == 4) {
#pragma unroll
    for (int d = 0; d < kD; d += 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(src + d));
      out[d] = (R)v.x; out[d + 1] = (R)v.y; out[d + 2] = (R)v.z; out[d + 3] = (R)v.w;
    }
    return;
  }
  if (kVec == 2 && sizeof(R) == 4) {
#pragma unroll
    for (int d = 0; d < kD; d += 2) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(src + d));
      out[d] = (R)v.x; out[d + 1] = (R)v.y;
    }
    return;
  }
  if (kVec == 2 && sizeof(R) == 8) {
#pragma unroll
    for (int d = 0; d < kD; d += 2) {
      const double2 v = __ldg(reinterpret_cast<const double2*>(src + d));
      out[d] = (R)v.x; out[d + 1] = (R)v.y;
    }
    return;
  }
#endif
#pragma unroll
  for (int d = 0; d < MDPP_MAX_DIM; ++d)
    if (d < D) out[d] = src[d];
}

template <typename R>
__device__ __forceinline__ void store_row(R* dst, int D, const R* v) {
#ifdef MDPP_JIT
  constexpr int kD = MDPP_C_DIM;
  constexpr int kVec = (kD * sizeof(R)) % 16 == 0 ? 16 / sizeof(R)
                     : (kD * sizeof(R)) % 8 == 0 ? 8 / sizeof(R) : 1;
  if (kVec == 4) {
#pragma unroll
    for (int d = 0; d < kD; d += 4)
      *reinterpret_cast<float4*>(dst + d) =
          make_float4((float)v[d], (float)v[d + 1], (float)v[d + 2], (float)v[d + 3]);
    return;
  }
  if (kVec == 2 && sizeof(R) == 4) {
#pragma unroll
    for (int d = 0; d < kD; d += 2)
      *reinterpret_cast<float2*>(dst + d) = make_float2((float)v[d], (float)v[d + 1]);
    return;
  }
  if (kVec == 2 && sizeof(R) == 8) {
#pragma unroll
    for (int d = 0; d < kD; d += 2)
      *reinterpret_cast<double2*>(dst + d) = make_double2((double)v[d], (double)v[d + 1]);
    return;
  }
#endif
#pragma unroll
  for (int d = 0; d < MDPP_MAX_DIM; ++d)
    if (d < D) dst[d] = v[d];
}

// np.linalg.norm of a short vector: sqrt of the sequentially accumulated,
// separately rounded sum of squares (bit-identical to numpy/OpenBLAS for the
// 1- and 2-element vectors that move_to_a_point uses; see DESIGN.md).
template <typename R, typename F>
__device__ __forceinline__ R seq_norm(int n, F elem) {
  R s = 0;
#pragma unroll
  for (int k = 0; k < MDPP_MAX_DIM; ++k)
    if (k < n) {
      R x = elem(k);
      s = RealOps<R>::add(s, RealOps<R>::mul(x, x));
    }
  return RealOps<R>::sqrt(s);
}

// Philox Box sample of one env (gymnasium Box.sample: uniform in [-max, max]
// when bounded, N(0,1) when unbounded, cast to dtype_s).
template <typename R>
__device__ __forceinline__ void box_sample(const ContinuousParams& p,
                                           const mdpp_continuous_config& cfg, int D,
                                           uint32_t gid, uint32_t ep,
                                           int attempt, R* out) {
  const bool bounded = isfinite(cfg.state_space_max);
  const double hi = (double)(R)cfg.state_space_max, lo = -hi;
#pragma unroll
  for (int c = 0; c < MDPP_MAX_DIM / 2; ++c) {
    if (2 * c < D) {
      U4 w = philox4x32_10(gid, ep, (uint32_t)attempt,
                           STREAM_RESET_BOX + (uint32_t)c, p.k0, p.k1);
      double v0, v1;
      if (bounded) {
        v0 = lo + (hi - lo) * uniform53(w.x, w.y);
        v1 = lo + (hi - lo) * uniform53(w.z, w.w);
      } else {
        normal_pair_f64(w.x, w.y, &v0, &v1);
      }
      out[2 * c] = (R)v0;
      if (2 * c + 1 < D) out[2 * c + 1] = (R)v1;
    }
  }
}

template <typename R>
__device__ __forceinline__ bool in_term_box(const mdpp_continuous_config& cfg, int NREL,
                                            const R* x /* full state */) {
  bool any = false;
  for (int b = 0; b < cfg.n_term_boxes; ++b) {
    bool in = true;
#pragma unroll
    for (int k = 0; k < MDPP_MAX_DIM; ++k)
      if (k < NREL) {
        const R v = x[rel_index(cfg, k)];
        in = in && v >= (R)cfg.term_low[b * MDPP_MAX_DIM + k] &&
             v <= (R)cfg.term_high[b * MDPP_MAX_DIM + k];
      }
    any = any || in;
  }
  return any;
}

template <typename R> struct RowVal { R v[MDPP_MAX_DIM]; };

// Initial state of a new episode (:2284-2323): Box sample, rejected while it
// falls into a terminal box.  Rare and big (Philox + fp64), so out of line;
// the row comes back by value and the caller's state stays in registers.
template <typename R>
__device__ __noinline__ RowVal<R> sample_reset_state(const ContinuousParams& p,
                                                     const mdpp_continuous_config& cfg,
                                                     int D, int NREL, int NBOX,
                                                     uint32_t gid, uint32_t ep) {
  RowVal<R> s0;
#pragma unroll 1
  for (int attempt = 0; attempt < 64; ++attempt) {
    box_sample<R>(p, cfg, D, gid, ep, attempt, s0.v);
    if (!(NBOX > 0 && in_term_box<R>(cfg, NREL, s0.v))) break;
  }
  return s0;
}

#ifdef MDPP_C_PREFETCH  // tuning override of the NVRTC build
constexpr int kActionPrefetch = MDPP_C_PREFETCH;
#else
constexpr int kActionPrefetch = 4;  // action rows in flight per env
#endif

// ---- move_along_a_line (rl_toy_env.py:1865-1910, :2546-2576) ----------------
// Reward = - (1 / L) sum of the distances of the last L emitted relevant states
// from the line fitted through them.  The reference takes the direction from a
// float32 SVD (numpy / LAPACK sgesdd) of the centred window and does
// everything after it in float64 (the end points are a float64 linspace times
// the direction).  Here: window mean in R with numpy's summation order (the
// reference's window is F-ordered, so `mean(axis=0)` runs the pairwise sum:
// sequential below 8 rows, 8 accumulators up to 128), principal direction from
// the float64 covariance (closed form for 2 relevant dimensions, cyclic Jacobi
// above), rounded to R like the SVD's output, distances by the reference's
// Pythagoras formula in float64.  Agreement with the reference is bounded by
// the fp32 direction (~1e-7 relative): the contract's 1e-5, not bit-exactness.
constexpr int kLineMaxSeq = 128;

template <typename R>
__device__ __noinline__ double line_reward(const R* hist, int64_t N, int64_t env,
                                           int NREL, int L, uint64_t step) {
  typedef RealOps<R> O;
  auto row = [&](int k) { return (int)((step + 1 + (uint64_t)k) % (uint64_t)L); };
  auto at = [&](int k, int d) { return hist[((int64_t)row(k) * NREL + d) * N + env]; };
  R mean[MDPP_MAX_DIM];
  for (int d = 0; d < NREL; ++d) {
    R s;
    if (L < 8) {
      s = (R)0;
      for (int k = 0; k < L; ++k) s = O::add(s, at(k, d));
    } else {  // numpy pairwise_sum for 8 <= n <= 128
      R r[8];
      for (int j = 0; j < 8; ++j) r[j] = at(j, d);
      int i = 8;
      for (; i < L - (L % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] = O::add(r[j], at(i + j, d));
      s = O::add(O::add(O::add(r[0], r[1]), O::add(r[2], r[3])),
                 O::add(O::add(r[4], r[5]), O::add(r[6], r[7])));
      for (; i < L; ++i) s = O::add(s, at(i, d));
    }
    mean[d] = (R)((double)s / (double)L);  // true_divide in float64, cast back
  }
  // covariance of the centred (R-rounded) window, float64
  double C[MDPP_MAX_DIM][MDPP_MAX_DIM];
  for (int a = 0; a < NREL; ++a)
    for (int b = 0; b < NREL; ++b) C[a][b] = 0.0;
  for (int k = 0; k < L; ++k) {
    double c[MDPP_MAX_DIM];
    for (int d = 0; d < NREL; ++d) c[d] = (double)O::add(at(k, d), -mean[d]);
    for (int a = 0; a < NREL; ++a)
      for (int b = a; b < NREL; ++b) C[a][b] += c[a] * c[b];
  }
  double v[MDPP_MAX_DIM];
  for (int d = 0; d < NREL; ++d) v[d] = d == 0 ? 1.0 : 0.0;
  if (NREL == 2) {
    const double th = 0.5 * atan2(2.0 * C[0][1], C[0][0] - C[1][1]);
    if (C[0][1] != 0.0 || C[0][0] != C[1][1]) { v[0] = cos(th); v[1] = sin(th); }
  } else if (NREL > 2) {
    double V[MDPP_MAX_DIM][MDPP_MAX_DIM];
    for (int a = 0; a < NREL; ++a)
      for (int b = 0; b < NREL; ++b) {
        V[a][b] = a == b ? 1.0 : 0.0;
        if (b < a) C[a][b] = C[b][a];
      }
    for (int sweep = 0; sweep < 12; ++sweep) {
      double off = 0.0;
      for (int a = 0; a < NREL; ++a)
        for (int b = a + 1; b < NREL; ++b) off += C[a][b] * C[a][b];
      if (off == 0.0) break;
      for (int pi = 0; pi < NREL; ++pi)
        for (int q = pi + 1; q < NREL; ++q) {
          if (C[pi][q] == 0.0) continue;
          const double tau = (C[q][q] - C[pi][pi]) / (2.0 * C[pi][q]);
          const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
          const double cs = 1.0 / sqrt(1.0 + t * t), sn = t * cs;
          for (int k = 0; k < NREL; ++k) {
            const double akp = C[k][pi], akq = C[k][q];
            C[k][pi] = cs * akp - sn * akq;
            C[k][q] = sn * akp + cs * akq;
          }
          for (int k = 0; k < NREL; ++k) {
            const double apk = C[pi][k], aqk = C[q][k];
            C[pi][k] = cs * apk - sn * aqk;
            C[q][k] = sn * apk + cs * aqk;
          }
          for (int k = 0; k < NREL; ++k) {
            const double vkp = V[k][pi], vkq = V[k][q];
            V[k][pi] = cs * vkp - sn * vkq;
            V[k][q] = sn * vkp + cs * vkq;
          }
        }
    }
    int best = 0;
    for (int a = 1; a < NREL; ++a)
      if (C[a][a] > C[best][best]) best = a;
    for (int d = 0; d < NREL; ++d) v[d] = V[d][best];
  }
  // the reference's float64 distance arithmetic on the R-typed direction / mean
  double A[MDPP_MAX_DIM], AB[MDPP_MAX_DIM];
  double nAB2 = 0.0;
  for (int d = 0; d < NREL; ++d) {
    const double vd = (double)(R)v[d], md = (double)mean[d];
    A[d] = __dadd_rn(-vd, md);                       // vv[0] * -1 + mean
    AB[d] = __dadd_rn(A[d], -__dadd_rn(vd, md));     // ptA - ptB
    nAB2 = __dadd_rn(nAB2, __dmul_rn(AB[d], AB[d]));
  }
  const double nAB = sqrt(nAB2);
  double total = 0.0;
  if (!(nAB < 1e-13)) {
    for (int k = 0; k < L; ++k) {
      double dot = 0.0, n2 = 0.0;
      for (int d = 0; d < NREL; ++d) {
        const double ap = __dadd_rn(A[d], -(double)at(k, d));
        dot = __dadd_rn(dot, __dmul_rn(AB[d], ap));
        n2 = __dadd_rn(n2, __dmul_rn(ap, ap));
      }
      const double proj = __ddiv_rn(dot, nAB), nap = sqrt(n2);
      double sq = __dadd_rn(__dmul_rn(nap, nap), -__dmul_rn(proj, proj));
      if (sq < 0.0) sq = 0.0;
      total = __dadd_rn(total, sqrt(sq));
    }
  }
  return __dadd_rn(0.0, __ddiv_rn(-total, (double)L));
}

// The configuration a thread works under: the launch's (kernel parameters,
// constant bank) or, in a heterogeneous launch, its CTA's group staged in
// shared memory, with the env range and Philox id base of that group.
struct ContinuousGroupSel {
  int64_t env;      // index into the state arrays
  int64_t local;    // index inside the group
  uint32_t gid;
  bool active;
  int group;
};

// (shared-memory copy of the CTA's group; empty in single-configuration builds)
template <bool G> struct GroupSmem { ContinuousGroupDev g; };
template <> struct GroupSmem<false> { int unused; };
__device__ __forceinline__ ContinuousGroupDev* group_ptr(GroupSmem<true>& s) { return &s.g; }
__device__ __forceinline__ ContinuousGroupDev* group_ptr(GroupSmem<false>&) { return nullptr; }

template <bool GROUPS>
__device__ __forceinline__ ContinuousGroupSel select_group(
    const ContinuousParams& p, ContinuousGroupDev* gsm, int64_t N) {
  ContinuousGroupSel s;
  if (GROUPS) {
    const CtaMapEntry me = p.cta_map[blockIdx.x];
    const uint32_t* src = reinterpret_cast<const uint32_t*>(p.groups + me.group);
    uint32_t* dst = reinterpret_cast<uint32_t*>(gsm);
    for (int i = threadIdx.x; i < (int)(sizeof(ContinuousGroupDev) / 4); i += kCBlock)
      dst[i] = src[i];
    __syncthreads();
    s.local = (int64_t)me.chunk * kCBlock + threadIdx.x;
    s.active = s.local < gsm->env_count;
    s.env = gsm->env_begin + (s.active ? s.local : 0);
    s.gid = (uint32_t)(p.env_id_offset + gsm->gid_base + (s.active ? s.local : 0));
    s.group = me.group;
  } else {
    const int64_t env_raw = (int64_t)blockIdx.x * kCBlock + threadIdx.x;
    s.active = env_raw < N;
    s.env = s.active ? env_raw : 0;
    s.local = s.env;
    s.gid = (uint32_t)(p.env_id_offset + s.env);
    s.group = 0;
  }
  return s;
}

// The rollout takes its actions from the action rows (NoContinuousAgent) or
// from an agent (ArsAgent, ars.cu), which loads its per-env state at launch
// begin (every thread of the CTA takes part), provides each step's action
// from the state the env last emitted, sees each step's returned reward,
// termination and truncation, and stores its state at launch end.  The agent
// also names the kernel's parameter struct.
struct NoContinuousAgent {
  static constexpr bool kActs = false;
  using Params = ContinuousParams;
  __device__ __forceinline__ explicit NoContinuousAgent(const ContinuousParams&) {}
};

template <typename R, int NOISE, bool GROUPS = false, typename AG = NoContinuousAgent>
__device__ __forceinline__ void continuous_body(const typename AG::Params& p) {
  using O = RealOps<R>;
  AG ag(p);
  __shared__ GroupSmem<GROUPS> gsm_store;
  ContinuousGroupDev* gsm = group_ptr(gsm_store);
  const int64_t N = MDPP_C_CONST(N_ENVS, p.st.n_envs);
  const ContinuousGroupSel sel = select_group<GROUPS>(p, gsm, N);
  const mdpp_continuous_config& cfg = GROUPS ? gsm->cfg : p.cfg;
  const double* tu_rt = GROUPS ? gsm->tu_pow : p.tu_pow;
  const int D = MDPP_C_CONST(DIM, cfg.dim);
  const int ORDER = MDPP_C_CONST(ORDER, cfg.order);
  const int NREL = MDPP_C_CONST(NREL, cfg.n_relevant);
  const int DELAY = MDPP_C_CONST(DELAY, cfg.delay);
  const int EVERY_N = MDPP_C_CONST(EVERY_N, cfg.reward_every_n_steps);
  const bool DENSE = MDPP_C_CONST(DENSE, cfg.dense != 0);
  const bool PNOISE = MDPP_C_CONST(PNOISE, cfg.has_transition_noise != 0);
  const bool RNOISE = MDPP_C_CONST(RNOISE, cfg.has_reward_noise != 0);
  const bool IMAGE = MDPP_C_CONST(IMAGE, cfg.image_mode != 0);
  const bool TARGET64 = MDPP_C_CONST(TARGET64, cfg.target_is_f64 != 0);
  // launch shape: literals in the specialised build.  FAST = the standard
  // rollout signature (obs, reward, terminated, truncated written, no
  // final_obs), so no per-step NULL tests survive in the loop.
  const int NBOX = MDPP_C_CONST(NBOX, cfg.n_term_boxes);
  const int HORIZON = MDPP_C_CONST(HORIZON, p.horizon);
  const bool AUTORESET = MDPP_C_CONST(AUTORESET, p.autoreset != 0);
  const bool FAST = MDPP_C_CONST(FAST, false);
  const bool FAST_NORMAL = MDPP_C_CONST(NORMAL, p.normal_mode) == MDPP_NORMAL_FAST;
  // numpy's Generator.normal algorithm (what the reference's noise calls run,
  // rl_toy_env.py:413 via :1683, :403 via :1982) on Philox words.  Opt-in for this kernel
  // (normal_precision="ziggurat"): with 7 normals per step the direct draws
  // below measured 5.6 ms against 4.3 ms with fp64 Box-Muller (1 M envs x 100
  // steps, D = 6) -- twice the Philox calls and an out-of-line slow path; the
  // staged design of the discrete rollout kernel has not been ported here
  const bool ZIG_NORMAL = MDPP_C_CONST(NORMAL, p.normal_mode) == MDPP_NORMAL_ZIGGURAT;
  const bool active = sel.active;
  const int64_t env = sel.env;
  const uint32_t gid = sel.gid;

  const R amax = (R)MDPP_C_F64(AMAX, cfg.action_space_max);
  const R smax = (R)MDPP_C_F64(SMAX, cfg.state_space_max);
  const R inertia = (R)MDPP_C_F64(INERTIA, cfg.inertia);
  const int IMODE = MDPP_C_CONST(IMODE, cfg.inertia_mode);  // per-dimension inertia
  const bool LINE = MDPP_C_CONST(LINE, cfg.reward_kind == MDPP_REWARD_LINE);
  const int SEQ = MDPP_C_CONST(SEQ, cfg.sequence_length);
  const double radius64 = MDPP_C_F64(RADIUS, cfg.target_radius);
  const R radius_r = (R)radius64;
  const double alw = MDPP_C_F64(ALW, cfg.action_loss_weight);
  const double r_scale = MDPP_C_F64(SCALE, cfg.reward_scale);
  const double r_shift = MDPP_C_F64(SHIFT, cfg.reward_shift);
  const double term_add = MDPP_C_F64(
      TERM_ADD, __dmul_rn(cfg.term_state_reward, cfg.reward_scale));
  const double p_std = MDPP_C_F64(P_STD, cfg.transition_noise_std);
  const double r_std = MDPP_C_F64(R_STD, cfg.reward_noise_std);
  const double tu_pow[MDPP_MAX_ORDER] = {
      MDPP_C_F64(TU1, tu_rt[0]), MDPP_C_F64(TU2, tu_rt[1]),
      MDPP_C_F64(TU3, tu_rt[2]), MDPP_C_F64(TU4, tu_rt[3])};

  R sd[MDPP_MAX_ORDER + 1][MDPP_MAX_DIM];
  R em[MDPP_MAX_DIM];
  R* derivs = reinterpret_cast<R*>(p.st.derivs);
  R* emitted = reinterpret_cast<R*>(p.st.emitted);
  R* ring = reinterpret_cast<R*>(p.st.ring);
#pragma unroll
  for (int k = 0; k <= MDPP_MAX_ORDER; ++k)
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (k <= ORDER && d < D) sd[k][d] = derivs[((int64_t)k * D + d) * N + env];
#pragma unroll
  for (int d = 0; d < MDPP_MAX_DIM; ++d)
    if (d < D) em[d] = emitted[(int64_t)d * N + env];
  int32_t tl = p.st.t_episode[env];
  uint32_t ep = p.st.episode[env];
  bool reached = p.st.reached[env] != 0;
  int32_t phase = tl % EVERY_N;
  const uint64_t step_base =
      p.step_index + (p.step_index_dev ? *p.step_index_dev : 0ull);
  int32_t ring_pos = DELAY > 0 ? (int32_t)(step_base % (uint64_t)DELAY) : 0;

  double sum_reward = 0, sum_abs_rnoise = 0, sum_abs_pnoise = 0;
  uint32_t n_episodes = 0, n_terminated = 0;
  if constexpr (AG::kActs) ag.begin(sel, cfg, D);
  if (active) {

  // distance of a state's relevant part to the target, in the dtype numpy
  // would use: R when target_point was given (cast to dtype_s :646), float64
  // for the default float64 zeros (:654)
  auto dist_to_target = [&](const R* x) -> double {
    if (LINE) return 0.0;  // (no target point)
    if (TARGET64) {
      return seq_norm<double>(NREL, [&](int k) {
        return __dadd_rn((double)x[rel_index(cfg, k)], -cfg.target_point[k]);
      });
    }
    return (double)seq_norm<R>(NREL, [&](int k) {
      return O::add(x[rel_index(cfg, k)], -(R)cfg.target_point[k]);
    });
  };

  // ||aug[-2][rel] - target||: the distance of the previous emitted state is
  // last step's dist_new, so it is carried instead of recomputed
  double dist_prev = dist_to_target(em);
  // Action rows are fetched kActionPrefetch steps ahead of their use, into a
  // register ring indexed statically (the time loop is unrolled by the ring
  // size): under a write-heavy DRAM stream a read takes several step times.
  // (with fp64 Box-Muller noise the body is too big to unroll: the
  // instruction cache would thrash; the generic build keeps one row as well)
#ifdef MDPP_JIT
  constexpr int PF = (MDPP_C_NOISE != MDPP_NOISE_OFF && (MDPP_C_PNOISE || MDPP_C_RNOISE) &&
                      MDPP_C_NORMAL != MDPP_NORMAL_FAST) ? 1 : kActionPrefetch;
#else
  constexpr int PF = 1;
#endif
  R abuf[PF][MDPP_MAX_DIM];
#pragma unroll
  for (int u = 0; u < PF; ++u)
    if (!AG::kActs && u < p.T)
      load_row<R>(reinterpret_cast<const R*>(p.io.actions) + ((int64_t)u * N + env) * D,
                  D, abuf[u]);
  auto one_step = [&](const int t, R* a_slot) {
    const uint64_t step = step_base + (uint64_t)t;
    const int64_t row = ((int64_t)t * N + env);
    R a[MDPP_MAX_DIM], nxt[MDPP_MAX_DIM];
    bool in_range = true;
    if constexpr (AG::kActs) ag.act(em, D, amax, row, a_slot);
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (d < D) {
        a[d] = a_slot[d];
        in_range = in_range && a[d] >= -amax && a[d] <= amax;  // Box.contains
      }
    if (!AG::kActs && t + PF < p.T)
      load_row<R>(reinterpret_cast<const R*>(p.io.actions) + (row + (int64_t)PF * N) * D,
                  D, a_slot);
    const double dist_old = dist_prev;

    // ---- transition -----------------------------------------------------
    if (in_range) {
      // top derivative = action / inertia (:1654).  A list / float64-array
      // inertia (IMODE 2, fp32 env) promotes it to float64: kept in top64 for
      // the Taylor terms that read it, stored rounded to dtype_s
      double top64[MDPP_MAX_DIM];
      const bool TOP64 = IMODE == 2 && sizeof(R) == 4;
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) {
          if (IMODE == 0) {
            sd[ORDER][d] = div_inertia(a[d], inertia);
          } else if (!TOP64) {
            sd[ORDER][d] = O::div(a[d], (R)cfg.inertia_vec[d]);
          } else {
            top64[d] = __ddiv_rn((double)a[d], cfg.inertia_vec[d]);
            sd[ORDER][d] = (R)top64[d];
          }
        }
#pragma unroll
      for (int i = 0; i < MDPP_MAX_ORDER; ++i)
#pragma unroll
        for (int j = 0; j < MDPP_MAX_ORDER; ++j)
          if (i < ORDER && j < ORDER - i) {
            const R tu = (R)tu_pow[j];
            // (j+1)! as the float64 scipy.special.factorial returns
            const double fact = j == 0 ? 1.0 : j == 1 ? 2.0 : j == 2 ? 6.0 : 24.0;
#pragma unroll
            for (int d = 0; d < MDPP_MAX_DIM; ++d)
              if (d < D) {
                if (TOP64 && i + j + 1 == ORDER) {
                  // float64 array * python float / float64, added into fp32
                  sd[i][d] = (R)__dadd_rn(
                      (double)sd[i][d],
                      __ddiv_rn(__dmul_rn(top64[d], tu_pow[j]), fact));
                  continue;
                }
                const R term = O::mul(sd[i + j + 1][d], tu);
                if (sizeof(R) == 4 && j <= 1) {
                  // f32(f64(x) + f64(t) / {1,2}): the quotient is exact and a
                  // sum rounded to 53 then 24 bits equals the sum rounded to
                  // 24 bits directly (53 >= 2*24 + 2), so this IS the
                  // reference's mixed-precision result, without conversions
                  sd[i][d] = O::add(sd[i][d], j == 0 ? term : O::mul(term, (R)0.5));
                } else {
                  sd[i][d] = (R)__dadd_rn((double)sd[i][d],
                                          __ddiv_rn((double)term, fact));
                }
              }
          }
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) nxt[d] = sd[0][d];
    } else {  // frozen state, derivatives kept (:1671-1679)
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) nxt[d] = em[d];
    }
    if (NOISE != MDPP_NOISE_OFF && PNOISE) {
      double nz[MDPP_MAX_DIM];
      if (NOISE == MDPP_NOISE_REPLAY) {
#pragma unroll
        for (int d = 0; d < MDPP_MAX_DIM; ++d)
          if (d < D) nz[d] = p.io.replay_state_noise[row * D + d];
      } else if (ZIG_NORMAL) {
        // one 64-bit word per normal: dimensions (2c, 2c + 1) share a call;
        // the 1.5 % of first attempts that are rejected go through ONE
        // out-of-line call site afterwards
        const uint4* kw = reinterpret_cast<const uint4*>(p.zig + kZigOffFast);
        uint32_t rej = 0;
#pragma unroll
        for (int c = 0; c < MDPP_MAX_DIM / 2; ++c)
          if (2 * c < D) {
            const U4 w = philox4x32_10_rk(gid, (uint32_t)step, (uint32_t)(step >> 32),
                                          STREAM_STATE_NOISE + (uint32_t)c, p.rk);
            bool ok0, ok1 = true;
            nz[2 * c] = zig_first(w.x, w.y, kw, &ok0);
            if (2 * c + 1 < D) nz[2 * c + 1] = zig_first(w.z, w.w, kw, &ok1);
            if (!ok0) rej |= 1u << (2 * c);
            if (!ok1) rej |= 2u << (2 * c);
          }
#pragma unroll 1
        while (rej) {
          const int jb = __ffs((int)rej) - 1;
          rej &= rej - 1;
          const double zz = zig_resolve_draw(gid, step, (uint32_t)jb, p.rk, p.zig);
#pragma unroll
          for (int d = 0; d < MDPP_MAX_DIM; ++d)
            if (d < D && d == jb) nz[d] = zz;
        }
#pragma unroll
        for (int d = 0; d < MDPP_MAX_DIM; ++d)
          if (d < D) nz[d] = __dmul_rn(p_std, nz[d]);  // numpy: 0 + sigma * z
      } else {
#pragma unroll
        for (int c = 0; c < MDPP_MAX_DIM / 4; ++c)
          if (4 * c < D) {
            U4 w = philox4x32_10_rk(gid, (uint32_t)step, (uint32_t)(step >> 32),
                                    STREAM_STATE_NOISE + (uint32_t)c, p.rk);
            double z[4];
            if (FAST_NORMAL) {
              normal_pair_fast(w.x, w.y, &z[0], &z[1]);
              normal_pair_fast(w.z, w.w, &z[2], &z[3]);
            } else {
              normal_pair_f64(w.x, w.y, &z[0], &z[1]);
              normal_pair_f64(w.z, w.w, &z[2], &z[3]);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (4 * c + k < D)
                nz[4 * c + k] = __dmul_rn(p_std, z[k]);
          }
      }
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) {
          sum_abs_pnoise += fabs(nz[d]);
          nxt[d] = (R)__dadd_rn((double)nxt[d], nz[d]);  // f32 += f64 array
        }
    }
    bool in_bounds = !IMAGE;
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (d < D) in_bounds = in_bounds && nxt[d] >= -smax && nxt[d] <= smax;
    if (!in_bounds) {  // clip, zero every derivative (:1702-1717)
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) {
          nxt[d] = nxt[d] < -smax ? -smax : (nxt[d] > smax ? smax : nxt[d]);
#pragma unroll
          for (int k = 1; k <= MDPP_MAX_ORDER; ++k)
            if (k <= ORDER) sd[k][d] = 0;
          sd[0][d] = nxt[d];
        }
    }
    const double dist_new = dist_to_target(nxt);
    dist_prev = dist_new;
    const double radius = TARGET64 ? radius64 : (double)radius_r;
    if (!LINE && dist_new < radius) reached = true;
    tl += 1;
    phase = (phase + 1 == EVERY_N) ? 0 : phase + 1;

    // ---- reward ------------------------------------------------------------
    // `rr` is the np.float32 (dtype_s) reward, `rd` the python-float one;
    // `is_real` says which of the two numpy would be carrying.
    R rr;
    double rd = 0.0;
    bool is_real = true;
    if (LINE) {
      R* hist = reinterpret_cast<R*>(p.st.hist);
      const int slot = (int)(step % (uint64_t)SEQ);
#pragma unroll
      for (int k = 0; k < MDPP_MAX_DIM; ++k)
        if (k < NREL) hist[((int64_t)slot * NREL + k) * N + env] = nxt[rel_index(cfg, k)];
      // NaN gate of the window (:1858): sequence_length + 1 states since the reset
      if (tl >= SEQ) rd = line_reward<R>(hist, N, env, NREL, SEQ, step);
      is_real = false;
      rr = (R)0;
    } else if (DENSE) {
      if (TARGET64) {  // float64 norms make the reward float64
        rd = __dadd_rn(-dist_new, dist_old);
        is_real = false;
      } else {
        rr = O::add(-(R)dist_new, (R)dist_old);
      }
    } else {
      rd = dist_new < radius ? 1.0 : 0.0;
      is_real = false;
    }
    if (!LINE) {  // reward -= action_loss_weight * ||action||  (always makes it dtype_s)
      // weight 0: 0 * ||a|| = 0 (finite actions); the subtraction still
      // happens for its dtype effect, the norm is skipped
      const R loss = alw == 0.0 ? (R)0
                                : O::mul((R)alw, seq_norm<R>(D, [&](int k) { return a[k]; }));
      if (is_real) rr = O::add(rr, -loss);
      else if (sizeof(R) == 4 && TARGET64 && DENSE)
        rd = __dadd_rn(rd, -(double)loss);  // float64 - float32 -> float64
      else { rr = O::add((R)rd, -loss); is_real = true; }
    }
    if (DELAY > 0) {
      const bool have = tl > DELAY;
      if (sizeof(R) == 4 && ((TARGET64 && DENSE) || LINE)) {
        // the reward is a python float here (float64 norms), and the
        // reference's reward_buffer keeps it one: the FIFO holds doubles and
        // the tail below stays on the float64 path (the caller allocates the
        // ring as float64 for this configuration)
        double* slot = reinterpret_cast<double*>(p.st.ring) + (int64_t)ring_pos * N + env;
        const double delayed = have ? *slot : 0.0;
        *slot = rd;
        rd = delayed;
        is_real = false;
      } else {
        R* slot = ring + (int64_t)ring_pos * N + env;
        const R delayed = have ? *slot : (R)0;
        *slot = is_real ? rr : (R)rd;
        if (have) { rr = delayed; is_real = true; }
        else { rd = 0.0; is_real = false; }  // zero-initialised python floats
      }
      ring_pos = (ring_pos + 1 == DELAY) ? 0 : ring_pos + 1;
    }
    if (phase != 0) { rd = 0.0; is_real = false; }
    sum_reward += is_real ? (double)rr : rd;
    double nrw = 0.0;
    if (NOISE != MDPP_NOISE_OFF && RNOISE) {
      if (NOISE == MDPP_NOISE_REPLAY) {
        nrw = p.io.replay_reward_noise[row];
      } else {
        U4 w = philox4x32_10_rk(gid, (uint32_t)step, (uint32_t)(step >> 32),
                                STREAM_NORMAL, p.rk);
        double z0, z1;
        if (ZIG_NORMAL) {
          bool ok;
          z0 = zig_first(w.x, w.y, reinterpret_cast<const uint4*>(p.zig + kZigOffFast), &ok);
          if (!ok) z0 = zig_resolve_draw(gid, step, kZigDrawReward, p.rk, p.zig);
        } else if (FAST_NORMAL) normal_pair_fast(w.x, w.y, &z0, &z1);
        else normal_pair_f64(w.x, w.y, &z0, &z1);
        nrw = __dmul_rn(r_std, z0);
      }
      sum_abs_rnoise += fabs(nrw);
    }
    const bool box = NBOX > 0 && in_term_box<R>(cfg, NREL, nxt);
    const bool done = box || reached;
    R out_r;
    if (is_real) {  // np.float32 op python-float: the scalar is cast first
      if (RNOISE) rr = O::add(rr, (R)nrw);
      rr = O::mul(rr, (R)r_scale);
      rr = O::add(rr, (R)r_shift);
      if (done) rr = O::add(rr, (R)term_add);
      out_r = rr;
    } else {
      if (RNOISE) rd = __dadd_rn(rd, nrw);
      rd = __dmul_rn(rd, r_scale);
      rd = __dadd_rn(rd, r_shift);
      if (done) rd = __dadd_rn(rd, term_add);
      out_r = (R)rd;
    }
    const bool trunc = HORIZON > 0 && tl >= HORIZON;
    n_terminated += done;
    if constexpr (AG::kActs) ag.step(out_r, AUTORESET && (done || trunc));
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (d < D) em[d] = nxt[d];
    if (!FAST && p.io.final_obs)
      store_row<R>(reinterpret_cast<R*>(p.io.final_obs) + row * D, D, nxt);
    if (AUTORESET && (done || trunc)) {
      R s0[MDPP_MAX_DIM];
      if (NOISE == MDPP_NOISE_REPLAY) {
        const R* rs = reinterpret_cast<const R*>(p.io.replay_reset_state) + row * D;
#pragma unroll
        for (int d = 0; d < MDPP_MAX_DIM; ++d)
          if (d < D) s0[d] = rs[d];
      } else {
        const RowVal<R> fresh = sample_reset_state<R>(p, cfg, D, NREL, NBOX, gid, ep);
#pragma unroll
        for (int d = 0; d < MDPP_MAX_DIM; ++d)
          if (d < D) s0[d] = fresh.v[d];
      }
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) {
          em[d] = s0[d];
#pragma unroll
          for (int k = 1; k <= MDPP_MAX_ORDER; ++k)
            if (k <= ORDER) sd[k][d] = 0;
          sd[0][d] = s0[d];
        }
      tl = 0; phase = 0; reached = false;
      ep += 1; n_episodes += 1;
      dist_prev = dist_to_target(em);
    }
    if (FAST || p.io.obs) store_row<R>(reinterpret_cast<R*>(p.io.obs) + row * D, D, em);
    if (FAST || p.io.reward) reinterpret_cast<R*>(p.io.reward)[row] = out_r;
    if (FAST || p.io.terminated) p.io.terminated[row] = (uint8_t)done;
    if (FAST || p.io.truncated) p.io.truncated[row] = (uint8_t)trunc;
  };
  int t = 0;
#pragma unroll 1
  for (; t + PF <= p.T; t += PF) {
#pragma unroll
    for (int u = 0; u < PF; ++u) one_step(t + u, abuf[u]);
  }
#pragma unroll
  for (int u = 0; u < PF - 1; ++u)  // tail: t is a multiple of PF here
    if (t + u < p.T) one_step(t + u, abuf[u]);

#pragma unroll
  for (int k = 0; k <= MDPP_MAX_ORDER; ++k)
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (k <= ORDER && d < D) derivs[((int64_t)k * D + d) * N + env] = sd[k][d];
#pragma unroll
  for (int d = 0; d < MDPP_MAX_DIM; ++d)
    if (d < D) emitted[(int64_t)d * N + env] = em[d];
  p.st.t_episode[env] = tl;
  p.st.episode[env] = ep;
  p.st.reached[env] = (uint8_t)reached;
  if constexpr (AG::kActs) ag.end(env);
  }  // active
  if (p.st.stats) {  // block-reduced: one atomic per CTA and counter (the
    // counters are single addresses; at T = 1 a per-warp atomic was the
    // launch's critical path)
    // (transitions = envs x T is known up front: one thread adds it)
    double vals[6] = {(double)n_episodes, 0.0, sum_reward,
                      sum_abs_rnoise, sum_abs_pnoise, (double)n_terminated};
    const int slots[6] = {MDPP_STAT_EPISODES, MDPP_STAT_TRANSITIONS,
                          MDPP_STAT_REWARD, MDPP_STAT_ABS_REWARD_NOISE,
                          MDPP_STAT_ABS_TRANSITION_NOISE, MDPP_STAT_TERMINATED};
    __shared__ double red[6][kCBlock / 32];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      double v = vals[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < kCBlock / 32; ++w) v += red[threadIdx.x][w];
      if (!GROUPS && blockIdx.x == 0 && threadIdx.x == 1) v = (double)N * (double)p.T;
      if (GROUPS && threadIdx.x == 1)  // this CTA's envs x T
        v = (double)max((int64_t)0, min((int64_t)kCBlock,
                                        gsm->env_count - (sel.local - threadIdx.x))) *
            (double)p.T;
      // CTAs spread their atomics over the `stats_slots` copies of the rows
      // [slot][group][MDPP_N_STATS]
      const int n_groups = GROUPS ? p.n_groups : 1;
      if (v != 0.0)
        atomicAdd(p.st.stats + ((int64_t)(blockIdx.x % (unsigned)max(p.st.stats_slots, 1)) *
                                    n_groups + sel.group) * MDPP_N_STATS +
                      slots[threadIdx.x], v);
    }
  }
}

template <typename R, bool GROUPS = false>
__device__ __forceinline__ void continuous_reset_body(const ContinuousParams& p) {
  __shared__ GroupSmem<GROUPS> gsm_store;
  ContinuousGroupDev* gsm = group_ptr(gsm_store);
  const int64_t N = p.st.n_envs;
  const ContinuousGroupSel sel = select_group<GROUPS>(p, gsm, N);
  const mdpp_continuous_config& cfg = GROUPS ? gsm->cfg : p.cfg;
  const int D = cfg.dim, ORDER = cfg.order, NREL = cfg.n_relevant;
  if (!sel.active) return;
  const int64_t env = sel.env;
  R* derivs = reinterpret_cast<R*>(p.st.derivs);
  R* emitted = reinterpret_cast<R*>(p.st.emitted);
  R* obs = reinterpret_cast<R*>(p.reset_obs);
  if (p.mask && !p.mask[env]) {
    if (obs)
      for (int d = 0; d < D; ++d) obs[env * D + d] = emitted[(int64_t)d * N + env];
    return;
  }
  const uint32_t gid = sel.gid;
  const uint32_t ep = p.st.episode[env];
  R s0[MDPP_MAX_DIM];
  if (p.init_states) {
    const R* src = reinterpret_cast<const R*>(p.init_states) + env * D;
    for (int d = 0; d < D; ++d) s0[d] = src[d];
  } else {
    for (int attempt = 0; attempt < 64; ++attempt) {
      box_sample<R>(p, cfg, D, gid, ep, attempt, s0);
      if (!(cfg.n_term_boxes > 0 && in_term_box<R>(cfg, NREL, s0))) break;
    }
  }
  if (p.st.stats && p.st.t_episode[env] > 0)
    atomicAdd(p.st.stats + ((int64_t)(blockIdx.x % (unsigned)max(p.st.stats_slots, 1)) *
                                (GROUPS ? p.n_groups : 1) + sel.group) * MDPP_N_STATS +
                  MDPP_STAT_EPISODES, 1.0);
  for (int d = 0; d < D; ++d) {
    emitted[(int64_t)d * N + env] = s0[d];
    for (int k = 0; k <= ORDER; ++k)
      derivs[((int64_t)k * D + d) * N + env] = k == 0 ? s0[d] : (R)0;
    if (obs) obs[env * D + d] = s0[d];
  }
  p.st.t_episode[env] = 0;
  p.st.episode[env] = ep + 1;
  p.st.reached[env] = 0;
}

template <typename R, int NOISE, bool GROUPS = false, typename AG = NoContinuousAgent>
__global__ void __launch_bounds__(kCBlock)
continuous_rollout_kernel(const __grid_constant__ typename AG::Params p) {
  continuous_body<R, NOISE, GROUPS, AG>(p);
}

template <typename R, bool GROUPS = false>
__global__ void __launch_bounds__(kCBlock)
continuous_reset_kernel(const __grid_constant__ ContinuousParams p) {
  continuous_reset_body<R, GROUPS>(p);
}

}  // namespace mdpp
