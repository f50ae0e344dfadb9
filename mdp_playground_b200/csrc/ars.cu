// Augmented random search (Mania, Guy & Recht 2018, "Simple random search
// provides a competitive approach to reinforcement learning", Algorithm 1,
// V1 / V1-t) on the continuous rollout: mdpp_continuous_ars,
// mdpp_continuous_ars_update and mdpp_continuous_ars_perturbations.
//
// A config group (or the single configuration) is one ARS run, its envs the
// perturbation population: local env 2p is the + member and 2p + 1 the -
// member of pair p.  The policy is linear, a = W [obs; 1], W = theta_g +
// (s nu) delta_p; delta_p is regenerated from a Philox counter (global id of
// the + member, iteration, STREAM_ARS_DELTA + word), so nothing but theta and
// the per-env fitness is stored.  The rollout kernel is continuous_body
// (continuous_kernels.cuh) with ArsAgent plugged into its agent hooks: the
// env state and counters end exactly as a rollout with the recorded actions
// leaves them.  Every float64 operation is rounded on its own (explicit _rn
// intrinsics, no FMA), so a numpy restatement in the same order gives the
// same bits (tests/ars_oracle.py).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "continuous_kernels.cuh"
#include "internal.h"

namespace mdpp {

constexpr int kArsMaxP = MDPP_MAX_DIM * (MDPP_MAX_DIM + 1);  // 272

struct ArsDev {
  const double* theta;  // [G][P]
  double* fitness;
  ReturnsDev ret;
  void* actions_taken;  // real [T][N][D] or NULL
  double noise_std;
  uint64_t iteration;
};

struct ArsParams : ContinuousParams {
  ArsDev a;
};

// delta_p entries of Philox word c: Box-Muller (fp64) of (w0, w1), (w2, w3)
__device__ __forceinline__ void ars_delta_word(uint32_t gid_plus, uint64_t it, int c,
                                               const uint32_t* rk, double* z) {
  const U4 w = philox4x32_10_rk(gid_plus, (uint32_t)it, (uint32_t)(it >> 32),
                                STREAM_ARS_DELTA + (uint32_t)c, rk);
  normal_pair_f64(w.x, w.y, &z[0], &z[1]);
  normal_pair_f64(w.z, w.w, &z[2], &z[3]);
}

template <typename R>
struct ArsAgent {
  static constexpr bool kActs = true;
  using Params = ArsParams;
  const ArsParams& p;
  double w[kArsMaxP];  // this env's perturbed weights, [D][D+1] row-major
  double fit, ep_ret;
  int64_t env;

  __device__ __forceinline__ explicit ArsAgent(const ArsParams& p_) : p(p_) {}

  // theta of the CTA's group (a CTA belongs to one group) goes through shared
  // memory; every env then draws its delta once per launch
  __device__ __forceinline__ void begin(const ContinuousGroupSel& sel,
                                        const mdpp_continuous_config&, int D) {
    __shared__ double th[kArsMaxP];
    const int P = D * (D + 1);
    const double* src = p.a.theta + (int64_t)sel.group * P;
    for (int j = threadIdx.x; j < P; j += kCBlock) th[j] = src[j];
    __syncthreads();
    if (!sel.active) return;
    env = sel.env;
    fit = p.a.fitness[env];
    ep_ret = p.a.ret.ep_return[env];
    const uint32_t gid_plus = sel.gid - (uint32_t)(sel.local & 1);
    const double snu = (sel.local & 1) ? -p.a.noise_std : p.a.noise_std;
#pragma unroll 1
    for (int c = 0; 4 * c < P; ++c) {
      double z[4];
      ars_delta_word(gid_plus, p.a.iteration, c, p.rk, z);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (4 * c + k < P) w[4 * c + k] = __dadd_rn(th[4 * c + k], __dmul_rn(snu, z[k]));
    }
  }

  // a_d = sum_k w[d][k] phi_k, phi = (em, 1), from the k = 0 product upward
  __device__ __forceinline__ void act(const R* em, int D, R amax, int64_t row, R* out) {
    const bool bounded = isfinite((double)amax);
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (d < D) {
        const double* wd = w + d * (D + 1);
        double acc = __dmul_rn(wd[0], (double)em[0]);
#pragma unroll
        for (int k = 1; k < MDPP_MAX_DIM; ++k)
          if (k < D) acc = __dadd_rn(acc, __dmul_rn(wd[k], (double)em[k]));
        acc = __dadd_rn(acc, wd[D]);  // (times phi_D = 1: exact)
        R a = (R)acc;
        if (bounded) a = a < -amax ? -amax : (a > amax ? amax : a);
        out[d] = a;
      }
    if (p.a.actions_taken) {
      R* dst = reinterpret_cast<R*>(p.a.actions_taken) + row * D;
#pragma unroll
      for (int d = 0; d < MDPP_MAX_DIM; ++d)
        if (d < D) dst[d] = out[d];
    }
  }

  // (the episode returns as TabularQ keeps them, written out here: through a
  // shared inline helper the double kernels, which spill, compile differently)
  __device__ __forceinline__ void step(R out_r, bool reset) {
    const double r = (double)out_r;
    fit = __dadd_rn(fit, r);
    ep_ret = __dadd_rn(ep_ret, r);
    if (reset) {
      p.a.ret.ret_sum[env] = __dadd_rn(p.a.ret.ret_sum[env], ep_ret);
      p.a.ret.ret_count[env] += 1;
      ep_ret = 0.0;
    }
  }

  __device__ __forceinline__ void end(int64_t) {
    p.a.fitness[env] = fit;
    p.a.ret.ep_return[env] = ep_ret;
  }
};

template <typename R, bool GROUPS>
__global__ void __launch_bounds__(kCBlock)
continuous_ars_kernel(const __grid_constant__ ArsParams p) {
  continuous_body<R, MDPP_NOISE_PHILOX, GROUPS, ArsAgent<R>>(p);
}

// ---- evaluation of theta (mdpp_continuous_ars_eval) -------------------------
// a = theta_g [obs; 1]: ArsAgent's policy with noise_std = 0, read straight
// from the shared-memory copy of theta_g (no delta, no per-thread weights, no
// fitness); the first ev.episodes episodes go to EvalEpisodes.
struct ArsEvalParams : ContinuousParams {
  const double* theta;  // [G][P]
  EvalDev ev;
};

template <typename R>
struct ArsEvalAgent {
  static constexpr bool kActs = true;
  using Params = ArsEvalParams;
  const ArsEvalParams& p;
  const double* th;  // theta of the CTA's group, in shared memory
  EvalEpisodes ep;

  __device__ __forceinline__ explicit ArsEvalAgent(const ArsEvalParams& p_) : p(p_) {}

  __device__ __forceinline__ void begin(const ContinuousGroupSel& sel,
                                        const mdpp_continuous_config&, int D) {
    __shared__ double th_s[kArsMaxP];
    const int P = D * (D + 1);
    const double* src = p.theta + (int64_t)sel.group * P;
    for (int j = threadIdx.x; j < P; j += kCBlock) th_s[j] = src[j];
    __syncthreads();
    th = th_s;
    ep.begin();
  }

  // ArsAgent::act's sums, casts and clipping, on theta (written out again:
  // the learner's kernels keep their code as it was)
  __device__ __forceinline__ void act(const R* em, int D, R amax, int64_t, R* out) const {
    const bool bounded = isfinite((double)amax);
#pragma unroll
    for (int d = 0; d < MDPP_MAX_DIM; ++d)
      if (d < D) {
        const double* wd = th + d * (D + 1);
        double acc = __dmul_rn(wd[0], (double)em[0]);
#pragma unroll
        for (int k = 1; k < MDPP_MAX_DIM; ++k)
          if (k < D) acc = __dadd_rn(acc, __dmul_rn(wd[k], (double)em[k]));
        acc = __dadd_rn(acc, wd[D]);
        R a = (R)acc;
        if (bounded) a = a < -amax ? -amax : (a > amax ? amax : a);
        out[d] = a;
      }
  }

  // (autoreset is required: `reset` is terminated or truncated)
  __device__ __forceinline__ void step(R out_r, bool reset) {
    ep.step(p.ev, (double)out_r, reset);
  }

  __device__ __forceinline__ void end(int64_t env) const { ep.end(p.ev, env); }
};

template <typename R, bool GROUPS>
__global__ void __launch_bounds__(kCBlock)
continuous_ars_eval_kernel(const __grid_constant__ ArsEvalParams p) {
  continuous_body<R, MDPP_NOISE_PHILOX, GROUPS, ArsEvalAgent<R>>(p);
}

// ---- the update --------------------------------------------------------------
struct ArsUpdateParams {
  const ContinuousGroupDev* groups;  // NULL: one group of all n_envs
  int64_t n_envs, env_id_offset;
  int32_t n_groups, P, b;
  double step_size;
  double* theta;
  const double* fitness;
  double* delta;       // [N/2][P]
  uint8_t* kept;       // [N/2] or NULL (perturbations only)
  double* factor;      // [G] step_size / (b sigma_R), 0 when not updated
  double* group_stats; // [G][3] or NULL
  uint64_t iteration;
  uint32_t rk[20];
};

struct ArsRange { int64_t begin, count, gid; };
__device__ __forceinline__ ArsRange ars_range(const ArsUpdateParams& u, int g) {
  if (!u.groups) return ArsRange{0, u.n_envs, 0};
  return ArsRange{u.groups[g].env_begin, u.groups[g].env_count, u.groups[g].gid_base};
}

// max(F+, F-) of pair q of a group whose envs start at `f`
__device__ __forceinline__ double ars_key(const double* f, int64_t q) {
  const double a = f[2 * q], b = f[2 * q + 1];
  return a > b ? a : b;
}

// one thread per (pair, group): delta_p, and whether the pair is among the
// group's top b (rank by counting: ties go to the lower p)
__global__ void ars_delta_rank_kernel(const __grid_constant__ ArsUpdateParams u) {
  const int g = blockIdx.y;
  const ArsRange r = ars_range(u, g);
  const int64_t pairs = r.count / 2;
  const int64_t pr = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pr >= pairs) return;
  const int64_t slot = r.begin / 2 + pr;  // global pair index
  const uint32_t gid_plus = (uint32_t)(u.env_id_offset + r.gid + 2 * pr);
  double* dst = u.delta + slot * u.P;
  for (int c = 0; 4 * c < u.P; ++c) {
    double z[4];
    ars_delta_word(gid_plus, u.iteration, c, u.rk, z);
    for (int k = 0; k < 4; ++k)
      if (4 * c + k < u.P) dst[4 * c + k] = z[k];
  }
  if (!u.kept) return;
  bool keep = true;
  if (u.b < pairs) {
    const double* f = u.fitness + r.begin;
    const double mine = ars_key(f, pr);
    int64_t rank = 0;
    for (int64_t q = 0; q < pairs; ++q) {
      const double k = ars_key(f, q);
      rank += (k > mine || (k == mine && q < pr)) ? 1 : 0;
    }
    keep = rank < u.b;
  }
  u.kept[slot] = keep;
}

// one thread per group: mean and population std of the 2b kept returns
// (ascending p, F+ before F-, sequential), and the step factor
__global__ void ars_sigma_kernel(const __grid_constant__ ArsUpdateParams u) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= max(u.n_groups, 1)) return;
  const ArsRange r = ars_range(u, g);
  const int64_t pairs = r.count / 2;
  const double* f = u.fitness + r.begin;
  const uint8_t* kept = u.kept + r.begin / 2;
  const double n = (double)(2 * (int64_t)u.b);
  double s = 0.0;
  for (int64_t q = 0; q < pairs; ++q)
    if (kept[q]) s = __dadd_rn(__dadd_rn(s, f[2 * q]), f[2 * q + 1]);
  const double m = __ddiv_rn(s, n);
  double v = 0.0;
  for (int64_t q = 0; q < pairs; ++q)
    if (kept[q]) {
      const double d0 = __dsub_rn(f[2 * q], m), d1 = __dsub_rn(f[2 * q + 1], m);
      v = __dadd_rn(__dadd_rn(v, __dmul_rn(d0, d0)), __dmul_rn(d1, d1));
    }
  const double sigma = __dsqrt_rn(__ddiv_rn(v, n));
  const bool upd = isfinite(sigma) && sigma > 0.0;
  u.factor[g] = upd ? __ddiv_rn(u.step_size, __dmul_rn((double)u.b, sigma)) : 0.0;
  if (u.group_stats) {
    u.group_stats[3 * g] = m;
    u.group_stats[3 * g + 1] = sigma;
    u.group_stats[3 * g + 2] = upd ? 1.0 : 0.0;
  }
}

// one thread per (entry, group): G_j over the kept pairs (ascending p,
// sequential), theta_j += factor * G_j.  No atomics: each entry has one owner.
__global__ void ars_theta_kernel(const __grid_constant__ ArsUpdateParams u) {
  const int g = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= u.P) return;
  const double fac = u.factor[g];
  if (fac == 0.0) return;  // not updated (sigma_R 0 or not finite)
  const ArsRange r = ars_range(u, g);
  const int64_t pairs = r.count / 2;
  const double* f = u.fitness + r.begin;
  const uint8_t* kept = u.kept + r.begin / 2;
  const double* dl = u.delta + (r.begin / 2) * u.P + j;
  double G = 0.0;
#pragma unroll 4
  for (int64_t q = 0; q < pairs; ++q)
    if (kept[q])
      G = __dadd_rn(G, __dmul_rn(__dsub_rn(f[2 * q], f[2 * q + 1]), dl[q * u.P]));
  double* th = u.theta + (int64_t)g * u.P + j;
  *th = __dadd_rn(*th, __dmul_rn(fac, G));
}

}  // namespace mdpp

using namespace mdpp;

// group sizes of the context's layout: (begin, count, gid) triples
static std::vector<int64_t> ars_ranges(mdpp_ctx* ctx, int64_t n_envs) {
  if (!ctx->c_group_ranges.empty()) return ctx->c_group_ranges;
  return {0, n_envs, 0};
}

// The parameter checks both entry points share (so that a learner set up
// with bad values fails on its first call, whichever it is).
static int check_ars(mdpp_ctx* ctx, int64_t n_envs, const mdpp_ars_params* ap,
                     bool need_state) {
  if (!ctx) return MDPP_EINVAL;
  if (!ctx->have_continuous)
    return fail(ctx, MDPP_EINVAL, "ars: mdpp_set_continuous_config was not called");
  if (!ap || !ap->theta || !ap->fitness || (need_state &&
      (!ap->ep_return || !ap->ret_sum || !ap->ret_count)))
    return fail(ctx, MDPP_EINVAL,
                "ars: theta, fitness, ep_return, ret_sum or ret_count is NULL");
  if (!ctx->c_group_ranges.empty() && n_envs != ctx->c_set.n_envs)
    return fail(ctx, MDPP_EINVAL, "ars: n_envs differs from the group set's");
  const std::vector<int64_t> rg = ars_ranges(ctx, n_envs);
  int64_t min_pairs = INT64_MAX;
  for (size_t g = 0; g < rg.size(); g += 3) {
    if (rg[g + 1] % 2 != 0 || rg[g + 1] < 2)
      return fail(ctx, MDPP_EINVAL, "ars: every group needs an even number (>= 2) of envs");
    min_pairs = std::min(min_pairs, rg[g + 1] / 2);
  }
  if (ap->top_directions < 1 || ap->top_directions > min_pairs)
    return fail(ctx, MDPP_EINVAL,
                "ars: top_directions must lie in [1, the smallest group's pairs]");
  if (!(std::isfinite(ap->step_size) && ap->step_size > 0.0))
    return fail(ctx, MDPP_EINVAL, "ars: step_size must be finite and > 0");
  if (!(std::isfinite(ap->noise_std) && ap->noise_std >= 0.0))
    return fail(ctx, MDPP_EINVAL, "ars: noise_std must be finite and >= 0");
  if (ctx->c_cfg.image_mode)
    return fail(ctx, MDPP_EINVAL, "ars: image observations are not supported");
  return MDPP_OK;
}

extern "C" int mdpp_continuous_ars(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                                   const mdpp_continuous_io* io, const mdpp_ars_params* ap,
                                   const mdpp_step_opts* opts, void* cuda_stream) {
  ArsParams k;
  int rc = fill_continuous_params(ctx, st, opts, &k);
  if (rc) return rc;
  rc = check_ars(ctx, st->n_envs, ap, true);
  if (rc) return rc;
  if (!io) return fail(ctx, MDPP_EINVAL, "ars: io is NULL");
  if (io->actions)
    return fail(ctx, MDPP_EINVAL, "ars: io->actions must be NULL (the policy acts)");
  if (opts->noise_mode != MDPP_NOISE_PHILOX)
    return fail(ctx, MDPP_EINVAL, "ars: Philox noise only");
  if (opts->n_steps < 1) return fail(ctx, MDPP_EINVAL, "ars: T must be >= 1");
  if (((uintptr_t)io->obs | (uintptr_t)io->final_obs) & 15)
    return fail(ctx, MDPP_EINVAL, "obs / final_obs must be 16-byte aligned");
  k.io = *io;
  k.a = ArsDev{ap->theta, ap->fitness, ReturnsDev{ap->ep_return, ap->ret_sum, ap->ret_count},
               ap->actions_taken, ap->noise_std, ap->iteration};
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool f64 = ctx->c_cfg.is_f64;
  if (k.groups) {
    const unsigned grid = (unsigned)ctx->c_set.n_ctas;
    if (f64) continuous_ars_kernel<double, true><<<grid, kCBlock, 0, s>>>(k);
    else continuous_ars_kernel<float, true><<<grid, kCBlock, 0, s>>>(k);
  } else {
    const unsigned grid = (unsigned)((k.st.n_envs + kCBlock - 1) / kCBlock);
    if (f64) continuous_ars_kernel<double, false><<<grid, kCBlock, 0, s>>>(k);
    else continuous_ars_kernel<float, false><<<grid, kCBlock, 0, s>>>(k);
  }
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

extern "C" int mdpp_continuous_ars_eval(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                                        const mdpp_continuous_io* io,
                                        const mdpp_eval_params* ep,
                                        const mdpp_step_opts* opts, void* cuda_stream) {
  ArsEvalParams k;
  int rc = fill_continuous_params(ctx, st, opts, &k);
  if (rc) return rc;
  if (!io) return fail(ctx, MDPP_EINVAL, "ars eval: io is NULL");
  if (ctx->c_cfg.image_mode)
    return fail(ctx, MDPP_EINVAL, "ars eval: image observations are not supported");
  rc = check_eval_params(ctx, "ars eval", io->actions != nullptr, opts, ep, -1, 0, &k.ev);
  if (rc) return rc;
  if (((uintptr_t)io->obs | (uintptr_t)io->final_obs) & 15)
    return fail(ctx, MDPP_EINVAL, "obs / final_obs must be 16-byte aligned");
  k.io = *io;
  k.theta = ep->theta;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool f64 = ctx->c_cfg.is_f64;
  if (k.groups) {
    const unsigned grid = (unsigned)ctx->c_set.n_ctas;
    if (f64) continuous_ars_eval_kernel<double, true><<<grid, kCBlock, 0, s>>>(k);
    else continuous_ars_eval_kernel<float, true><<<grid, kCBlock, 0, s>>>(k);
  } else {
    const unsigned grid = (unsigned)((k.st.n_envs + kCBlock - 1) / kCBlock);
    if (f64) continuous_ars_eval_kernel<double, false><<<grid, kCBlock, 0, s>>>(k);
    else continuous_ars_eval_kernel<float, false><<<grid, kCBlock, 0, s>>>(k);
  }
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

// delta of every pair (and, with `update`, the update itself); delta goes to
// ap->delta_out, or to a stream-ordered scratch buffer
static int ars_update_impl(mdpp_ctx* ctx, int64_t n_envs, const mdpp_ars_params* ap,
                           bool update, cudaStream_t s) {
  int rc = check_ars(ctx, n_envs, ap, false);
  if (rc) return rc;
  if (!update && !ap->delta_out)
    return fail(ctx, MDPP_EINVAL, "ars perturbations: delta_out is NULL");
  const std::vector<int64_t> rg = ars_ranges(ctx, n_envs);
  const int G = (int)(rg.size() / 3);
  int64_t max_pairs = 0;
  for (int g = 0; g < G; ++g) max_pairs = std::max(max_pairs, rg[3 * g + 1] / 2);
  ArsUpdateParams u;
  std::memset(&u, 0, sizeof u);
  u.groups = ctx->c_group_ranges.empty()
                 ? nullptr : static_cast<const ContinuousGroupDev*>(ctx->c_set.groups);
  u.n_envs = n_envs;
  u.env_id_offset = ap->env_id_offset;
  u.n_groups = G;
  u.P = ctx->c_cfg.dim * (ctx->c_cfg.dim + 1);
  u.b = ap->top_directions;
  u.step_size = ap->step_size;
  u.theta = ap->theta;
  u.fitness = ap->fitness;
  u.group_stats = ap->group_stats;
  u.iteration = ap->iteration;
  philox_round_keys((uint32_t)ap->seed, (uint32_t)(ap->seed >> 32), u.rk);
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t n_pairs = n_envs / 2;
  const size_t delta_bytes = ap->delta_out ? 0 : (size_t)n_pairs * u.P * sizeof(double);
  const size_t kept_bytes = update ? (size_t)n_pairs : 0;
  const size_t fac_off = (delta_bytes + kept_bytes + 7) & ~(size_t)7;
  const size_t bytes = fac_off + (update ? (size_t)G * sizeof(double) : 0);
  uint8_t* scratch = nullptr;
  if (bytes) MDPP_CUDA(ctx, cudaMallocAsync((void**)&scratch, bytes, s));
  u.delta = ap->delta_out ? ap->delta_out : reinterpret_cast<double*>(scratch);
  u.kept = update ? scratch + delta_bytes : nullptr;
  u.factor = update ? reinterpret_cast<double*>(scratch + fac_off) : nullptr;
  const dim3 grid_pairs((unsigned)((max_pairs + 127) / 128), (unsigned)G);
  ars_delta_rank_kernel<<<grid_pairs, 128, 0, s>>>(u);
  if (update) {
    ars_sigma_kernel<<<(G + 127) / 128, 128, 0, s>>>(u);
    ars_theta_kernel<<<dim3((unsigned)((u.P + 63) / 64), (unsigned)G), 64, 0, s>>>(u);
    MDPP_CUDA(ctx, cudaMemsetAsync(ap->fitness, 0, (size_t)n_envs * sizeof(double), s));
  }
  MDPP_CUDA(ctx, cudaGetLastError());
  if (scratch) MDPP_CUDA(ctx, cudaFreeAsync(scratch, s));
  return MDPP_OK;
}

extern "C" int mdpp_continuous_ars_update(mdpp_ctx* ctx, int64_t n_envs,
                                          mdpp_ars_params* ap, void* cuda_stream) {
  const int rc = ars_update_impl(ctx, n_envs, ap, true, (cudaStream_t)cuda_stream);
  if (rc == MDPP_OK) ap->iteration += 1;
  return rc;
}

extern "C" int mdpp_continuous_ars_perturbations(mdpp_ctx* ctx, int64_t n_envs,
                                                 const mdpp_ars_params* ap,
                                                 void* cuda_stream) {
  return ars_update_impl(ctx, n_envs, ap, false, (cudaStream_t)cuda_stream);
}
