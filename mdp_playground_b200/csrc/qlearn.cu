// Tabular Q-learning fused into the discrete rollout (mdpp_discrete_qlearn).
//
// The kernel is rollout_body (discrete_kernels.cuh) with a QAgent plugged into
// its agent hooks: the same group staging, Philox draws, chain step, delay
// ring, reward normals, auto-reset and statistics, so the env state and the
// counters end exactly as a rollout with the same actions leaves them.  Per
// env and step (global step `step`, Philox id g, state s):
//   w = philox(g, step, STREAM_ACTION)               (phase A, the random policy's word)
//   explore = (double)w.z < epsilon * 2^32
//   a = explore ? umulhi(w.x, A) : argmax_a' Q[s][a']  (lowest index on ties)
//   step -> r, nxt (before any auto-reset), terminated
//   target = terminated ? r : r + gamma * max_a' Q[nxt][a']
//   Q[s][a] = q + alpha * (target - q)
// with every float64 operation rounded on its own (no FMA contraction), so a
// numpy restatement in the same order gives the same bits.
//
// Q is float64 [N][q_states][q_actions], env-major: each env walks its own
// contiguous table (64 rows of 64 B at 8 x 8; 32 MB for 65 536 envs, which
// stays resident in the 126 MB L2).  One row load per step sits on the
// dependent chain: Q[nxt] gives both the target's max and, when no
// auto-reset follows, the next step's greedy action.
#include <algorithm>
#include <cmath>

#include "discrete_launch.h"

namespace mdpp {

struct QlearnParams {
  RolloutParams base;
  QlearnDev q;
};

struct QAgent {
  static constexpr bool kStepOut = true;
  const QlearnDev& d;
  double* tab;       // this env's Q-table
  int32_t greedy;    // argmax of the current state's row
  uint32_t explore;  // bit j: step j of the chunk explores
  int32_t s, a;      // the step's state and action
  double ep_ret;     // return of the running episode
  // (the rest lives in the kernel parameters and the group view: registers
  // are what bounds the chain's occupancy)

  __device__ __forceinline__ explicit QAgent(const QlearnDev& dev) : d(dev) {}

  // (max, lowest argmax) of row st; numpy.argmax order
  __device__ __forceinline__ int32_t row_argmax(const GroupView& v, int32_t st,
                                                double& m) const {
    const double* row = tab + (int64_t)st * d.q_actions;
    m = row[0];
    int32_t am = 0;
#pragma unroll 4
    for (int k = 1; k < v.A; ++k) {
      const double x = row[k];
      if (x > m) { m = x; am = k; }
    }
    return am;
  }

  __device__ __forceinline__ void begin(const GroupView& v, int64_t env, int32_t s0) {
    tab = d.q + env * (int64_t)d.q_states * d.q_actions;
    double m;
    greedy = row_argmax(v, s0, m);
    ep_ret = d.ep_return[env];
  }

  __device__ __forceinline__ void draw(int j, const U4& w) {
    if (j == 0) explore = 0;
    explore |= (uint32_t)((uint64_t)w.z < d.explore_below) << j;
  }

  __device__ __forceinline__ int32_t act(int j, int32_t a_rand, int32_t st) {
    s = st;
    a = ((explore >> j) & 1u) ? a_rand : greedy;
    return a;
  }

  __device__ __forceinline__ void update(const RolloutParams& p, const GroupView& v,
                                         const StepOut& o, int32_t s_after,
                                         int64_t env, int64_t off) {
    double* q_at = tab + (int64_t)s * d.q_actions + a;
    const double q = *q_at;  // (loaded beside the row of nxt)
    double m;
    const int32_t am = row_argmax(v, o.nxt, m);
    const double target = o.done ? o.r : __dadd_rn(o.r, __dmul_rn(d.gamma, m));
    const double qn = __dadd_rn(q, __dmul_rn(d.alpha, __dsub_rn(target, q)));
    *q_at = qn;
    const bool reset = autoreset_of(p) && (o.done || o.trunc);
    if (reset) {
      greedy = row_argmax(v, s_after, m);
    } else if (o.nxt != s) {
      greedy = am;
    } else if (a != am) {  // the row just loaded changed in entry a only
      greedy = (qn > m || (qn == m && a < am)) ? a : am;
    } else {  // the maximum itself changed: rescan unless it only grew
      greedy = qn >= m ? am : row_argmax(v, s, m);
    }
    ep_ret = __dadd_rn(ep_ret, o.r);
    if (reset) {
      d.ret_sum[env] = __dadd_rn(d.ret_sum[env], ep_ret);
      d.ret_count[env] += 1;
      ep_ret = 0.0;
    }
    if (d.actions_taken) st_stream(d.actions_taken + off, a);
  }

  __device__ __forceinline__ void end(int64_t env) { d.ep_return[env] = ep_ret; }
};

// 65 536 envs are 1024 CTAs of 64, 7 per SM: 144 registers a thread keep 7
// CTAs resident (one wave) and leave room for the agent state
template <typename C>
__global__ void __maxnreg__(144)
discrete_qlearn_kernel(const __grid_constant__ QlearnParams qp) {
  QAgent ag(qp.q);
  rollout_body<C>(qp.base, ag);
}

template <int NORMAL>
static int launch_qlearn(mdpp_ctx* ctx, QlearnParams& qp, cudaStream_t stream) {
  RolloutParams& p = qp.base;
  const int smem_tab = ctx->max_group_blob;
  bool ring_ok;
  if (tables_in_smem(ctx, p, &ring_ok) && ring_ok) {
    using Cs = Cfg<MDPP_NOISE_PHILOX, NORMAL, true, true, false, -1>;
    return launch_kernel<Cs>(ctx, p, smem_tab, stream, discrete_qlearn_kernel<Cs>, qp);
  }
  using Cg = Cfg<MDPP_NOISE_PHILOX, NORMAL, false, false, false, -1>;
  return launch_kernel<Cg>(ctx, p, smem_tab, stream, discrete_qlearn_kernel<Cg>, qp);
}

int check_qlearn_params(mdpp_ctx* ctx, const mdpp_qlearn_params* qp, int64_t n_states,
                        int64_t n_actions, QlearnDev* d) {
  if (!qp || !qp->q || !qp->ep_return || !qp->ret_sum || !qp->ret_count)
    return fail(ctx, MDPP_EINVAL, "qlearn: q, ep_return, ret_sum or ret_count is NULL");
  if (qp->q_states < n_states || qp->q_actions < n_actions)
    return fail(ctx, MDPP_EINVAL, "qlearn: q_states / q_actions smaller than a group's S / A");
  // (written so that NaN fails too)
  if (!(qp->alpha >= 0.0 && qp->alpha <= 1.0) || !(qp->gamma >= 0.0 && qp->gamma <= 1.0) ||
      !(qp->epsilon >= 0.0 && qp->epsilon <= 1.0))
    return fail(ctx, MDPP_EINVAL, "qlearn: alpha, gamma and epsilon must lie in [0, 1]");
  d->q = qp->q;
  d->q_states = qp->q_states;
  d->q_actions = qp->q_actions;
  d->alpha = qp->alpha;
  d->gamma = qp->gamma;
  // w < x for an integer w <=> w < ceil(x); x = epsilon * 2^32 is exact
  d->explore_below = (uint64_t)std::ceil(qp->epsilon * 4294967296.0);
  d->ep_return = qp->ep_return;
  d->ret_sum = qp->ret_sum;
  d->ret_count = qp->ret_count;
  d->actions_taken = qp->actions_taken;
  return MDPP_OK;
}

}  // namespace mdpp

using namespace mdpp;

extern "C" int mdpp_discrete_qlearn(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                                    const mdpp_discrete_io* io,
                                    const mdpp_qlearn_params* qp,
                                    const mdpp_step_opts* opts, void* cuda_stream) {
  QlearnParams k;
  int rc = prepare_rollout(ctx, st, io, opts, k.base);
  if (rc) return rc;
  if (io->actions)
    return fail(ctx, MDPP_EINVAL, "qlearn: io->actions must be NULL (the agent acts)");
  if (opts->noise_mode != MDPP_NOISE_PHILOX)
    return fail(ctx, MDPP_EINVAL, "qlearn: Philox noise only");
  if (ctx->d_irr)
    return fail(ctx, MDPP_EINVAL, "qlearn: irrelevant features are not supported");
  int64_t S = 0, A = 0;
  for (auto& g : ctx->d_groups_host) {
    S = std::max<int64_t>(S, g.S);
    A = std::max<int64_t>(A, g.A);
  }
  rc = check_qlearn_params(ctx, qp, S, A, &k.q);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  switch (opts->normal_mode) {
    case MDPP_NORMAL_FAST: return launch_qlearn<MDPP_NORMAL_FAST>(ctx, k, s);
    case MDPP_NORMAL_ZIGGURAT: return launch_qlearn<MDPP_NORMAL_ZIGGURAT>(ctx, k, s);
    default: return launch_qlearn<MDPP_NORMAL_F64>(ctx, k, s);
  }
}
