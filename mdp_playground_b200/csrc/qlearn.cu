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
// then the update of TabularQ (tabular_q.cuh).
//
// Each env walks its own contiguous table (64 rows of 64 B at 8 x 8; 32 MB
// for 65 536 envs, which stays resident in the 126 MB L2).
#include <algorithm>
#include <cmath>
#include <string>

#include "discrete_launch.h"
#include "tabular_q.cuh"

namespace mdpp {

struct QlearnParams {
  RolloutParams base;
  QlearnDev q;
};

// The group's A bounds the row scans (a run-time value: TabularQ<0>).
struct QAgent : TabularQ<0> {
  static constexpr bool kStepOut = true;
  uint32_t explore;  // bit j: step j of the chunk explores
  // (the rest lives in the kernel parameters and the group view: registers
  // are what bounds the chain's occupancy)

  __device__ __forceinline__ explicit QAgent(const QlearnDev& dev) : TabularQ(dev) {}

  __device__ __forceinline__ void begin(const GroupView& v, int64_t env, int32_t s0) {
    TabularQ::begin(env, [=] { return s0; }, v.A);
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
    TabularQ::update(p, o, v.A, env, [=] { return s_after; });
    if (d.actions_taken) st_stream(d.actions_taken + off, a);
  }
};

// 65 536 envs are 1024 CTAs of 64, 7 per SM: 144 registers a thread keep 7
// CTAs resident (one wave) and leave room for the agent state
template <typename C>
__global__ void __maxnreg__(144)
discrete_qlearn_kernel(const __grid_constant__ QlearnParams qp) {
  QAgent ag(qp.q);
  rollout_body<C>(qp.base, ag);
}

// The greedy evaluation of a fixed Q-table (mdpp_discrete_qeval): the action
// is argmax_a Q[s][a] (GreedyQ, tabular_q.cuh); the random policy's word of
// phase A is drawn and ignored.
struct QevalParams {
  RolloutParams base;
  QevalDev q;
};

struct QEvalAgent : GreedyQ<0> {
  static constexpr bool kStepOut = true;

  __device__ __forceinline__ explicit QEvalAgent(const QevalDev& dev) : GreedyQ(dev) {}

  __device__ __forceinline__ void begin(const GroupView& v, int64_t env, int32_t s0) {
    GreedyQ::begin(env, [=] { return s0; }, v.A);
  }
  __device__ __forceinline__ void draw(int, const U4&) {}
  __device__ __forceinline__ int32_t act(int, int32_t, int32_t) { return greedy; }
  __device__ __forceinline__ void update(const RolloutParams& p, const GroupView& v,
                                         const StepOut& o, int32_t s_after, int64_t,
                                         int64_t) {
    GreedyQ::update(p, o, v.A, [=] { return s_after; });
  }
};

// (the learner's occupancy target: 7 CTAs of 64 a SM for 65 536 envs)
template <typename C>
__global__ void __maxnreg__(144)
discrete_qeval_kernel(const __grid_constant__ QevalParams qp) {
  QEvalAgent ag(qp.q);
  rollout_body<C>(qp.base, ag);
}

// The kernel variant of a learner or evaluation launch: tables and ring in
// shared memory when they fit, else the generic build
template <int NORMAL, typename KP>
static int launch_agent(mdpp_ctx* ctx, KP& kp, cudaStream_t stream,
                        void (*smem_kern)(KP), void (*gen_kern)(KP)) {
  RolloutParams& p = kp.base;
  bool ring_ok;
  if (tables_in_smem(ctx, p, &ring_ok) && ring_ok) {
    using Cs = Cfg<MDPP_NOISE_PHILOX, NORMAL, true, true, false, -1>;
    return launch_kernel<Cs>(ctx, p, ctx->max_group_blob, stream, smem_kern, kp);
  }
  using Cg = Cfg<MDPP_NOISE_PHILOX, NORMAL, false, false, false, -1>;
  return launch_kernel<Cg>(ctx, p, ctx->max_group_blob, stream, gen_kern, kp);
}

template <int NORMAL>
static int launch_qeval(mdpp_ctx* ctx, QevalParams& qp, cudaStream_t stream) {
  return launch_agent<NORMAL>(
      ctx, qp, stream,
      discrete_qeval_kernel<Cfg<MDPP_NOISE_PHILOX, NORMAL, true, true, false, -1>>,
      discrete_qeval_kernel<Cfg<MDPP_NOISE_PHILOX, NORMAL, false, false, false, -1>>);
}

template <int NORMAL>
static int launch_qlearn(mdpp_ctx* ctx, QlearnParams& qp, cudaStream_t stream) {
  return launch_agent<NORMAL>(
      ctx, qp, stream,
      discrete_qlearn_kernel<Cfg<MDPP_NOISE_PHILOX, NORMAL, true, true, false, -1>>,
      discrete_qlearn_kernel<Cfg<MDPP_NOISE_PHILOX, NORMAL, false, false, false, -1>>);
}

// A Q-table of q_states x q_actions rows must hold every group's S x A
static int check_q_table(mdpp_ctx* ctx, const char* who, int64_t q_states, int64_t q_actions,
                         int64_t n_states, int64_t n_actions) {
  if (q_states < n_states || q_actions < n_actions)
    return fail(ctx, MDPP_EINVAL,
                std::string(who) + ": q_states / q_actions smaller than a group's S / A");
  return MDPP_OK;
}

int check_qlearn_params(mdpp_ctx* ctx, const mdpp_qlearn_params* qp, int64_t n_states,
                        int64_t n_actions, QlearnDev* d) {
  if (!qp || !qp->q || !qp->ep_return || !qp->ret_sum || !qp->ret_count)
    return fail(ctx, MDPP_EINVAL, "qlearn: q, ep_return, ret_sum or ret_count is NULL");
  int rc = check_q_table(ctx, "qlearn", qp->q_states, qp->q_actions, n_states, n_actions);
  if (rc) return rc;
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
  d->ret = ReturnsDev{qp->ep_return, qp->ret_sum, qp->ret_count};
  d->actions_taken = qp->actions_taken;
  return MDPP_OK;
}

int check_eval_params(mdpp_ctx* ctx, const char* who, bool has_actions,
                      const mdpp_step_opts* opts, const mdpp_eval_params* ep,
                      int64_t n_states, int64_t n_actions, EvalDev* d) {
  const std::string w(who);
  if (has_actions) return fail(ctx, MDPP_EINVAL, w + ": io->actions must be NULL (the policy acts)");
  if (opts->noise_mode != MDPP_NOISE_PHILOX) return fail(ctx, MDPP_EINVAL, w + ": Philox noise only");
  if (!opts->autoreset)
    return fail(ctx, MDPP_EINVAL, w + ": needs autoreset (episodes end in an auto-reset)");
  if (opts->horizon < 1) return fail(ctx, MDPP_EINVAL, w + ": horizon must be >= 1");
  if (!ep) return fail(ctx, MDPP_EINVAL, w + ": params is NULL");
  if (ep->episodes < 1) return fail(ctx, MDPP_EINVAL, w + ": episodes must be >= 1");
  if (opts->n_steps < (int64_t)ep->episodes * opts->horizon)
    return fail(ctx, MDPP_EINVAL, w + ": n_steps must be >= episodes * horizon");
  const bool tabular = n_states >= 0;
  if ((tabular ? !ep->q : !ep->theta) || !ep->ret_sum || !ep->ret_count || !ep->len_sum)
    return fail(ctx, MDPP_EINVAL, w + (tabular ? ": q" : ": theta") +
                                      ", ret_sum, ret_count or len_sum is NULL");
  if (tabular) {
    int rc = check_q_table(ctx, who, ep->q_states, ep->q_actions, n_states, n_actions);
    if (rc) return rc;
  }
  *d = EvalDev{ep->ret_sum, ep->ret_count, ep->len_sum, ep->episodes};
  return MDPP_OK;
}

}  // namespace mdpp

using namespace mdpp;

extern "C" int mdpp_discrete_qeval(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                                   const mdpp_discrete_io* io, const mdpp_eval_params* ep,
                                   const mdpp_step_opts* opts, void* cuda_stream) {
  QevalParams k;
  int rc = prepare_rollout(ctx, st, io, opts, k.base);
  if (rc) return rc;
  if (ctx->d_irr)
    return fail(ctx, MDPP_EINVAL, "qeval: irrelevant features are not supported");
  int64_t S = 0, A = 0;
  for (auto& g : ctx->d_groups_host) {
    S = std::max<int64_t>(S, g.S);
    A = std::max<int64_t>(A, g.A);
  }
  rc = check_eval_params(ctx, "qeval", io->actions != nullptr, opts, ep, S, A, &k.q.ev);
  if (rc) return rc;
  k.q.q = ep->q;
  k.q.q_states = ep->q_states;
  k.q.q_actions = ep->q_actions;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  switch (opts->normal_mode) {
    case MDPP_NORMAL_FAST: return launch_qeval<MDPP_NORMAL_FAST>(ctx, k, s);
    case MDPP_NORMAL_ZIGGURAT: return launch_qeval<MDPP_NORMAL_ZIGGURAT>(ctx, k, s);
    default: return launch_qeval<MDPP_NORMAL_F64>(ctx, k, s);
  }
}

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
