// The tabular Q-learning core of the learners riding along a rollout kernel
// (QAgent in qlearn.cu, GridQAgent in grid.cu).  Every float64 operation is
// an explicit _rn intrinsic (no FMA contraction), so a numpy restatement in
// the same order gives the same bits (tests/qlearn_oracle.py,
// tests/grid_qlearn_oracle.py).
#pragma once
#include "device_types.h"

namespace mdpp {

// (max, lowest argmax) of a Q row; numpy.argmax order.  A > 0: A entries
// known at compile time, scanned fully unrolled; A == 0: `n` entries, a
// run-time bound (unrolled by 4).
template <int A>
__device__ __forceinline__ int32_t row_argmax(const double* row, int n, double& m) {
  m = row[0];
  int32_t am = 0;
  if constexpr (A > 0) {
#pragma unroll
    for (int k = 1; k < A; ++k) {
      const double x = row[k];
      if (x > m) { m = x; am = k; }
    }
  } else {
#pragma unroll 4
    for (int k = 1; k < n; ++k) {
      const double x = row[k];
      if (x > m) { m = x; am = k; }
    }
  }
  return am;
}

// One env's tabular Q-learner.  Per step (state s, action a):
//   target = terminated ? r : r + gamma * max_a' Q[nxt][a']
//   Q[s][a] = q + alpha * (target - q)
//   ep_return += r; an episode that ends in an auto-reset adds its return to
//   ret_sum and one to ret_count (ReturnsDev), and the next starts at 0
// Q is float64 [N][q_states][q_actions], env-major.  The greedy action of the
// current state is tracked incrementally: the row Q[nxt] that the target
// loads also gives the next step's argmax unless an auto-reset follows.
// A > 0: rows of A actions known at compile time, scanned fully unrolled;
// A == 0: the scan's bound `n` is a run-time value (unrolled by 4).  The
// agent's launch parameters P give autoreset_of(p).  The states come as
// functors, evaluated where the agents computed them before this core was
// shared: their SASS depends on that order.
template <int A>
struct TabularQ {
  const QlearnDev& d;
  double* tab;        // this env's Q-table
  int32_t greedy;     // argmax of the current state's row
  int32_t s, a;       // the step's state and action
  double ep_ret;      // return of the running episode

  __device__ __forceinline__ explicit TabularQ(const QlearnDev& dev) : d(dev) {}

  // (max, lowest argmax) of row st; numpy.argmax order
  __device__ __forceinline__ int32_t row_argmax(int32_t st, int n, double& m) const {
    return mdpp::row_argmax<A>(tab + (int64_t)st * d.q_actions, n, m);
  }

  // state(): the env's state at the start of the launch
  template <typename F>
  __device__ __forceinline__ void begin(int64_t env, F state, int n) {
    tab = d.q + env * (int64_t)d.q_states * d.q_actions;
    s = state();
    double m;
    greedy = row_argmax(s, n, m);
    ep_ret = d.ret.ep_return[env];
  }

  // The update of Q[s][a] from the step's outcome o, then the state the env
  // is in now (o.nxt, or state_after() after an auto-reset), its greedy
  // action and the episode return.
  template <typename P, typename F>
  __device__ __forceinline__ void update(const P& p, const StepOut& o, int n, int64_t env,
                                         F state_after) {
    double* q_at = tab + (int64_t)s * d.q_actions + a;
    const double q = *q_at;  // (loaded beside the row of nxt)
    double m;
    const int32_t am = row_argmax(o.nxt, n, m);
    const double target = o.done ? o.r : __dadd_rn(o.r, __dmul_rn(d.gamma, m));
    const double qn = __dadd_rn(q, __dmul_rn(d.alpha, __dsub_rn(target, q)));
    *q_at = qn;
    const bool reset = autoreset_of(p) && (o.done || o.trunc);
    if (reset) {
      const int32_t s_after = state_after();
      greedy = row_argmax(s_after, n, m);
      s = s_after;
    } else {
      if (o.nxt != s) {
        greedy = am;
      } else if (a != am) {  // the row just loaded changed in entry a only
        greedy = (qn > m || (qn == m && a < am)) ? a : am;
      } else {  // the maximum itself changed: rescan unless it only grew
        greedy = qn >= m ? am : row_argmax(s, n, m);
      }
      s = o.nxt;
    }
    ep_ret = __dadd_rn(ep_ret, o.r);
    if (reset) {
      d.ret.ret_sum[env] = __dadd_rn(d.ret.ret_sum[env], ep_ret);
      d.ret.ret_count[env] += 1;
      ep_ret = 0.0;
    }
  }

  __device__ __forceinline__ void end(int64_t env) { d.ret.ep_return[env] = ep_ret; }
};

// One env's greedy policy over a fixed Q-table, for the evaluation launches
// (mdpp_discrete_qeval, mdpp_grid_qeval): the action is always
// argmax_a Q[s][a] (lowest index on ties), Q is only read, and the return and
// length of the first ev.episodes episodes go to EvalEpisodes.  Per step one
// row is loaded: that of the state the env is in after the step (o.nxt, or
// state_after() after an auto-reset), whose argmax is the next action.
template <int A>
struct GreedyQ {
  const QevalDev& d;
  const double* tab;  // this env's Q-table
  int32_t greedy;     // argmax of the current state's row
  EvalEpisodes ep;

  __device__ __forceinline__ explicit GreedyQ(const QevalDev& dev) : d(dev) {}

  __device__ __forceinline__ int32_t argmax_of(int32_t st, int n) const {
    double m;
    return row_argmax<A>(tab + (int64_t)st * d.q_actions, n, m);
  }

  template <typename F>
  __device__ __forceinline__ void begin(int64_t env, F state, int n) {
    tab = d.q + env * (int64_t)d.q_states * d.q_actions;
    greedy = argmax_of(state(), n);
    ep.begin();
  }

  template <typename P, typename F>
  __device__ __forceinline__ void update(const P& p, const StepOut& o, int n, F state_after) {
    const bool ended = o.done || o.trunc;
    greedy = argmax_of(autoreset_of(p) && ended ? state_after() : o.nxt, n);
    ep.step(d.ev, o.r, ended);
  }

  __device__ __forceinline__ void end(int64_t env) const { ep.end(d.ev, env); }
};

}  // namespace mdpp
