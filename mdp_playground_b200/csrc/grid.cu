// Grid environments on sm_100a: K8 `grid_rollout` (T fused steps) and the
// (masked) reset.  Restates, per env and step, rl_toy_env.py
//   transition_function :1727-1778  unit move with wall bounce; with prob. p
//                                   the action is replaced by a different
//                                   GridActionSpace sample; invalid = no-op
//   reward_function     :1947-1965  Manhattan progress towards the target
//                                   (dense) or +1 on it (sparse)
//                       :1968-1990  every-n gate, noise, scale, shift
//   step epilogue       :2098-2109  done = sticky reached_terminal, terminal reward
//   reset               :2325-2345  every coordinate uniform on [0, shape]
// One thread = one env, the cell lives in registers for the whole launch; I/O
// is time-major with one 16- / 32-byte row per env and step (action rows are
// prefetched a step ahead).  Integer arithmetic and fp64 rewards in the
// reference's operation order: bit-exact.
// The second half of the file is mdpp_grid_qlearn: the same rollout kernel with
// a tabular Q-learner choosing the actions instead of the action rows.
#include <algorithm>
#include <cstring>
#include <vector>

#include "internal.h"
#include "tabular_q.cuh"
#include "philox.cuh"
#include "ziggurat.cuh"

namespace mdpp {

constexpr int kGBlock = 128;

struct GridParams {
  mdpp_grid_config cfg;
  mdpp_grid_state st;
  mdpp_grid_io io;
  int32_t T, autoreset, horizon, noise_mode, normal_mode;
  uint32_t k0, k1;
  uint64_t step_index;
  const uint64_t* step_index_dev;
  int64_t env_id_offset;
  // reset
  const uint8_t* mask;
  const int64_t* init_states;
  int64_t* reset_obs;
  uint32_t rk[20];     // Philox round keys (MDPP_NORMAL_ZIGGURAT draws)
  const uint8_t* zig;  // the context's ziggurat tables (ziggurat.cuh layout)
  // heterogeneous launches (mdpp_set_grid_groups): CTA -> (group, chunk of
  // kGBlock envs); every CTA reads its group's configuration from `groups`.
  const struct GridGroupDev* groups;
  const CtaMapEntry* cta_map;
  int32_t n_groups, reserved1;
};

// One configuration group of a heterogeneous grid launch (all groups share
// n_dims, i.e. the row layout of the state arrays and of the I/O).
struct GridGroupDev {
  mdpp_grid_config cfg;
  int64_t env_begin, env_count, gid_base;
};

struct GridSel {
  int64_t env;   // index into the state arrays
  uint32_t gid;
  bool active;
  int group;
};

// (shared-memory copy of the CTA's group; empty in single-configuration builds)
template <bool G> struct GridGroupSmem { GridGroupDev g; };
template <> struct GridGroupSmem<false> { int unused; };
__device__ __forceinline__ const mdpp_grid_config* group_cfg(const GridGroupSmem<true>& s) { return &s.g.cfg; }
__device__ __forceinline__ const mdpp_grid_config* group_cfg(const GridGroupSmem<false>&) { return nullptr; }

template <bool GROUPS>
__device__ __forceinline__ GridSel select_group(const GridParams& p,
                                                GridGroupSmem<GROUPS>& gsm) {
  GridSel s;
  if constexpr (GROUPS) {
    const CtaMapEntry me = p.cta_map[blockIdx.x];
    const uint32_t* src = reinterpret_cast<const uint32_t*>(p.groups + me.group);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&gsm.g);
    for (int i = threadIdx.x; i < (int)(sizeof(GridGroupDev) / 4); i += kGBlock)
      dst[i] = src[i];
    __syncthreads();
    const int64_t local = (int64_t)me.chunk * kGBlock + threadIdx.x;
    s.active = local < gsm.g.env_count;
    s.env = gsm.g.env_begin + (s.active ? local : 0);
    s.gid = (uint32_t)(p.env_id_offset + gsm.g.gid_base + (s.active ? local : 0));
    s.group = me.group;
  } else {
    const int64_t env = (int64_t)blockIdx.x * kGBlock + threadIdx.x;
    s.active = env < p.st.n_envs;
    s.env = s.active ? env : 0;
    s.gid = (uint32_t)(p.env_id_offset + s.env);
    s.group = 0;
  }
  return s;
}

template <int ND>
struct Row { int64_t v[ND]; };

template <int ND>
__device__ __forceinline__ Row<ND> ld_row(const int64_t* p) {
  Row<ND> r;
#pragma unroll
  for (int k = 0; k < ND; k += 2) {
    const longlong2 x = __ldcs(reinterpret_cast<const longlong2*>(p + k));
    r.v[k] = x.x; r.v[k + 1] = x.y;
  }
  return r;
}
// An action row, validated and packed: 2 bits per entry (value + 1), bit 31 =
// not a GridActionSpace member (-> no-op).
template <int ND>
__device__ __forceinline__ uint32_t pack_action(const Row<ND>& r) {
  uint32_t code = 0;
  bool valid = true;
  int moves = 0;
#pragma unroll
  for (int k = 0; k < ND; ++k) {
    const uint64_t u = (uint64_t)r.v[k] + 1ull;  // {-1, 0, 1} -> {0, 1, 2}
    valid &= u <= 2ull;
    moves += u != 1ull;
    code |= ((uint32_t)u & 3u) << (2 * k);
  }
  return (valid && moves <= 1) ? code : 0x80000000u;
}

// Q-table row of a cell: row-major over [0, shape_k] (reset draws the cell one
// past the grid too)
template <int ND>
__device__ __forceinline__ int32_t cell_index(const mdpp_grid_config& c, const int32_t* pos) {
  int32_t s = pos[0];
#pragma unroll
  for (int k = 1; k < ND; ++k) s = s * (c.shape[k] + 1) + pos[k];
  return s;
}

template <int ND>
__device__ __forceinline__ void st_row(int64_t* p, const int32_t* c) {
#pragma unroll
  for (int k = 0; k < ND; k += 2)
    __stcs(reinterpret_cast<longlong2*>(p + k), make_longlong2(c[k], c[k + 1]));
}

// Uniform over the GridActionSpace samples that differ from `a` (the
// reference's rejection loop :1737-1750 in closed form): a sample is (dim,
// value in {-1, 0, 1}), all ND zero-valued ones being the same no-op action.
template <int ND>
__device__ __forceinline__ void substitute_action(uint32_t w, int32_t* a) {
  int dim = -1, val = 0;  // the valid action as (dim, val); no-op: dim = -1
#pragma unroll
  for (int k = 0; k < ND; ++k)
    if (a[k] != 0) { dim = k; val = a[k]; }
  int pick;  // index into the 3 * ND samples (dim * 3 + val + 1)
  if (dim < 0) {  // current action is the no-op: one of the 2 * ND moves
    const int q = (int)__umulhi(w, 2u * ND);
    pick = (q >> 1) * 3 + ((q & 1) ? 2 : 0);
  } else {        // one of the other 3 * ND - 1 samples
    const int cur = dim * 3 + val + 1;
    const int q = (int)__umulhi(w, 3u * ND - 1u);
    pick = q + (q >= cur);
  }
#pragma unroll
  for (int k = 0; k < ND; ++k) a[k] = 0;
  const int d = (pick * 11) >> 5, v = pick - d * 3 - 1;  // pick / 3, pick < 12
#pragma unroll
  for (int k = 0; k < ND; ++k)
    if (k == d) a[k] = v;
}

__device__ __forceinline__ double block_sum(double x, double* smem) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = x;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int k = 0; k < kGBlock / 32; ++k) s += smem[k];
  __syncthreads();
  return s;
}

// Registers of one environment + the launch's running statistics.
template <int ND>
struct GridEnv {
  int32_t pos[ND];
  int32_t prev[2];    // relevant cell before the last step (-1: none yet)
  int32_t tl, phase;  // phase = tl % reward_every_n_steps, kept incrementally
  uint32_t ep;
  bool reached;
  double sum_reward, sum_abs_rnoise;
  uint32_t n_noisy, n_episodes, n_term;
  // Philox draws shared by consecutive steps (see grid_step)
  uint64_t cached_pair, cached_quad;
  U4 w_pair, w_zig;
  double zq[4];
};

// One environment step.  FAST: the standard rollout signature (obs, reward,
// terminated, truncated written, no final_obs), so no per-step NULL tests.
// NORMAL: generator of the reward normals (MDPP_NORMAL_*), a template
// parameter so that each kernel carries one generator's registers only.
// `so` (a learner's launch only): the step's outcome before any auto-reset.
template <int ND, int NOISE, bool FAST, int NORMAL>
__device__ __forceinline__ void grid_step(const GridParams& p, const mdpp_grid_config& c,
                                          GridEnv<ND>& g,
                                          uint32_t code, int64_t off, uint64_t step,
                                          uint32_t gid, uint32_t pn_T, double term_add,
                                          StepOut* so = nullptr) {
  // GridActionSpace.contains: entries in {-1, 0, 1}, at most one move
  const bool valid = (code >> 31) == 0;
  int32_t a[ND];
#pragma unroll
  for (int k = 0; k < ND; ++k)
    a[k] = valid ? (int32_t)((code >> (2 * k)) & 3u) - 1 : 0;
  // Philox draws are shared by consecutive steps (the step index is uniform
  // over the launch, so these refills are uniform branches):
  // STREAM_GRID_STEP, counter = step >> 1: words (0, 1) / (2, 3) = noise
  // decision and substitute action of the even / odd step;
  // STREAM_GRID_NORMAL, counter = step >> 2: two Box-Muller pairs = the reward
  // normals of 4 steps (MDPP_NORMAL_F64 / _FAST);
  // STREAM_GRID_ZIG, counter = step >> 1: the 64-bit ziggurat words of 2 steps
  // (MDPP_NORMAL_ZIGGURAT: numpy's Generator.normal algorithm.  Opt-in here:
  // the out-of-line call of its rare slow path makes the compiler keep part
  // of the env state in local memory -- 1.82 ms against 1.54 ms with fp64
  // Box-Muller for 1 M envs x 100 steps; the staged design of the discrete
  // rollout kernel has not been ported to this one)
  if (NOISE != MDPP_NOISE_OFF && c.has_transition_noise) {
    if (NOISE == MDPP_NOISE_REPLAY) {
      if (valid && __ldcs(p.io.replay_noise_u + off) < c.transition_noise) {
        const Row<ND> r = ld_row<ND>(p.io.replay_noise_action + off * ND);
#pragma unroll
        for (int k = 0; k < ND; ++k) a[k] = (int32_t)r.v[k];
        g.n_noisy += 1;
      }
    } else {
      if ((step >> 1) != g.cached_pair) {
        g.cached_pair = step >> 1;
        g.w_pair = philox4x32_10(gid, (uint32_t)g.cached_pair,
                                 (uint32_t)(g.cached_pair >> 32), STREAM_GRID_STEP,
                                 p.k0, p.k1);
      }
      const uint32_t w_u = (step & 1) ? g.w_pair.z : g.w_pair.x;
      const uint32_t w_sub = (step & 1) ? g.w_pair.w : g.w_pair.y;
      if (valid && w_u < pn_T) {
        substitute_action<ND>(w_sub, a);
        g.n_noisy += 1;
      }
    }
  }
  // dense reward: Manhattan distance moved towards the target
  const int d_old = abs(g.pos[0] - c.target[0]) + abs(g.pos[1] - c.target[1]);
  g.prev[0] = g.pos[0]; g.prev[1] = g.pos[1];
  if (valid) {
#pragma unroll
    for (int k = 0; k < ND; ++k) {
      int v = g.pos[k] + a[k];
      v = max(v, 0);                            // bounce back from the walls;
      g.pos[k] = min(v, c.shape[k] - 1);        // (also pulls a one-past reset
    }                                           //  cell in when it moves)
  }
  const bool at_target = g.pos[0] == c.target[0] && g.pos[1] == c.target[1];
  g.reached |= at_target;
  g.tl += 1;
  g.phase = (g.phase + 1 == c.reward_every_n_steps) ? 0 : g.phase + 1;
  double r = 0.0;
  if (c.dense) {
    const int d_new = abs(g.pos[0] - c.target[0]) + abs(g.pos[1] - c.target[1]);
    r = (double)(d_old - d_new);
  } else if (at_target) {
    r = 1.0;
  }
  if (g.phase != 0) r = 0.0;
  g.sum_reward += r;
  if (NOISE != MDPP_NOISE_OFF && c.has_reward_noise) {
    double z;
    if (NOISE == MDPP_NOISE_REPLAY) {
      z = __ldcs(p.io.replay_reward_noise + off);
    } else if (NORMAL == MDPP_NORMAL_ZIGGURAT) {
      if ((step >> 1) != g.cached_quad) {
        g.cached_quad = step >> 1;
        g.w_zig = philox4x32_10_rk(gid, (uint32_t)g.cached_quad,
                                   (uint32_t)(g.cached_quad >> 32), STREAM_GRID_ZIG, p.rk);
      }
      bool ok;
      double z0 = zig_first((step & 1) ? g.w_zig.z : g.w_zig.x,
                            (step & 1) ? g.w_zig.w : g.w_zig.y,
                            reinterpret_cast<const uint4*>(p.zig + kZigOffFast), &ok);
      if (!ok) z0 = zig_resolve_draw(gid, step, kZigDrawGridReward, p.rk, p.zig);
      z = __dmul_rn(c.reward_noise_std, z0);  // numpy: normal(0, sigma) = 0 + sigma * z
    } else {
      if ((step >> 2) != g.cached_quad) {
        g.cached_quad = step >> 2;
        const U4 wn = philox4x32_10(gid, (uint32_t)g.cached_quad,
                                    (uint32_t)(g.cached_quad >> 32),
                                    STREAM_GRID_NORMAL, p.k0, p.k1);
        if (NORMAL == MDPP_NORMAL_FAST) {
          normal_pair_fast(wn.x, wn.y, &g.zq[0], &g.zq[1]);
          normal_pair_fast(wn.z, wn.w, &g.zq[2], &g.zq[3]);
        } else {
          normal_pair_f64(wn.x, wn.y, &g.zq[0], &g.zq[1]);
          normal_pair_f64(wn.z, wn.w, &g.zq[2], &g.zq[3]);
        }
      }
      const int j4 = (int)(step & 3);
      const double z0 = j4 == 0 ? g.zq[0] : j4 == 1 ? g.zq[1] : j4 == 2 ? g.zq[2] : g.zq[3];
      z = __dmul_rn(c.reward_noise_std, z0);
    }
    g.sum_abs_rnoise += fabs(z);
    r = __dadd_rn(r, z);
  }
  r = __dmul_rn(r, c.reward_scale);
  r = __dadd_rn(r, c.reward_shift);
  const bool done = g.reached;
  if (done) r = __dadd_rn(r, term_add);
  const bool trunc = p.horizon > 0 && g.tl >= p.horizon;
  g.n_term += done;
  if (so) *so = StepOut{r, cell_index<ND>(c, g.pos), done, trunc};
  if (!FAST && p.io.final_obs) st_row<ND>(p.io.final_obs + off * ND, g.pos);
  if (p.autoreset && (done || trunc)) {
    if (NOISE == MDPP_NOISE_REPLAY) {
      const Row<ND> r0 = ld_row<ND>(p.io.replay_reset_state + off * ND);
#pragma unroll
      for (int k = 0; k < ND; ++k) g.pos[k] = (int32_t)r0.v[k];
    } else {
      U4 wr = philox4x32_10(gid, (uint32_t)step, (uint32_t)(step >> 32),
                            STREAM_GRID_AUTORESET, p.k0, p.k1);
      const uint32_t ww[4] = {wr.x, wr.y, wr.z, wr.w};
#pragma unroll
      for (int k = 0; k < ND; ++k)
        g.pos[k] = (int32_t)__umulhi(ww[k], (uint32_t)c.shape[k] + 1u);
    }
    g.tl = 0; g.phase = 0; g.ep += 1; g.reached = false; g.n_episodes += 1;
    g.prev[0] = g.prev[1] = -1;
  }
  if (FAST || p.io.obs) st_row<ND>(p.io.obs + off * ND, g.pos);
  if (FAST || p.io.reward) __stcs(p.io.reward + off, r);
  if (FAST || p.io.terminated) __stcs(p.io.terminated + off, (uint8_t)done);
  if (FAST || p.io.truncated) __stcs(p.io.truncated + off, (uint8_t)trunc);
}

// The rollout takes its actions from the action rows (NoGridAgent) or from a
// learner (GridQAgent below), which acts, sees each step's StepOut and the
// cell after any auto-reset, and loads / stores its per-env state around the
// launch (begin / end).  The agent also names the kernel's parameter struct
// and its occupancy target (kMinBlocks; 0: the rollout's own).
struct NoGridAgent {
  static constexpr bool kActs = false;
  static constexpr int kMinBlocks = 0;
  using Params = GridParams;
  __device__ __forceinline__ explicit NoGridAgent(const GridParams&) {}
};

template <int ND, int NOISE, bool FAST, bool GROUPS = false, int NORMAL = MDPP_NORMAL_F64,
          typename AG = NoGridAgent>
__global__ void __launch_bounds__(kGBlock, AG::kMinBlocks ? AG::kMinBlocks : ND == 2 ? 5 : 4)
grid_rollout_kernel(const __grid_constant__ typename AG::Params p) {
  AG ag(p);
  __shared__ double red[kGBlock / 32];
  __shared__ GridGroupSmem<GROUPS> gsm;
  const GridSel sel = select_group<GROUPS>(p, gsm);
  const mdpp_grid_config& c = GROUPS ? *group_cfg(gsm) : p.cfg;
  const int64_t N = p.st.n_envs;
  const bool active = sel.active;
  const int64_t e = sel.env;
  const uint32_t gid = sel.gid;
  const uint64_t step_base =
      p.step_index + (p.step_index_dev ? *p.step_index_dev : 0ull);
  GridEnv<ND> g;
#pragma unroll
  for (int k = 0; k < ND; ++k) g.pos[k] = p.st.pos[(int64_t)k * N + e];
  g.tl = p.st.t_episode[e];
  g.phase = g.tl % c.reward_every_n_steps;
  g.ep = p.st.episode[e];
  g.reached = p.st.reached[e] != 0;
  g.prev[0] = g.prev[1] = -1;
  g.sum_reward = g.sum_abs_rnoise = 0.0;
  g.n_noisy = g.n_episodes = g.n_term = 0;
  g.cached_pair = g.cached_quad = ~0ull;
  g.w_pair = g.w_zig = U4{0u, 0u, 0u, 0u};
  g.zq[0] = g.zq[1] = g.zq[2] = g.zq[3] = 0.0;
  const uint32_t pn_T = (uint32_t)fmin(
      floor(c.transition_noise * 4294967296.0 + 0.5), 4294967295.0);
  const double term_add = c.term_state_reward * c.reward_scale;
  if constexpr (AG::kActs) {
    if (active) {
      ag.begin(c, e, g.pos);
      for (int t = 0; t < p.T; ++t) {
        const int64_t off = (int64_t)t * N + e;
        const uint64_t step = step_base + (uint64_t)t;
        StepOut so;
        grid_step<ND, NOISE, FAST, NORMAL>(p, c, g, ag.act(p, gid, step), off, step, gid,
                                           pn_T, term_add, &so);
        ag.update(p, c, so, g.pos, e, off);
      }
      ag.end(e);
    }
  } else if (active) {
    // Action rows run 4 steps ahead of their use (a DRAM read under the
    // write-heavy stream takes longer than one step's arithmetic).  The ring
    // holds the RAW rows: touching a row before its turn would stall on the
    // load and void the prefetch.
    constexpr int kAhead = 4;
    const int64_t stride = N * ND;  // one time step of rows
    const int64_t* arow = p.io.actions + e * ND;
    Row<ND> ring[kAhead];
#pragma unroll
    for (int j = 0; j < kAhead; ++j) {
#pragma unroll
      for (int k = 0; k < ND; ++k) ring[j].v[k] = 2;  // invalid: no-op
      if (j < p.T) ring[j] = ld_row<ND>(arow + j * stride);
    }
    int t0 = 0;
    for (; t0 + kAhead <= p.T; t0 += kAhead) {  // whole groups, no step guards
      uint32_t cur[kAhead];
      const int64_t* nxt = arow + (int64_t)(t0 + kAhead) * stride;
#pragma unroll
      for (int j = 0; j < kAhead; ++j) {
        cur[j] = pack_action<ND>(ring[j]);
        if (t0 + kAhead + j < p.T) ring[j] = ld_row<ND>(nxt + j * stride);
      }
#pragma unroll
      for (int j = 0; j < kAhead; ++j)
        grid_step<ND, NOISE, FAST, NORMAL>(p, c, g, cur[j], (int64_t)(t0 + j) * N + e,
                                   step_base + (uint64_t)(t0 + j), gid, pn_T, term_add);
    }
#pragma unroll
    for (int j = 0; j < kAhead - 1; ++j)  // the last T % 4 steps
      if (t0 + j < p.T)
        grid_step<ND, NOISE, FAST, NORMAL>(p, c, g, pack_action<ND>(ring[j]),
                                   (int64_t)(t0 + j) * N + e,
                                   step_base + (uint64_t)(t0 + j), gid, pn_T, term_add);
  }
  if (active) {
#pragma unroll
    for (int k = 0; k < ND; ++k) p.st.pos[(int64_t)k * N + e] = g.pos[k];
    p.st.t_episode[e] = g.tl;
    p.st.episode[e] = g.ep;
    p.st.reached[e] = (uint8_t)g.reached;
    if (p.st.prev) {
      p.st.prev[e] = g.prev[0];
      p.st.prev[N + e] = g.prev[1];
    }
  }
  if (p.st.stats) {
    const double vals[MDPP_N_STATS] = {
        (double)g.n_episodes, active ? (double)p.T : 0.0, g.sum_reward,
        (double)g.n_noisy, g.sum_abs_rnoise, 0.0, 0.0, (double)g.n_term};
#pragma unroll
    for (int k = 0; k < MDPP_N_STATS; ++k) {
      if (k == MDPP_STAT_ABS_TRANSITION_NOISE || k == MDPP_STAT_RESERVED) continue;
      const double s = block_sum(vals[k], red);
      if (threadIdx.x == 0 && s != 0.0)  // rows [slot][group]
        atomicAdd(p.st.stats + ((int64_t)(blockIdx.x % (unsigned)max(p.st.stats_slots, 1)) *
                                    (GROUPS ? p.n_groups : 1) + sel.group) *
                                   MDPP_N_STATS + k, s);
    }
  }
}

template <int ND, bool GROUPS = false>
__global__ void __launch_bounds__(kGBlock)
grid_reset_kernel(const __grid_constant__ GridParams p) {
  __shared__ GridGroupSmem<GROUPS> gsm;
  const GridSel sel = select_group<GROUPS>(p, gsm);
  const mdpp_grid_config& c = GROUPS ? *group_cfg(gsm) : p.cfg;
  const int64_t N = p.st.n_envs;
  const int64_t env = sel.env;
  if (!sel.active) return;
  int32_t pos[ND];
  if (p.mask && !p.mask[env]) {
    if (p.reset_obs)
      for (int k = 0; k < ND; ++k)
        p.reset_obs[env * ND + k] = p.st.pos[(int64_t)k * N + env];
    return;
  }
  const uint32_t ep = p.st.episode[env];
  if (p.init_states) {
    for (int k = 0; k < ND; ++k) pos[k] = (int32_t)p.init_states[env * ND + k];
  } else {
    U4 w = philox4x32_10(sel.gid, ep, 0u, STREAM_GRID_RESET, p.k0, p.k1);
    const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
    for (int k = 0; k < ND; ++k)
      pos[k] = (int32_t)__umulhi(ww[k], (uint32_t)c.shape[k] + 1u);
  }
  if (p.st.stats && p.st.t_episode[env] > 0)
    atomicAdd(p.st.stats + ((int64_t)(blockIdx.x % (unsigned)max(p.st.stats_slots, 1)) *
                                (GROUPS ? p.n_groups : 1) + sel.group) *
                               MDPP_N_STATS + MDPP_STAT_EPISODES, 1.0);
  for (int k = 0; k < ND; ++k) {
    p.st.pos[(int64_t)k * N + env] = pos[k];
    if (p.reset_obs) p.reset_obs[env * ND + k] = pos[k];
  }
  p.st.t_episode[env] = 0;
  p.st.episode[env] = ep + 1;
  p.st.reached[env] = 0;
  if (p.st.prev) p.st.prev[env] = p.st.prev[N + env] = -1;
}

// ---- tabular Q-learning (mdpp_grid_qlearn) ----------------------------------
// Per env and step (global step `step`, Philox id g, cell index s):
//   w = philox(g, step >> 1, STREAM_GRID_ACTION), (x, y) / (z, w) = even / odd step
//   a = first word < ceil(epsilon * 2^32) ? umulhi(second word, A) : argmax Q[s]
//   step -> r, nxt (before any auto-reset), terminated
// then the update of TabularQ (tabular_q.cuh), like QAgent (qlearn.cu).
// Action index a: 0 = no-op, 1 + 2k = -1 on dim k, 2 + 2k = +1 on dim k.
// The host passes q_actions = 8 for 2-D grids, so a row is one 64-byte line.
struct GridQlearnParams : GridParams {
  QlearnDev q;
};

__device__ __forceinline__ bool autoreset_of(const GridParams& p) { return p.autoreset != 0; }

template <int ND>
struct GridQAgent : TabularQ<2 * ND + 1> {
  using Q = TabularQ<2 * ND + 1>;
  using Q::d; using Q::greedy; using Q::a;
  static constexpr bool kActs = true;
  // 65 536 envs are 512 CTAs of 128, 4 per SM on 148 SMs: at most 128
  // registers a thread keep them resident (one wave)
  static constexpr int kMinBlocks = 4;
  using Params = GridQlearnParams;
  static constexpr int A = 2 * ND + 1;
  uint64_t cached;  // step >> 1 of w
  U4 w;

  __device__ __forceinline__ explicit GridQAgent(const GridQlearnParams& p) : Q(p.q) {}

  __device__ __forceinline__ void begin(const mdpp_grid_config& c, int64_t env,
                                        const int32_t* pos) {
    Q::begin(env, [&] { return cell_index<ND>(c, pos); }, A);
    cached = ~0ull;
  }

  // the step's action, packed like pack_action
  __device__ __forceinline__ uint32_t act(const GridParams& p, uint32_t gid, uint64_t step) {
    if ((step >> 1) != cached) {  // uniform over the launch
      cached = step >> 1;
      w = philox4x32_10(gid, (uint32_t)cached, (uint32_t)(cached >> 32), STREAM_GRID_ACTION,
                        p.k0, p.k1);
    }
    const uint32_t w_explore = (step & 1) ? w.z : w.x;
    const uint32_t w_action = (step & 1) ? w.w : w.y;
    a = (uint64_t)w_explore < d.explore_below ? (int32_t)__umulhi(w_action, (uint32_t)A)
                                              : greedy;
    constexpr uint32_t noop = ND == 2 ? 0x5u : 0x55u;  // every entry 0 (code 1)
    const uint32_t one = 1u << (2 * ((a - 1) >> 1));
    return a == 0 ? noop : (a & 1) ? noop - one : noop + one;
  }

  __device__ __forceinline__ void update(const GridParams& p, const mdpp_grid_config& c,
                                         const StepOut& o, const int32_t* pos_after,
                                         int64_t env, int64_t off) {
    Q::update(p, o, A, env, [&] { return cell_index<ND>(c, pos_after); });
    if (d.actions_taken) __stcs(d.actions_taken + off, a);
  }
};

// ---- greedy evaluation (mdpp_grid_qeval) ------------------------------------
// a = argmax Q[s] (GreedyQ, tabular_q.cuh): no STREAM_GRID_ACTION draw.
struct GridQevalParams : GridParams {
  QevalDev q;
};

template <int ND>
struct GridQEvalAgent : GreedyQ<2 * ND + 1> {
  using Q = GreedyQ<2 * ND + 1>;
  using Q::greedy;
  static constexpr bool kActs = true;
  static constexpr int kMinBlocks = 4;  // the learner's: one wave at 65 536 envs
  using Params = GridQevalParams;
  static constexpr int A = 2 * ND + 1;

  __device__ __forceinline__ explicit GridQEvalAgent(const GridQevalParams& p) : Q(p.q) {}

  __device__ __forceinline__ void begin(const mdpp_grid_config& c, int64_t env,
                                        const int32_t* pos) {
    Q::begin(env, [&] { return cell_index<ND>(c, pos); }, A);
  }

  // the greedy action, packed like pack_action
  __device__ __forceinline__ uint32_t act(const GridParams&, uint32_t, uint64_t) const {
    const int32_t a = greedy;
    constexpr uint32_t noop = ND == 2 ? 0x5u : 0x55u;
    const uint32_t one = 1u << (2 * ((a - 1) >> 1));
    return a == 0 ? noop : (a & 1) ? noop - one : noop + one;
  }

  __device__ __forceinline__ void update(const GridParams& p, const mdpp_grid_config& c,
                                         const StepOut& o, const int32_t* pos_after,
                                         int64_t, int64_t) {
    Q::update(p, o, A, [&] { return cell_index<ND>(c, pos_after); });
  }
};

}  // namespace mdpp

using namespace mdpp;

// prod_k (shape_k + 1), the cells of a grid (one past the grid included),
// capped at 2^31
static int64_t grid_states(const mdpp_grid_config& c) {
  int64_t n = 1;
  for (int k = 0; k < c.n_dims; ++k)
    n = std::min<int64_t>(n * ((int64_t)c.shape[k] + 1), (int64_t)1 << 31);
  return n;
}

static int check_grid_config(mdpp_ctx* ctx, const mdpp_grid_config* cfg) {
  if (!cfg) return fail(ctx, MDPP_EINVAL, "cfg is NULL");
  if (cfg->n_dims != 2 && cfg->n_dims != 4)
    return fail(ctx, MDPP_EINVAL, "grid: n_dims must be 2 or 4");
  for (int k = 0; k < cfg->n_dims; ++k)
    if (cfg->shape[k] < 1)
      return fail(ctx, MDPP_EINVAL, "grid: bad grid_shape");
  if (cfg->reward_every_n_steps < 1)
    return fail(ctx, MDPP_EINVAL, "grid: bad reward_every_n_steps");
  if (cfg->has_transition_noise &&
      !(cfg->transition_noise > 0.0 && cfg->transition_noise <= 1.0))
    return fail(ctx, MDPP_EINVAL, "grid: transition_noise must be in (0, 1]");
  return MDPP_OK;
}

extern "C" int mdpp_set_grid_config(mdpp_ctx* ctx, const mdpp_grid_config* cfg) {
  if (!ctx) return MDPP_EINVAL;
  int rc = check_grid_config(ctx, cfg);
  if (rc) return rc;
  release_groups(ctx->g_set);
  ctx->g_cfg = *cfg;
  ctx->g_states = grid_states(*cfg);
  ctx->have_grid = true;
  return MDPP_OK;
}

extern "C" int mdpp_set_grid_groups(mdpp_ctx* ctx, const mdpp_grid_group* groups,
                                    int32_t n_groups) {
  if (!ctx) return MDPP_EINVAL;
  int rc = validate_groups(ctx, __func__, groups, n_groups, /*env_map=*/false);
  if (rc) return rc;
  std::vector<GridGroupDev> dev(n_groups);
  // the launch-wide view: flags any group has (which replay arrays are needed)
  mdpp_grid_config view = groups[0].cfg;
  int64_t states = 0;
  for (int g = 0; g < n_groups; ++g) {
    const mdpp_grid_config& c = groups[g].cfg;
    rc = check_grid_config(ctx, &c);
    if (rc) return rc;
    if (c.n_dims != groups[0].cfg.n_dims)  // the row layout of state and I/O
      return fail(ctx, MDPP_EINVAL, "grid groups must agree on n_dims");
    std::memset(&dev[g], 0, sizeof dev[g]);
    dev[g].cfg = c;
    dev[g].env_begin = groups[g].env_begin;
    dev[g].env_count = groups[g].env_count;
    dev[g].gid_base = groups[g].global_id_base;
    view.has_transition_noise |= c.has_transition_noise;
    view.has_reward_noise |= c.has_reward_noise;
    states = std::max(states, grid_states(c));
  }
  rc = install_groups(ctx, ctx->g_set, dev.data(), n_groups, kGBlock);
  if (rc) return rc;
  ctx->g_cfg = view;
  ctx->g_states = states;
  ctx->have_grid = true;
  return MDPP_OK;
}

static int fill_grid(mdpp_ctx* ctx, const mdpp_grid_state* st,
                     const mdpp_step_opts* opts, GridParams* p) {
  if (!ctx) return MDPP_EINVAL;
  if (!ctx->have_grid)
    return fail(ctx, MDPP_EINVAL, "mdpp_set_grid_config was not called");
  if (!st || !st->pos || !st->t_episode || !st->episode || !st->reached ||
      st->n_envs < 1)
    return fail(ctx, MDPP_EINVAL, "grid state has NULL arrays");
  if (!opts) return fail(ctx, MDPP_EINVAL, "opts is NULL");
  std::memset(p, 0, sizeof(*p));
  p->cfg = ctx->g_cfg;
  p->st = *st;
  p->T = opts->n_steps;
  p->autoreset = opts->autoreset;
  p->horizon = opts->horizon;
  p->noise_mode = opts->noise_mode;
  p->normal_mode = opts->normal_mode;
  p->k0 = (uint32_t)opts->seed;
  p->k1 = (uint32_t)(opts->seed >> 32);
  p->step_index = opts->step_index;
  p->step_index_dev = opts->step_index_dev;
  p->env_id_offset = opts->env_id_offset;
  philox_round_keys(p->k0, p->k1, p->rk);
  p->zig = ctx->d_zig;
  if (ctx->g_set.n_groups > 0) {
    int rc = bind_groups(ctx, ctx->g_set, "grid launch", st->n_envs);
    if (rc) return rc;
    p->groups = static_cast<const GridGroupDev*>(ctx->g_set.groups);
    p->cta_map = ctx->g_set.cta_map;
    p->n_groups = ctx->g_set.n_groups;
  }
  return MDPP_OK;
}

// CTAs of a grid launch: the group set's, or one per kGBlock envs
static unsigned grid_ctas(const mdpp_ctx* ctx, const GridParams& p) {
  return p.groups ? (unsigned)ctx->g_set.n_ctas
                  : (unsigned)((p.st.n_envs + kGBlock - 1) / kGBlock);
}

// The Philox-noise rollout with agent AG acting, one kernel per generator of
// the reward normals (p.normal_mode)
template <int ND, bool FAST, bool GROUPS, typename AG>
static int launch_grid_philox(mdpp_ctx* ctx, const typename AG::Params& p, cudaStream_t s) {
  const unsigned grid = grid_ctas(ctx, p);
  if (p.normal_mode == MDPP_NORMAL_ZIGGURAT)
    grid_rollout_kernel<ND, MDPP_NOISE_PHILOX, FAST, GROUPS, MDPP_NORMAL_ZIGGURAT, AG>
        <<<grid, kGBlock, 0, s>>>(p);
  else if (p.normal_mode == MDPP_NORMAL_FAST)
    grid_rollout_kernel<ND, MDPP_NOISE_PHILOX, FAST, GROUPS, MDPP_NORMAL_FAST, AG>
        <<<grid, kGBlock, 0, s>>>(p);
  else
    grid_rollout_kernel<ND, MDPP_NOISE_PHILOX, FAST, GROUPS, MDPP_NORMAL_F64, AG>
        <<<grid, kGBlock, 0, s>>>(p);
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

template <int ND, bool FAST, bool GROUPS>
static int launch_grid(mdpp_ctx* ctx, const GridParams& p, cudaStream_t s) {
  if (p.noise_mode == MDPP_NOISE_PHILOX)
    return launch_grid_philox<ND, FAST, GROUPS, NoGridAgent>(ctx, p, s);
  const unsigned grid = grid_ctas(ctx, p);
  if (p.noise_mode == MDPP_NOISE_OFF)
    grid_rollout_kernel<ND, MDPP_NOISE_OFF, FAST, GROUPS><<<grid, kGBlock, 0, s>>>(p);
  else
    grid_rollout_kernel<ND, MDPP_NOISE_REPLAY, FAST, GROUPS><<<grid, kGBlock, 0, s>>>(p);
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

extern "C" int mdpp_grid_rollout(mdpp_ctx* ctx, const mdpp_grid_state* st,
                                 const mdpp_grid_io* io,
                                 const mdpp_step_opts* opts, void* cuda_stream) {
  GridParams p;
  int rc = fill_grid(ctx, st, opts, &p);
  if (rc) return rc;
  if (!io || !io->actions || opts->n_steps < 1)
    return fail(ctx, MDPP_EINVAL, "grid rollout needs actions and T >= 1");
  if (opts->noise_mode < MDPP_NOISE_OFF || opts->noise_mode > MDPP_NOISE_PHILOX)
    return fail(ctx, MDPP_EINVAL, "unknown noise_mode");
  if (opts->noise_mode == MDPP_NOISE_REPLAY) {
    if ((ctx->g_cfg.has_transition_noise &&
         (!io->replay_noise_u || !io->replay_noise_action)) ||
        (ctx->g_cfg.has_reward_noise && !io->replay_reward_noise) ||
        (opts->autoreset && !io->replay_reset_state))
      return fail(ctx, MDPP_EINVAL, "replay mode: missing replay array");
  }
  if (((uintptr_t)io->actions | (uintptr_t)io->obs | (uintptr_t)io->final_obs |
       (uintptr_t)io->replay_noise_action | (uintptr_t)io->replay_reset_state) & 15)
    return fail(ctx, MDPP_EINVAL, "grid rows must be 16-byte aligned");
  p.io = *io;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool fast = io->obs && io->reward && io->terminated && io->truncated &&
                    !io->final_obs;
  if (p.groups) {  // heterogeneous launch: every CTA under its own group's scalars
    if (ctx->g_cfg.n_dims == 4)
      return fast ? launch_grid<4, true, true>(ctx, p, s)
                  : launch_grid<4, false, true>(ctx, p, s);
    return fast ? launch_grid<2, true, true>(ctx, p, s)
                : launch_grid<2, false, true>(ctx, p, s);
  }
  if (ctx->g_cfg.n_dims == 4)
    return fast ? launch_grid<4, true, false>(ctx, p, s)
                : launch_grid<4, false, false>(ctx, p, s);
  return fast ? launch_grid<2, true, false>(ctx, p, s)
              : launch_grid<2, false, false>(ctx, p, s);
}

extern "C" int mdpp_grid_reset(mdpp_ctx* ctx, const mdpp_grid_state* st,
                               const uint8_t* mask, const int64_t* init_states,
                               int64_t* obs, const mdpp_step_opts* opts,
                               void* cuda_stream) {
  GridParams p;
  int rc = fill_grid(ctx, st, opts, &p);
  if (rc) return rc;
  if (!init_states && opts->noise_mode == MDPP_NOISE_REPLAY)
    return fail(ctx, MDPP_EINVAL, "replay reset needs init_states");
  p.mask = mask;
  p.init_states = init_states;
  p.reset_obs = obs;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned grid = grid_ctas(ctx, p);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (p.groups && ctx->g_cfg.n_dims == 4) grid_reset_kernel<4, true><<<grid, kGBlock, 0, s>>>(p);
  else if (p.groups) grid_reset_kernel<2, true><<<grid, kGBlock, 0, s>>>(p);
  else if (ctx->g_cfg.n_dims == 4) grid_reset_kernel<4><<<grid, kGBlock, 0, s>>>(p);
  else grid_reset_kernel<2><<<grid, kGBlock, 0, s>>>(p);
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

extern "C" int mdpp_grid_qlearn(mdpp_ctx* ctx, const mdpp_grid_state* st,
                                const mdpp_grid_io* io, const mdpp_qlearn_params* qp,
                                const mdpp_step_opts* opts, void* cuda_stream) {
  GridQlearnParams k;
  int rc = fill_grid(ctx, st, opts, &k);
  if (rc) return rc;
  if (!io) return fail(ctx, MDPP_EINVAL, "grid qlearn: io is NULL");
  if (io->actions)
    return fail(ctx, MDPP_EINVAL, "grid qlearn: io->actions must be NULL (the agent acts)");
  if (opts->noise_mode != MDPP_NOISE_PHILOX)
    return fail(ctx, MDPP_EINVAL, "grid qlearn: Philox noise only");
  if (opts->n_steps < 1) return fail(ctx, MDPP_EINVAL, "grid qlearn: T must be >= 1");
  if (ctx->g_states > INT32_MAX)
    return fail(ctx, MDPP_EINVAL, "grid qlearn: a group has more than 2^31 - 1 cells");
  const int nd = ctx->g_cfg.n_dims;
  rc = check_qlearn_params(ctx, qp, ctx->g_states, 2 * nd + 1, &k.q);
  if (rc) return rc;
  if (((uintptr_t)io->obs | (uintptr_t)io->final_obs) & 15)
    return fail(ctx, MDPP_EINVAL, "grid rows must be 16-byte aligned");
  k.io = *io;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (k.groups)
    return nd == 4 ? launch_grid_philox<4, false, true, GridQAgent<4>>(ctx, k, s)
                   : launch_grid_philox<2, false, true, GridQAgent<2>>(ctx, k, s);
  return nd == 4 ? launch_grid_philox<4, false, false, GridQAgent<4>>(ctx, k, s)
                 : launch_grid_philox<2, false, false, GridQAgent<2>>(ctx, k, s);
}

extern "C" int mdpp_grid_qeval(mdpp_ctx* ctx, const mdpp_grid_state* st,
                               const mdpp_grid_io* io, const mdpp_eval_params* ep,
                               const mdpp_step_opts* opts, void* cuda_stream) {
  GridQevalParams k;
  int rc = fill_grid(ctx, st, opts, &k);
  if (rc) return rc;
  if (!io) return fail(ctx, MDPP_EINVAL, "grid qeval: io is NULL");
  if (ctx->g_states > INT32_MAX)
    return fail(ctx, MDPP_EINVAL, "grid qeval: a group has more than 2^31 - 1 cells");
  const int nd = ctx->g_cfg.n_dims;
  rc = check_eval_params(ctx, "grid qeval", io->actions != nullptr, opts, ep, ctx->g_states,
                         2 * nd + 1, &k.q.ev);
  if (rc) return rc;
  if (((uintptr_t)io->obs | (uintptr_t)io->final_obs) & 15)
    return fail(ctx, MDPP_EINVAL, "grid rows must be 16-byte aligned");
  k.q.q = ep->q;
  k.q.q_states = ep->q_states;
  k.q.q_actions = ep->q_actions;
  k.io = *io;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (k.groups)
    return nd == 4 ? launch_grid_philox<4, false, true, GridQEvalAgent<4>>(ctx, k, s)
                   : launch_grid_philox<2, false, true, GridQEvalAgent<2>>(ctx, k, s);
  return nd == 4 ? launch_grid_philox<4, false, false, GridQEvalAgent<4>>(ctx, k, s)
                 : launch_grid_philox<2, false, false, GridQEvalAgent<2>>(ctx, k, s);
}
