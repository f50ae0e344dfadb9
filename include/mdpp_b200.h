/*
 * mdpp_b200.h -- C ABI of the B200-native RLToyEnv step path.
 *
 * The reference (automl/mdp-playground) has no FFI: its boundary is the
 * Python class `RLToyEnv` (mdp_playground/envs/rl_toy_env.py:216 ctor,
 * :2217 reset, :1992 step).  This header is the C-ABI a binding for that
 * class calls into; `mdp_playground_b200/vector_env.py` is that binding
 * (ctypes) and INTEGRATION.md shows the stub a reference maintainer would
 * add.  Plain pointers and sizes only; every device buffer is owned by the
 * caller (PyTorch in our binding) and borrowed for the duration of a call.
 * All launches are enqueued on the caller's stream; nothing synchronises.
 *
 * Every function returns 0 on success or a negative MDPP_E* code;
 * mdpp_last_error() returns the message of the last failure on that context
 * (or of the last failed mdpp_create when ctx == NULL).
 */
#ifndef MDPP_B200_H
#define MDPP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDPP_ABI_VERSION 4

#define MDPP_OK 0
#define MDPP_EINVAL (-1)   /* bad argument / unsupported configuration      */
#define MDPP_ECUDA (-2)    /* a CUDA runtime call or launch failed          */
#define MDPP_ENOMEM (-3)

/* Where the step path's random draws come from (SURVEY.md 8b "Modes").     */
#define MDPP_NOISE_OFF 0     /* no draw is consumed                         */
#define MDPP_NOISE_REPLAY 1  /* draws are read from caller-provided arrays  */
#define MDPP_NOISE_PHILOX 2  /* Philox4x32-10, counter = (env, step, stream)*/

/* Per-group episode statistics (rl_toy_env.py:2360-2369 counters, summed
 * over envs and episodes).  Layout of one row of `stats`.                  */
#define MDPP_STAT_EPISODES 0          /* episodes ended (auto-reset or reset()) */
#define MDPP_STAT_TRANSITIONS 1       /* total_transitions_episode          */
#define MDPP_STAT_REWARD 2            /* total_reward_episode (pre-noise)   */
#define MDPP_STAT_NOISY_TRANSITIONS 3 /* total_noisy_transitions_episode    */
#define MDPP_STAT_ABS_REWARD_NOISE 4  /* total_abs_noise_in_reward_episode  */
#define MDPP_STAT_ABS_TRANSITION_NOISE 5 /* ..._in_transition_episode (sum over dims) */
#define MDPP_STAT_RESERVED 6
#define MDPP_STAT_TERMINATED 7        /* steps that returned terminated     */
#define MDPP_N_STATS 8

typedef struct mdpp_ctx mdpp_ctx;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_abi_version(void);
int mdpp_create(int device, mdpp_ctx** out_ctx);
void mdpp_destroy(mdpp_ctx* ctx);
const char* mdpp_last_error(const mdpp_ctx* ctx);
/* Host copies of the ziggurat tables behind MDPP_NORMAL_ZIGGURAT (numpy's
 * ki_double / wi_double / fi_double, doubles as bit patterns), 256 entries
 * each; for tests -- no GPU needed.                                         */
void mdpp_ziggurat_tables(const uint64_t** ki, const uint64_t** wi_bits,
                          const uint64_t** fi_bits);
#endif

/* Runtime specialisation (NVRTC) of the rollout kernel for single-group
 * launches.  On by default (MDPP_JIT=0 in the environment, or
 * mdpp_set_jit(ctx, 0), disables it; the ahead-of-time kernels then run).
 * mdpp_jit_last_used() tells whether the last rollout ran a specialised
 * kernel, mdpp_jit_log() why not.  mdpp_jit_selftest() compiles (does not
 * load) one specialisation with NVRTC only -- no GPU needed -- and returns 0
 * on success, copying the compiler log into `log`.                          */
#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
void mdpp_set_jit(mdpp_ctx* ctx, int enabled);
int mdpp_jit_last_used(const mdpp_ctx* ctx);
const char* mdpp_jit_log(const mdpp_ctx* ctx);
int mdpp_jit_selftest(char* log, int log_bytes);
#endif

/* ------------------------------------------------------------------------
 * Discrete environments (replaces RLToyEnv.transition_function :1602-1622,
 * reward_function :1817-1846 + tail :1968-1990, step epilogue :2098-2125,
 * reset :2250-2278).
 * --------------------------------------------------------------------- */

/* One configuration group = one (P, R, scalars) set shared by a contiguous
 * range of environments.  All pointers are HOST pointers, copied during the
 * call.  Tables come from the host-side generators (seeded numpy, same draws
 * as init_transition_function :1042 / init_reward_function :1253).        */
typedef struct mdpp_discrete_group {
  int32_t n_states;              /* S                                        */
  int32_t n_actions;             /* A                                        */
  int32_t sequence_length;       /* L >= 1                                   */
  int32_t delay;                 /* d >= 0                                   */
  int32_t reward_every_n_steps;  /* >= 1                                     */
  int32_t custom_reward;         /* 1: r = R[s, a] (use_custom_mdp :1817)    */
  int32_t n_sequences;           /* full-length rewardable sequences         */
  int32_t has_transition_noise;  /* truthy transition_noise (:1604)          */
  int32_t has_reward_noise;      /* "reward_noise" key present (:398, :1982) */
  int32_t reserved0;
  double transition_noise;       /* p: MDPP_NOISE_PHILOX draws the noisy state
                                    from (p, S) in closed form -- P[s,a] w.p.
                                    1 - p, each other state p / (S - 1), the
                                    distribution of :1606-1617               */
  double reward_noise_std;       /* sigma                                    */
  double reward_scale;
  double reward_shift;
  double term_state_reward;
  const int32_t* transition;     /* [S*A]  P[s,a]                            */
  const uint8_t* terminal;       /* [S]    1 = terminal                      */
  const double* init_cdf;        /* [S]    cumsum(init_dist)/last            */
  const double* noise_cdf;       /* [S*S]  row s' = cdf of the noisy draw
                                           around s' (:1605-1612), searched with
                                           the recorded uniform in
                                           MDPP_NOISE_REPLAY; may be NULL when
                                           !has_transition_noise             */
  const int32_t* sequences;      /* [n_sequences*L] rewardable sequences     */
  const double* sequence_rewards;/* [n_sequences]                            */
  const double* reward_matrix;   /* [S*A] when custom_reward, else NULL      */
  int64_t env_begin;             /* first env (local index) of the group     */
  int64_t env_count;
  int64_t global_id_base;        /* Philox id of the group's first env, added
                                    to opts->env_id_offset: keeps the noise of
                                    an env independent of how groups / envs
                                    are sharded over GPUs                    */
  /* irrelevant_features (:1154-1230, :2062-2082, :2260-2264): a second,
   * reward-free sub-MDP with its own transition table, uniform start and the
   * same transition_noise p.  n_states_irr == 0 = none; all groups of a
   * context must agree on having one.                                       */
  int32_t n_states_irr;          /* S1                                       */
  int32_t n_actions_irr;         /* A1                                       */
  const int32_t* transition_irr; /* [S1*A1]                                  */
  const double* init_cdf_irr;    /* [S1]                                     */
  const double* noise_cdf_irr;   /* [S1*S1], may be NULL without noise       */
} mdpp_discrete_group;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_set_discrete_groups(mdpp_ctx* ctx, const mdpp_discrete_group* groups,
                             int32_t n_groups);
#endif

/* Persistent per-env state, struct-of-arrays, DEVICE pointers owned by the
 * caller.  `ring` holds the reward-delay FIFO (:1970-1973) as a ring of
 * `ring_depth` rows (>= max delay over groups; NULL when that is 0).
 * `history` (optional) keeps the last `history_depth` emitted states so the
 * binding can rebuild `augmented_state` (:2127).                           */
typedef struct mdpp_discrete_state {
  int64_t n_envs;
  int32_t* cur_state;   /* [N]                                              */
  uint64_t* seq_key;    /* [N] last L states, key_bits each, newest lowest  */
  int32_t* t_episode;   /* [N] total_transitions_episode                    */
  uint32_t* episode;    /* [N] episodes started (reset-draw counter)        */
  double* ring;         /* [ring_depth*N] or NULL                           */
  int32_t ring_depth;
  int32_t history_depth;
  int32_t* history;     /* [history_depth*N] or NULL                        */
  double* stats;        /* [stats_slots][n_groups][MDPP_N_STATS], accumulated
                           atomically; the counters are the SUM over slots   */
  int32_t* cur_state_irr; /* [N] irrelevant sub-state (irrelevant_features)  */
  int32_t stats_slots;  /* >= 1 (0 reads as 1): CTAs spread their atomics over
                           this many copies of the counter rows -- thousands
                           of same-address fp64 atomics were 15 of the 19 us
                           of a T = 1 launch                                  */
  int32_t reserved1;
} mdpp_discrete_state;

/* Inputs/outputs of T consecutive steps, time-major [T*N], DEVICE pointers.
 * Any output pointer may be NULL (that output is skipped).
 * With irrelevant_features every state-like quantity is a ROW OF 2 per env,
 * (relevant, irrelevant) -- the reference's (s, s_irr) tuples (:2085-2088):
 * actions, obs, final_obs, replay_transition_u and replay_reset_u are then
 * [T*N*2] (one 8- / 16-byte vector access per env and step).                */
typedef struct mdpp_discrete_io {
  const int32_t* actions;            /* [T*N]; NULL => uniform Philox policy */
  int64_t* obs;                      /* [T*N] state after the step (after the
                                        auto-reset when one happened)        */
  int64_t* final_obs;                /* [T*N] state before any auto-reset    */
  double* reward;                    /* [T*N]                                */
  uint8_t* terminated;               /* [T*N]                                */
  uint8_t* truncated;                /* [T*N]                                */
  const double* replay_transition_u; /* [T*N] uniform of choice(p=) (:1612)  */
  const double* replay_reward_noise; /* [T*N] value of normal(0,sigma) :1982 */
  const double* replay_reset_u;      /* [T*N] uniform of the reset choice    */
  int32_t obs_dtype;                 /* element type of obs / final_obs: the
                                        reference's dtype_o (rl_toy_env.py:571,
                                        :611-614); MDPP_OBS_I64 (default, the
                                        pointers above), _I32 or _U8: the same
                                        pointers then address int32_t / uint8_t
                                        arrays of the same shape              */
  int32_t reserved0;
} mdpp_discrete_io;
#define MDPP_OBS_I64 0
#define MDPP_OBS_I32 1
#define MDPP_OBS_U8 2

/* How the Philox mode turns words into N(0,1) noise (reward noise; the
 * transition noise of continuous envs).                                     */
#define MDPP_NORMAL_F64 0   /* Box-Muller in fp64 (log, sqrt, sincospi)      */
#define MDPP_NORMAL_FAST 1  /* Box-Muller on the SFU in fp32 (~1e-6 rel.)    */
#define MDPP_NORMAL_ZIGGURAT 2 /* fp64, numpy's 256-layer ziggurat (the
                                  algorithm behind Generator.normal, which the
                                  reference calls at rl_toy_env.py:1683 and
                                  :1982) on Philox words.  The fastest fp64
                                  generator of the discrete kernels (staged in
                                  shared memory); the continuous and grid
                                  kernels run it too, but slower than
                                  MDPP_NORMAL_F64 (direct draws)              */

/* mdpp_render_discrete only: the launch may START before the previous kernel
 * of the stream has finished (programmatic dependent launch): its prologue --
 * the zero fill of `out` -- depends on nothing; it waits for that kernel
 * before it reads `states`.  The rollout kernels signal their dependents at
 * once, so a step -> render pair overlaps.  `out` must not be read or written
 * by the previous kernel.                                                    */
#define MDPP_LAUNCH_OVERLAP_PREVIOUS 1

typedef struct mdpp_step_opts {
  int32_t n_steps;        /* T >= 1                                          */
  int32_t noise_mode;     /* MDPP_NOISE_*                                    */
  int32_t autoreset;      /* 1: reset in the same step on terminated/truncated */
  int32_t horizon;        /* > 0: truncated = (t_episode >= horizon)         */
  int32_t normal_mode;    /* MDPP_NORMAL_* (Philox mode only)                */
  int32_t flags;          /* MDPP_LAUNCH_*                                   */
  uint64_t seed;          /* Philox key                                      */
  uint64_t step_index;    /* global index of the first step of this call     */
  int64_t env_id_offset;  /* global id of local env 0 (multi-GPU sharding)   */
  const uint64_t* step_index_dev; /* optional DEVICE counter added to
                                     step_index when the kernel runs: lets a
                                     captured CUDA graph advance the Philox
                                     step without re-recording (NULL = unused) */
} mdpp_step_opts;

/* K1/K2: T fused steps, one thread per env, tables staged in shared memory. */
#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_discrete_rollout(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                          const mdpp_discrete_io* io,
                          const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* Tabular Q-learning fused into the discrete rollout: T steps of epsilon-
 * greedy Q-learning, one Q-table per env, in one launch.  At global step
 * `step` env i (global Philox id g) in state s draws
 * w = philox(g, step, STREAM_ACTION) -- the random policy's word --, explores
 * iff (double)w.z < epsilon * 2^32 (then a = the random policy's action
 * umulhi(w.x, A)), else a = argmax_a' q[i][s][a'] (ties: lowest index), steps
 * like mdpp_discrete_rollout, and updates, with r the returned reward and nxt
 * the state before any auto-reset,
 *   target = terminated ? r : r + gamma * max_a' q[i][nxt][a']
 *   q[i][s][a] += alpha * (target - q[i][s][a])
 * in float64 with every operation rounded on its own (no FMA).  Truncation
 * bootstraps.  The env state and statistics end as mdpp_discrete_rollout
 * leaves them with the same actions.  `io->actions` must be NULL; the other
 * outputs of `io` and `actions_taken` may be NULL (skipped).  Philox noise,
 * no irrelevant features.                                                  */
typedef struct mdpp_qlearn_params {
  double alpha, gamma, epsilon;   /* each in [0, 1]                          */
  double* q;                      /* [N][q_states][q_actions], env-major     */
  int32_t q_states, q_actions;    /* >= every group's S / A                  */
  double* ep_return;              /* [N] return of the running episode       */
  double* ret_sum;                /* [N] sum of the returns of the episodes  */
  int32_t* ret_count;             /* [N] ... that ended in an auto-reset     */
  int32_t* actions_taken;         /* [T*N] or NULL                           */
} mdpp_qlearn_params;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_discrete_qlearn(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                         const mdpp_discrete_io* io,
                         const mdpp_qlearn_params* qp,
                         const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* K6: (masked) reset.  mask NULL = all envs.  The initial state comes from
 * `init_states` when given, else from the init cdf driven by `replay_reset_u`
 * (MDPP_NOISE_REPLAY) or Philox.  `obs` may be NULL.  With
 * irrelevant_features init_states, replay_reset_u and obs are [N*2] rows.    */
#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_discrete_reset(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                        const uint8_t* mask, const int32_t* init_states,
                        const double* replay_reset_u, int64_t* obs,
                        const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* ------------------------------------------------------------------------
 * Continuous environments, reward_function "move_to_a_point" (replaces
 * RLToyEnv.transition_function :1625-1725, reward_function :1848-1864 +
 * :1912-1945 + tail :1968-1990, step epilogue :2098-2109, reset :2284-2323).
 * One configuration per context.  `real` is float (dtype_s float32, the
 * reference default) or double (the fp64 verification build).
 * --------------------------------------------------------------------- */
#define MDPP_MAX_DIM 16
#define MDPP_MAX_ORDER 4
#define MDPP_MAX_TERM_BOXES 8

typedef struct mdpp_continuous_config {
  int32_t dim;                  /* state_space_dim = action_space_dim        */
  int32_t order;                /* transition_dynamics_order, 1..4           */
  int32_t n_relevant;           /* len(relevant_indices)                     */
  int32_t delay;
  int32_t reward_every_n_steps;
  int32_t dense;                /* make_denser (:1915) vs sparse (:1931)     */
  int32_t has_transition_noise; /* "transition_noise" key present (:407)     */
  int32_t has_reward_noise;     /* "reward_noise" key present (:398)         */
  int32_t image_mode;           /* image observations: every step takes the
                                   out-of-bounds branch (:1694, quirk q4)    */
  int32_t target_is_f64;        /* default target_point (float64 zeros :654) */
  int32_t n_term_boxes;
  int32_t is_f64;               /* 1: real = double                          */
  double inertia, time_unit;
  double state_space_max, action_space_max;   /* +inf = unbounded            */
  double target_radius, action_loss_weight;
  double transition_noise_std, reward_noise_std;
  double reward_scale, reward_shift, term_state_reward;
  int32_t relevant_indices[MDPP_MAX_DIM];
  double target_point[MDPP_MAX_DIM];          /* [n_relevant]                */
  double term_low[MDPP_MAX_TERM_BOXES * MDPP_MAX_DIM];   /* [box][relevant], */
  double term_high[MDPP_MAX_TERM_BOXES * MDPP_MAX_DIM];  /* cast to dtype_s  */
  /* per-dimension inertia (rl_toy_env.py:519-537, `action / self.inertia` at
   * :1654): 0 = the scalar `inertia` above; 1 = `inertia_vec`, an array of
   * dtype_s (the division stays in dtype_s); 2 = `inertia_vec` given as a list
   * / float64 array: numpy promotes the quotient, so the top derivative and
   * every Taylor term that reads it are float64                             */
  int32_t inertia_mode;
  /* reward_function: MDPP_REWARD_POINT = move_to_a_point (the target fields
   * above); MDPP_REWARD_LINE = move_along_a_line (rl_toy_env.py:1865-1910,
   * :2546-2576): minus the mean distance of the last `sequence_length`
   * relevant states from the line fitted through them (principal direction);
   * no target, no reached_terminal; state.hist holds the window             */
  int32_t reward_kind;
  double inertia_vec[MDPP_MAX_DIM];
  int32_t sequence_length;      /* MDPP_REWARD_LINE: 1..128                  */
  int32_t reserved_cfg;
} mdpp_continuous_config;
#define MDPP_REWARD_POINT 0
#define MDPP_REWARD_LINE 1

/* One configuration group of a heterogeneous continuous launch (a sweep over
 * time_unit / action_space_max / noise / delay / ... cells in ONE launch, like
 * mdpp_set_discrete_groups): groups tile the env range contiguously and must
 * agree on dim, relevant_indices, dtype, reward function and image mode --
 * what shapes the state arrays and I/O rows (`derivs` then has max(order) + 1
 * planes).  The delay ring has the
 * depth of the largest delay; statistics rows are [slot][group][MDPP_N_STATS]. */
typedef struct mdpp_continuous_group {
  mdpp_continuous_config cfg;
  int64_t env_begin, env_count;
  int64_t global_id_base;  /* global Philox id of the group's first env      */
} mdpp_continuous_group;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_set_continuous_config(mdpp_ctx* ctx, const mdpp_continuous_config* cfg);
int mdpp_set_continuous_groups(mdpp_ctx* ctx, const mdpp_continuous_group* groups,
                               int32_t n_groups);
#endif

/* Persistent state, struct-of-arrays over envs (DEVICE pointers, `real`).   */
typedef struct mdpp_continuous_state {
  int64_t n_envs;
  void* derivs;        /* real [(order+1)][dim][N]  state_derivatives        */
  void* emitted;       /* real [dim][N]  curr_state (noised / clipped)       */
  int32_t* t_episode;  /* [N]                                                */
  uint32_t* episode;   /* [N]                                                */
  uint8_t* reached;    /* [N] sticky reached_terminal (:1725)                */
  void* ring;          /* real [delay][N] reward FIFO, or NULL; DOUBLE when
                          real = float, target_is_f64 and dense (the reward
                          is a python float there, rl_toy_env.py:1915-1923) */
  double* stats;       /* [stats_slots][MDPP_N_STATS], summed over slots      */
  int32_t stats_slots; /* >= 1 (0 reads as 1), see mdpp_discrete_state        */
  int32_t reserved1;
  void* hist;          /* MDPP_REWARD_LINE: real [sequence_length][n_relevant][N],
                          the last emitted relevant states, slot = step % L  */
} mdpp_continuous_state;

/* T steps, time-major; actions / obs are env-major rows of `dim` reals
 * ([T][N][dim], the gym layout).                                            */
typedef struct mdpp_continuous_io {
  const void* actions;             /* real [T][N][dim]                       */
  void* obs;                       /* real [T][N][dim] emitted state (after
                                      the auto-reset when one happened)      */
  void* final_obs;                 /* real [T][N][dim] before any auto-reset */
  void* reward;                    /* real [T][N]                            */
  uint8_t* terminated;             /* [T][N]                                 */
  uint8_t* truncated;              /* [T][N]                                 */
  const double* replay_state_noise;  /* [T][N][dim] normal(0,s,dim) :413     */
  const double* replay_reward_noise; /* [T][N]                               */
  const void* replay_reset_state;    /* real [T][N][dim] accepted Box sample */
} mdpp_continuous_io;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_continuous_rollout(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                            const mdpp_continuous_io* io,
                            const mdpp_step_opts* opts, void* cuda_stream);
/* (masked) reset: `init_states` real [N][dim] when given, else Philox Box
 * sampling with rejection of the terminal boxes.  `obs` real [N][dim].      */
int mdpp_continuous_reset(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                          const uint8_t* mask, const void* init_states,
                          void* obs, const mdpp_step_opts* opts,
                          void* cuda_stream);
#endif

/* Augmented random search (Mania, Guy & Recht 2018, Algorithm 1, V1 / V1-t)
 * fused into the continuous rollout: every config group (or the single
 * configuration) is one ARS run whose envs are the perturbation population.
 * D = dim, P = D (D + 1); the policy of group g is a = W [obs; 1] with
 * theta[g] float64 [D][D+1] row-major.  Group sizes are even; local env 2p is
 * the + member and 2p + 1 the - member of pair p.
 *   delta_p: word c < ceil(P / 4) = philox(g+ = global id of the + member,
 *     iteration lo, iteration hi, STREAM_ARS_DELTA = 0x20000 + c); Box-Muller
 *     (fp64) of (w0, w1) -> entries 4c, 4c + 1, of (w2, w3) -> 4c + 2, 4c + 3
 *   w = theta + (s noise_std) delta_p, s = +1 / -1, rounded per entry
 *   a_d = sum_{k=0..D} w[d][k] phi_k, phi = (obs as fp64, 1), every product
 *     and sum rounded on its own, cast to real, clipped to
 *     [-(real)action_space_max, (real)action_space_max] when finite
 * where obs is the state the env last emitted (after any auto-reset).
 * mdpp_continuous_ars runs T fused steps and adds each returned reward
 * (as fp64) to fitness[i]; ep_return / ret_sum / ret_count are those of
 * mdpp_qlearn_params.  mdpp_continuous_ars_update, per group: keeps the
 * top_directions pairs by max(F+, F-) (ties: lower p), m / sigma_R = mean /
 * population std of the kept returns (sequential fp64 sums, ascending p, F+
 * before F-), and, when sigma_R is finite and > 0,
 *   theta[j] += (step_size / (b sigma_R)) * sum_{kept p} (F+ - F-) delta_p[j]
 * (sequential, ascending p); then zeroes fitness and increments `iteration`.
 * `io->actions` must be NULL; the outputs of `io`, `actions_taken`,
 * `delta_out` and `group_stats` may be NULL.  Philox noise, no image
 * observations.  The group layout is the context's (mdpp_set_continuous_
 * groups), or one group of all envs.                                        */
typedef struct mdpp_ars_params {
  double step_size;               /* alpha > 0                               */
  double noise_std;               /* nu >= 0 (0: every env acts with theta)  */
  double* theta;                  /* [G][D][D+1] float64 master weights      */
  double* fitness;                /* [N] reward sum since the last update    */
  double* ep_return;              /* [N] return of the running episode       */
  double* ret_sum;                /* [N] sum of the returns of the episodes  */
  int32_t* ret_count;             /* [N] ... that ended in an auto-reset     */
  void* actions_taken;            /* real [T][N][D] or NULL                  */
  int32_t top_directions;         /* b in [1, smallest group's pairs]        */
  int32_t reserved0;
  uint64_t iteration;             /* counter word of delta; update adds 1    */
  uint64_t seed;                  /* update / perturbations: the Philox seed */
  int64_t env_id_offset;          /* and env_id_offset of the learn launches
                                     (mdpp_continuous_ars takes opts')       */
  double* delta_out;             /* [N/2][D][D+1] float64 or NULL           */
  double* group_stats;            /* update: [G][3] (m, sigma_R, updated 0/1)
                                     or NULL                                 */
} mdpp_ars_params;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_continuous_ars(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                        const mdpp_continuous_io* io, const mdpp_ars_params* ap,
                        const mdpp_step_opts* opts, void* cuda_stream);
/* the update above; writes the iteration's delta to delta_out when given    */
int mdpp_continuous_ars_update(mdpp_ctx* ctx, int64_t n_envs, mdpp_ars_params* ap,
                               void* cuda_stream);
/* writes the current iteration's delta to delta_out only (no update)        */
int mdpp_continuous_ars_perturbations(mdpp_ctx* ctx, int64_t n_envs,
                                      const mdpp_ars_params* ap, void* cuda_stream);
#endif

/* ------------------------------------------------------------------------
 * Grid environments, reward_function "move_to_a_point" (replaces
 * RLToyEnv.transition_function :1727-1778, reward_function :1947-1965 + tail
 * :1968-1990, step epilogue :2098-2109, reset :2325-2345).  One configuration
 * per context.  Cells are int64 rows of n_dims coordinates ([x, y] or, with
 * irrelevant_features, [x, y, x_irr, y_irr]); an action is a row of n_dims
 * values in {-1, 0, 1} with at most one non-zero entry (GridActionSpace,
 * spaces/grid_action_space.py:25-39) -- anything else is a no-op, like the
 * reference's warning branch (:1765-1770).
 * Reference quirks kept: terminal cells never terminate (:958-987 test a float
 * array against an int64 Box), only the sticky `reached_terminal` (:1775) ends
 * an episode; reset() samples every coordinate from [0, shape] INCLUSIVE
 * (gymnasium's int Box), one past the grid; delay / sequence_length other than
 * 0 / 1 crash in the reference (:1950) and are rejected by the binding.
 * --------------------------------------------------------------------- */
#define MDPP_MAX_GRID_DIMS 4

typedef struct mdpp_grid_config {
  int32_t n_dims;               /* 2, or 4 with irrelevant_features           */
  int32_t dense;                /* make_denser: Manhattan progress vs +1 at target */
  int32_t reward_every_n_steps;
  int32_t has_transition_noise; /* truthy transition_noise (:1734)            */
  int32_t has_reward_noise;     /* "reward_noise" key present                 */
  int32_t reserved0;
  int32_t shape[MDPP_MAX_GRID_DIMS];  /* grid_shape (repeated when 4 dims)    */
  int32_t target[2];            /* target_point (relevant cell)               */
  double transition_noise;      /* p: the action is replaced by a different
                                   GridActionSpace sample w.p. p (:1736-1750) */
  double reward_noise_std, reward_scale, reward_shift, term_state_reward;
} mdpp_grid_config;

typedef struct mdpp_grid_state {   /* DEVICE pointers, struct-of-arrays      */
  int64_t n_envs;
  int32_t* pos;         /* [n_dims][N] current cell                           */
  int32_t* t_episode;   /* [N]                                                */
  uint32_t* episode;    /* [N]                                                */
  uint8_t* reached;     /* [N] sticky reached_terminal                        */
  double* stats;        /* [stats_slots][MDPP_N_STATS], summed over slots     */
  int32_t stats_slots;  /* >= 1 (0 reads as 1), see mdpp_discrete_state       */
  int32_t reserved1;
  int32_t* prev;        /* optional [2][N]: relevant cell BEFORE the last step
                           (the other entry of `augmented_state`, :2055-2056);
                           -1 right after a reset (the reference holds NaN)   */
} mdpp_grid_state;

typedef struct mdpp_grid_io {      /* T steps, time-major, rows of n_dims    */
  const int64_t* actions;          /* [T][N][n_dims]                          */
  int64_t* obs;                    /* [T][N][n_dims] cell after the step (after
                                      the auto-reset when one happened)       */
  int64_t* final_obs;              /* [T][N][n_dims] before any auto-reset    */
  double* reward;                  /* [T][N]                                  */
  uint8_t* terminated;             /* [T][N]                                  */
  uint8_t* truncated;              /* [T][N]                                  */
  const double* replay_noise_u;      /* [T][N] uniform() of :1736             */
  const int64_t* replay_noise_action;/* [T][N][n_dims] action applied when
                                        that uniform is < p                   */
  const double* replay_reward_noise; /* [T][N]                                */
  const int64_t* replay_reset_state; /* [T][N][n_dims] cell of an auto-reset  */
} mdpp_grid_io;

/* A heterogeneous grid launch (the `config_groups` of a sweep, like
 * mdpp_set_discrete_groups / mdpp_set_continuous_groups): group g owns the
 * envs [env_begin, env_begin + env_count) of the state arrays and steps them
 * under its own configuration; groups tile the env range in order and agree
 * on n_dims.  Statistics rows are [slot][group][MDPP_N_STATS].  Replaces any
 * earlier mdpp_set_grid_config (and vice versa).                            */
typedef struct mdpp_grid_group {
  mdpp_grid_config cfg;
  int64_t env_begin, env_count;
  int64_t global_id_base;  /* global Philox id of the group's first env      */
} mdpp_grid_group;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_set_grid_config(mdpp_ctx* ctx, const mdpp_grid_config* cfg);
int mdpp_set_grid_groups(mdpp_ctx* ctx, const mdpp_grid_group* groups,
                         int32_t n_groups);
int mdpp_grid_rollout(mdpp_ctx* ctx, const mdpp_grid_state* st,
                      const mdpp_grid_io* io, const mdpp_step_opts* opts,
                      void* cuda_stream);
/* (masked) reset: `init_states` int64 [N][n_dims] when given, else Philox
 * (every coordinate uniform on [0, shape]).  `obs` int64 [N][n_dims] or NULL. */
int mdpp_grid_reset(mdpp_ctx* ctx, const mdpp_grid_state* st,
                    const uint8_t* mask, const int64_t* init_states,
                    int64_t* obs, const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* Tabular Q-learning fused into the grid rollout (like mdpp_discrete_qlearn):
 * T steps of epsilon-greedy Q-learning, one Q-table per env, in one launch.
 * The state of env i is its cell pos[0..n_dims), every coordinate in
 * [0, shape_k] (the cell one past the grid included; the caller keeps the
 * cells in that range), indexed row-major:
 *   s = sum_k pos[k] * prod_{j>k} (shape_j + 1),  S = prod_k (shape_k + 1).
 * Action index a in [0, A), A = 2 n_dims + 1: 0 = the no-op, 1 + 2k = -1 on
 * dim k, 2 + 2k = +1 on dim k (the distinct GridActionSpace members).  At
 * global step `step` env i (global Philox id g) draws
 * w = philox(g, step >> 1, STREAM_GRID_ACTION = 45); words (x, y) belong to
 * the even step, (z, w) to the odd one.  It explores iff the first word
 * < ceil(epsilon * 2^32) (then a = umulhi(second word, A)), else
 * a = argmax_a' q[i][s][a'] (ties: lowest index), steps like
 * mdpp_grid_rollout with that action row (transition noise may substitute
 * the move; the update is still made for a), and updates, with r the
 * returned reward and nxt the cell before any auto-reset,
 *   target = terminated ? r : r + gamma * max_a' q[i][nxt][a']
 *   q[i][s][a] += alpha * (target - q[i][s][a])
 * in float64 with every operation rounded on its own (no FMA).  Truncation
 * bootstraps.  The env state and statistics end as mdpp_grid_rollout leaves
 * them with the same action rows.  q is [N][q_states][q_actions] with
 * q_states >= every group's S and q_actions >= A; `actions_taken` receives
 * the action index.  `io->actions` must be NULL; the other outputs of `io`
 * and `actions_taken` may be NULL (skipped).  Philox noise only.            */
#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_grid_qlearn(mdpp_ctx* ctx, const mdpp_grid_state* st,
                     const mdpp_grid_io* io, const mdpp_qlearn_params* qp,
                     const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* ------------------------------------------------------------------------
 * Evaluation of the learners' current policies: E episodes per env on an
 * evaluation env, with nothing learned and no exploration.
 *   mdpp_discrete_qeval / mdpp_grid_qeval: a = argmax_a' q[i][s][a'] (ties:
 *     lowest index), with s and the table layout of mdpp_discrete_qlearn /
 *     mdpp_grid_qlearn; q is only read.
 *   mdpp_continuous_ars_eval: a = theta_g [obs; 1] with the product and sum
 *     order, cast and clipping of mdpp_continuous_ars (noise_std = 0).
 * The env steps exactly as the rollout with those actions.  The caller
 * resets the env first, so every env starts a fresh episode; an episode
 * ends on terminated or truncated.  Of each env, the first `episodes`
 * episodes are counted: ret_sum[i] = the sum of their returns (fp64,
 * sequential), ret_count[i] = how many completed (= episodes when
 * n_steps >= episodes * horizon), len_sum[i] = the sum of their lengths; the
 * steps after them are stepped and discarded.  Needs Philox noise,
 * autoreset, horizon >= 1, episodes >= 1, n_steps >= episodes * horizon and
 * io->actions == NULL (the other outputs of io may be NULL: skipped).
 * mdpp_discrete_qeval: no irrelevant features.                              */
typedef struct mdpp_eval_params {
  const double* q;                /* qeval: [N][q_states][q_actions]         */
  int32_t q_states, q_actions;    /* >= every group's S / A                  */
  const double* theta;            /* ars_eval: [G][D][D+1] float64           */
  int32_t episodes;               /* E >= 1 counted episodes per env         */
  int32_t reserved0;
  double* ret_sum;                /* [N] return sum of the first E episodes  */
  int32_t* ret_count;             /* [N] episodes counted (<= E)             */
  int64_t* len_sum;               /* [N] length sum of the counted episodes  */
} mdpp_eval_params;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
int mdpp_discrete_qeval(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                        const mdpp_discrete_io* io, const mdpp_eval_params* ep,
                        const mdpp_step_opts* opts, void* cuda_stream);
int mdpp_grid_qeval(mdpp_ctx* ctx, const mdpp_grid_state* st, const mdpp_grid_io* io,
                    const mdpp_eval_params* ep, const mdpp_step_opts* opts,
                    void* cuda_stream);
int mdpp_continuous_ars_eval(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                             const mdpp_continuous_io* io, const mdpp_eval_params* ep,
                             const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* ------------------------------------------------------------------------
 * Image observations (replaces ImageMultiDiscrete.generate_image,
 * spaces/image_multi_discrete.py:129-270, and ImageContinuous.generate_image
 * / get_image_representation, spaces/image_continuous.py:116-277).
 * Stateless kernels: states in, uint8 images out, obs[x][y] = pil[y][x].
 * The tables are DEVICE arrays built on the host by
 * mdp_playground_b200/image_tables.py (Pillow is the raster authority).
 * --------------------------------------------------------------------- */
typedef struct mdpp_image_discrete_tables {
  int32_t width, height, n_states;
  int32_t r_min, n_radii;          /* polygon radius R in [r_min, r_min+n)   */
  int32_t n_xvar, n_yvar;          /* vertex-offset variants per (state, R)  */
  int32_t has_scale, has_shift, has_rotate, has_flip;
  int32_t sh_quant, ro_quant;
  int32_t n_sub_images;            /* 0 / 1: one image per env; 2: the images
                                      of the (relevant, irrelevant) sub-states,
                                      consecutive in `states` and `out`, i.e.
                                      stacked along x (:272-288)              */
  const uint64_t* mask_bits;       /* [n_masks][64] row bitmaps              */
  const int32_t* mask_index;       /* [S][n_radii][n_xvar][n_yvar]           */
  const uint8_t* xvar;             /* [S][n_radii][width]  by shift_w        */
  const uint8_t* yvar;             /* [S][n_radii][height] by shift_h        */
  const int32_t* rot_coeff;        /* [360][6] 16.16 inverse affine          */
  const double* r_thresholds;      /* [n_radii-1] uniform -> R               */
} mdpp_image_discrete_tables;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
/* Renders n_images polygon images.  Image m belongs to env (m % n_envs) at
 * step opts->step_index + m / n_envs (so a [T][N] block of states renders in
 * one launch); with n_sub_images = 2, m / 2 takes that role and sub-image
 * m % 2 draws from Philox stream image_stream + 16 * (m % 2).  params_in [n_images][5] = (R, shift_w, shift_h, rotation or
 * -1, flip 0/1 LR/2 TB) replays recorded transforms; NULL draws them from
 * Philox (stream `image_stream`: 3 for step observations, 6 for reset
 * observations).  params_out (optional) receives the parameters used.      */
int mdpp_render_discrete(mdpp_ctx* ctx, const mdpp_image_discrete_tables* tb,
                         const int64_t* states, const int32_t* params_in,
                         int32_t* params_out, uint8_t* out, int64_t n_images,
                         int64_t n_envs, int32_t image_stream,
                         const mdpp_step_opts* opts, void* cuda_stream);
#endif

/* Per-group renderer configurations of a heterogeneous launch (config groups
 * that differ in image_transforms, sh_quant, ro_quant, scale range or state
 * count): group g renders the envs [env_begin, env_begin + env_count) with
 * its own tables `tb` (DEVICE pointers, borrowed until the next set call or
 * mdpp_destroy).  Groups tile the env range in order (at most 65 535) and
 * agree on width, height and n_sub_images.  The Philox id of env e of group
 * g is opts->env_id_offset + global_id_base + (e - env_begin), like the step
 * kernels' (mdpp_discrete_group), so a group's image transforms do not
 * depend on how the job is sharded.                                          */
typedef struct mdpp_image_discrete_group {
  mdpp_image_discrete_tables tb;
  int64_t env_begin, env_count;
  int64_t global_id_base;
} mdpp_image_discrete_group;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
/* Replaces any earlier set; the descriptors are copied.                      */
int mdpp_set_image_discrete_groups(mdpp_ctx* ctx,
                                   const mdpp_image_discrete_group* groups,
                                   int32_t n_groups);
/* mdpp_render_discrete with the tables of each image's group: image m is
 * env (m / n_sub) % n_envs, the same indexing; n_envs must equal the
 * groups' total.                                                            */
int mdpp_render_discrete_groups(mdpp_ctx* ctx, const int64_t* states,
                                const int32_t* params_in, int32_t* params_out,
                                uint8_t* out, int64_t n_images, int64_t n_envs,
                                int32_t image_stream, const mdpp_step_opts* opts,
                                void* cuda_stream);
#endif

#define MDPP_MAX_STAMP_ROWS 32

typedef struct mdpp_image_continuous_config {
  int32_t width, height;
  int32_t dim;                     /* state_space_dim                        */
  int32_t n_sub_images;            /* 1, or 2 with irrelevant dimensions     */
  int32_t rel_index[2];            /* ImageContinuous.relevant_indices [0,1] */
  int32_t irr_index[2];
  int32_t is_f64;                  /* dtype of the states                    */
  int32_t n_rects;                 /* terminal regions (relevant image only) */
  int32_t has_target;
  int32_t stamp_rows;              /* 2*radius+1                             */
  int32_t stamp_radius;
  int32_t reserved0;
  double feat_low[2], feat_high[2];    /* feature-space bounds of rel_index   */
  int32_t rect[MDPP_MAX_TERM_BOXES][4];  /* x0, y0, x1, y1 inclusive pixels   */
  int32_t target_pixel[2];
  int32_t stamp[MDPP_MAX_STAMP_ROWS][2]; /* row: x offset, width (Pillow)     */
  /* grid envs (image_continuous.py:139-164): white grid lines, drawn first.
   * Bit x of vline[sub] = a full-height line in column x of sub-image `sub`
   * (0 relevant, 1 irrelevant), bit y of hline[sub] = a full-width line in
   * row y; width, height <= 256 when any bit is set.                         */
  uint64_t vline[2][4];
  uint64_t hline[2][4];
} mdpp_image_continuous_config;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
/* states: real [n_images][dim]; out: uint8 [n_images][n_sub*width][height][3] */
int mdpp_render_continuous(mdpp_ctx* ctx, const mdpp_image_continuous_config* cfg,
                           const void* states, uint8_t* out, int64_t n_images,
                           void* cuda_stream);
#endif

/* Per-group configurations of continuous and grid image observations (the
 * target, terminal rectangles, feature bounds and grid lines of each config
 * group): group g renders the envs [env_begin, env_begin + env_count).
 * Groups tile the env range in order (at most 65 535) and agree on width,
 * height, n_sub_images, dim and is_f64.                                      */
typedef struct mdpp_image_continuous_group {
  mdpp_image_continuous_config cfg;
  int64_t env_begin, env_count;
} mdpp_image_continuous_group;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
/* Replaces any earlier set; the configurations are copied.                   */
int mdpp_set_image_continuous_groups(mdpp_ctx* ctx,
                                     const mdpp_image_continuous_group* groups,
                                     int32_t n_groups);
/* mdpp_render_continuous with the configuration of each image's group:
 * image m is env m % n_envs; n_envs must equal the groups' total.           */
int mdpp_render_continuous_groups(mdpp_ctx* ctx, const void* states,
                                  uint8_t* out, int64_t n_images,
                                  int64_t n_envs, void* cuda_stream);
#endif

/* ------------------------------------------------------------------------
 * GymEnvWrapper's post-processing tail for EXTERNAL vector environments
 * (replaces envs/gym_env_wrapper.py:350-439 and get_transformed_image
 * :523-618; SURVEY.md 8f row N3).  The caller steps its own environments in
 * between: mdpp_tail_actions before, mdpp_tail_post / mdpp_tail_image_shift
 * after.  Noise comes from replay arrays (opts->noise_mode == REPLAY) or from
 * Philox streams keyed by (seed, env, step_index) like the step kernels.
 * --------------------------------------------------------------------- */
typedef struct mdpp_tail_config {
  int32_t discrete;             /* state_space_type == "discrete" (:353)     */
  int32_t n_actions;            /* env.action_space.n (discrete)             */
  int32_t obs_dim;              /* continuous: length of the observation     */
  int32_t obs_is_f64;           /* continuous: observations are double       */
  int32_t delay;                /* reward delay FIFO depth (:91-96)          */
  int32_t has_transition_noise; /* "transition_noise" given and truthy       */
  int32_t has_reward_noise;     /* "reward_noise" key present                */
  int32_t image_side;           /* image shift: side of the (square) images  */
  int32_t image_channels;       /* 3 (the reference's RGB path)              */
  int32_t image_padding;        /* :161-164, default 20                      */
  int32_t sh_quant;             /* image_sh_quant                            */
  int32_t has_shift;            /* "shift" in image_transforms               */
  double transition_noise;      /* discrete: probability; continuous: sigma  */
  double reward_noise_std;
  double reward_scale, reward_shift, term_state_reward;
} mdpp_tail_config;

typedef struct mdpp_tail_state {
  int64_t n_envs;
  double* ring;        /* [delay][N] delayed rewards, slot = step % delay     */
  int32_t* t_episode;  /* [N] steps since the FIFO was cleared                */
} mdpp_tail_state;

#ifndef __CUDACC_RTC__ /* NVRTC sees the types only */
/* :353-366: applied[i] = actions[i], or one of the other n_actions - 1 with
 * probability transition_noise.  Replay: `replay_u` [N] is the uniform numpy's
 * choice(n, p=probs) consumed (cumsum / searchsorted restated in fp64).       */
int mdpp_tail_actions(mdpp_ctx* ctx, const mdpp_tail_config* cfg,
                      const int32_t* actions, int32_t* applied,
                      const double* replay_u, int64_t n_envs,
                      const mdpp_step_opts* opts, void* cuda_stream);
/* :405-436: continuous observations get N(0, sigma) noise (out_obs = obs +
 * noise, NULL obs / out_obs skips it); rewards go through the delay FIFO, the
 * flush at `done`, noise, scale, shift.  At done the FIFO is cleared.  The
 * reference raises TypeError on every terminal step (:414 multiplies a list by
 * a float); the flush implements the line with the buffer read as an array.  */
int mdpp_tail_post(mdpp_ctx* ctx, const mdpp_tail_config* cfg,
                   const mdpp_tail_state* st, const void* obs, void* out_obs,
                   const double* reward, const uint8_t* done, double* out_reward,
                   const double* replay_reward_noise, const double* replay_obs_noise,
                   const mdpp_step_opts* opts, void* cuda_stream);
/* :523-618: img uint8 [N][side][side][3] -> out uint8 [N][tot][tot][3], tot =
 * side + 2 padding, out[x][y] = canvas[y][x]; the shift is drawn
 * (integers(-padding + 1, padding) per axis, truncated to sh_quant) or replayed
 * from `replay_shift` int32 [N][2] (the two raw integers); `shift_out` [N][2]
 * (optional) receives the raw draws.                                         */
int mdpp_tail_image_shift(mdpp_ctx* ctx, const mdpp_tail_config* cfg,
                          const uint8_t* img, uint8_t* out,
                          const int32_t* replay_shift, int32_t* shift_out,
                          int64_t n_envs, const mdpp_step_opts* opts,
                          void* cuda_stream);
#endif

#ifdef __cplusplus
}
#endif
#endif /* MDPP_B200_H */
