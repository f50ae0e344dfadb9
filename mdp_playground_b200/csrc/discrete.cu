// C entry points of the discrete step path (include/mdpp_b200.h) and the reset
// kernel (K6).  The rollout kernels live in discrete_kernels.cuh and are
// instantiated per noise mode in discrete_{off,replay,philox_f64,philox_fast}.cu
// so they compile in parallel.
#include "discrete_kernels.cuh"
#include "internal.h"

namespace mdpp {

int launch_rollout_off(mdpp_ctx*, RolloutParams&, cudaStream_t);
int launch_rollout_replay(mdpp_ctx*, RolloutParams&, cudaStream_t);
int launch_rollout_philox_f64(mdpp_ctx*, RolloutParams&, cudaStream_t);
int launch_rollout_philox_fast(mdpp_ctx*, RolloutParams&, cudaStream_t);
int launch_rollout_philox_zig(mdpp_ctx*, RolloutParams&, cudaStream_t);


__global__ void __launch_bounds__(kBlock)
discrete_reset_kernel(const __grid_constant__ ResetParams p) {
  const CtaMapEntry me = p.cta_map[blockIdx.x];
  const DiscreteGroupDev& g = p.groups[me.group];
  const int64_t local = (int64_t)me.chunk * kBlock + threadIdx.x;
  if (local >= g.env_count) return;
  const int64_t env = g.env_begin + local;
  const int64_t N = p.st.n_envs;
  const bool irr = p.irr != 0;  // rows (relevant, irrelevant) in init / u / obs
  if (p.mask && !p.mask[env]) {
    if (p.obs && irr) {
      p.obs[2 * env] = p.st.cur_state[env];
      p.obs[2 * env + 1] = p.st.cur_state_irr[env];
    } else if (p.obs) {
      p.obs[env] = p.st.cur_state[env];
    }
    return;
  }
  const uint32_t gid = (uint32_t)(p.env_id_offset + g.gid_base + local);
  const uint32_t ep = p.st.episode[env];
  int32_t s0, s0_irr = 0;
  if (p.init_states) {
    s0 = p.init_states[irr ? 2 * env : env];
    if (irr) s0_irr = p.init_states[2 * env + 1];
  } else {
    double u, u_irr = 0.0;
    if (p.noise_mode == MDPP_NOISE_REPLAY) {
      u = p.replay_reset_u[irr ? 2 * env : env];
      if (irr) u_irr = p.replay_reset_u[2 * env + 1];
    } else {
      U4 w = philox4x32_10(gid, ep, 0u, STREAM_RESET, p.k0, p.k1);
      u = uniform53(w.x, w.y);
      u_irr = uniform53(w.z, w.w);  // second E draw of reset() (:2260-2264)
    }
    const double* cdf =
        reinterpret_cast<const double*>(p.blob + g.blob_offset + g.off_init_cdf);
    s0 = cdf_search<-1>(cdf, g.cdf_log2, g.S, u);
    if (irr) {
      const double* cdf1 = reinterpret_cast<const double*>(
          p.blob + g.blob_offset + g.off_init_cdf_irr);
      s0_irr = cdf_search<-1>(cdf1, g.irr_cdf_log2, g.S1, u_irr);
    }
  }
  if (p.st.stats && p.st.t_episode[env] > 0) {
    const int slot = (int)(blockIdx.x % (unsigned)max(p.st.stats_slots, 1));
    atomicAdd(p.st.stats + ((int64_t)slot * p.n_groups + me.group) * MDPP_N_STATS +
                  MDPP_STAT_EPISODES, 1.0);
  }
  p.st.cur_state[env] = s0;
  if (irr) p.st.cur_state_irr[env] = min(max(s0_irr, 0), g.S1 - 1);
  p.st.seq_key[env] = (uint64_t)s0;
  p.st.t_episode[env] = 0;
  p.st.episode[env] = ep + 1;
  if (p.st.history)
    p.st.history[(int64_t)(p.step_index % (uint64_t)p.st.history_depth) * N + env] = s0;
  if (p.obs && irr) {
    p.obs[2 * env] = s0;
    p.obs[2 * env + 1] = p.st.cur_state_irr[env];
  } else if (p.obs) {
    p.obs[env] = s0;
  }
}

}  // namespace mdpp

using namespace mdpp;

static int check_state(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                       const char* entry) {
  if (!ctx) return MDPP_EINVAL;
  if (ctx->d_groups_host.empty())
    return fail(ctx, MDPP_EINVAL, "mdpp_set_discrete_groups was not called");
  if (!st || !st->cur_state || !st->seq_key || !st->t_episode || !st->episode)
    return fail(ctx, MDPP_EINVAL, "discrete state has NULL arrays");
  int rc = bind_groups(ctx, ctx->d_set, entry, st->n_envs);
  if (rc) return rc;
  if (ctx->max_delay > 0 && (!st->ring || st->ring_depth < ctx->max_delay))
    return fail(ctx, MDPP_EINVAL, "delay ring missing or too shallow");
  if (st->history && st->history_depth < 1)
    return fail(ctx, MDPP_EINVAL, "history_depth must be >= 1");
  if (ctx->d_irr && !st->cur_state_irr)
    return fail(ctx, MDPP_EINVAL, "irrelevant sub-MDP: cur_state_irr is NULL");
  return MDPP_OK;
}

// Checks and kernel parameters shared by mdpp_discrete_rollout and
// mdpp_discrete_qlearn (qlearn.cu).
int mdpp::prepare_rollout(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                          const mdpp_discrete_io* io, const mdpp_step_opts* opts,
                          RolloutParams& p) {
  int rc = check_state(ctx, st, "discrete rollout");
  if (rc) return rc;
  if (!io || !opts || opts->n_steps < 1)
    return fail(ctx, MDPP_EINVAL, "bad io/opts");
  if (io->obs_dtype < MDPP_OBS_I64 || io->obs_dtype > MDPP_OBS_U8)
    return fail(ctx, MDPP_EINVAL, "unknown obs_dtype");
  if (io->obs_dtype == MDPP_OBS_U8)
    for (auto& g : ctx->d_groups_host)
      if (g.S > 256 || g.S1 > 256)
        return fail(ctx, MDPP_EINVAL, "obs_dtype u8 needs <= 256 states");
  if (opts->noise_mode == MDPP_NOISE_REPLAY) {
    bool need_p = false, need_r = false;
    for (auto& g : ctx->d_groups_host) {
      need_p |= g.has_pnoise != 0;
      need_r |= g.has_rnoise != 0;
    }
    if ((need_p && !io->replay_transition_u) ||
        (need_r && !io->replay_reward_noise) ||
        (opts->autoreset && !io->replay_reset_u))
      return fail(ctx, MDPP_EINVAL, "replay mode: missing replay array");
  }
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  p.group0 = ctx->d_groups_host[0];
  p.groups = static_cast<const DiscreteGroupDev*>(ctx->d_set.groups);
  p.blob = ctx->d_blob;
  p.cta_map = ctx->d_set.cta_map;
  p.st = *st;
  p.io = *io;
  p.T = opts->n_steps;
  p.autoreset = opts->autoreset;
  p.horizon = opts->horizon;
  p.k0 = (uint32_t)opts->seed;
  p.k1 = (uint32_t)(opts->seed >> 32);
  philox_round_keys(p.k0, p.k1, p.rk);
  p.step_index = opts->step_index;
  p.step_index_dev = opts->step_index_dev;
  p.env_id_offset = opts->env_id_offset;
  p.irr = ctx->d_irr;
  p.n_groups = ctx->d_set.n_groups;
  p.zig = ctx->d_zig;
  p.tab_smem_bytes = 0;
  return MDPP_OK;
}

extern "C" int mdpp_discrete_rollout(mdpp_ctx* ctx,
                                     const mdpp_discrete_state* st,
                                     const mdpp_discrete_io* io,
                                     const mdpp_step_opts* opts,
                                     void* cuda_stream) {
  RolloutParams p;
  int rc = prepare_rollout(ctx, st, io, opts, p);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (opts->noise_mode < MDPP_NOISE_OFF || opts->noise_mode > MDPP_NOISE_PHILOX)
    return fail(ctx, MDPP_EINVAL, "unknown noise_mode");
  // single-group launches: a kernel compiled for exactly this configuration
  rc = jit_try_rollout(ctx, p, opts->noise_mode, opts->normal_mode, s);
  if (rc != 0) return rc < 0 ? rc : MDPP_OK;
  switch (opts->noise_mode) {
    case MDPP_NOISE_OFF: return launch_rollout_off(ctx, p, s);
    case MDPP_NOISE_REPLAY: return launch_rollout_replay(ctx, p, s);
    case MDPP_NOISE_PHILOX:
      return opts->normal_mode == MDPP_NORMAL_FAST
                 ? launch_rollout_philox_fast(ctx, p, s)
                 : opts->normal_mode == MDPP_NORMAL_ZIGGURAT
                       ? launch_rollout_philox_zig(ctx, p, s)
                       : launch_rollout_philox_f64(ctx, p, s);
  }
  return fail(ctx, MDPP_EINVAL, "unknown noise_mode");
}

extern "C" int mdpp_discrete_reset(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                                   const uint8_t* mask,
                                   const int32_t* init_states,
                                   const double* replay_reset_u, int64_t* obs,
                                   const mdpp_step_opts* opts,
                                   void* cuda_stream) {
  int rc = check_state(ctx, st, "discrete reset");
  if (rc) return rc;
  if (!opts) return fail(ctx, MDPP_EINVAL, "opts is NULL");
  if (!init_states && opts->noise_mode == MDPP_NOISE_REPLAY && !replay_reset_u)
    return fail(ctx, MDPP_EINVAL, "replay reset needs replay_reset_u");
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  ResetParams p;
  p.groups = static_cast<const DiscreteGroupDev*>(ctx->d_set.groups);
  p.blob = ctx->d_blob;
  p.cta_map = ctx->d_set.cta_map;
  p.st = *st;
  p.mask = mask;
  p.init_states = init_states;
  p.replay_reset_u = replay_reset_u;
  p.obs = obs;
  p.noise_mode = opts->noise_mode;
  p.k0 = (uint32_t)opts->seed;
  p.k1 = (uint32_t)(opts->seed >> 32);
  p.step_index = opts->step_index;
  p.env_id_offset = opts->env_id_offset;
  p.irr = ctx->d_irr;
  p.n_groups = ctx->d_set.n_groups;
  discrete_reset_kernel<<<(unsigned)ctx->d_set.n_ctas, kBlock, 0,
                          (cudaStream_t)cuda_stream>>>(p);
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}
