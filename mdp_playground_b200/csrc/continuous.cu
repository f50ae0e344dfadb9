// C entry points of the continuous step path (include/mdpp_b200.h).  The
// kernels are in continuous_kernels.cuh; the product path is the NVRTC
// specialisation (jit.cu), the ahead-of-time instantiations below are the
// fallback for hosts without NVRTC.
#include <cmath>
#include <cstring>
#include <vector>

#include "continuous_kernels.cuh"
#include "internal.h"

using namespace mdpp;

static int check_config(mdpp_ctx* ctx, const mdpp_continuous_config* cfg) {
  if (!cfg) return fail(ctx, MDPP_EINVAL, "cfg is NULL");
  if (cfg->dim < 1 || cfg->dim > MDPP_MAX_DIM)
    return fail(ctx, MDPP_EINVAL, "state_space_dim must be in 1..16");
  if (cfg->order < 1 || cfg->order > MDPP_MAX_ORDER)
    return fail(ctx, MDPP_EINVAL, "transition_dynamics_order must be in 1..4");
  if (cfg->n_relevant < 1 || cfg->n_relevant > cfg->dim)
    return fail(ctx, MDPP_EINVAL, "bad relevant_indices");
  for (int k = 0; k < cfg->n_relevant; ++k)
    if (cfg->relevant_indices[k] < 0 || cfg->relevant_indices[k] >= cfg->dim)
      return fail(ctx, MDPP_EINVAL, "relevant index out of range");
  if (cfg->delay < 0 || cfg->reward_every_n_steps < 1)
    return fail(ctx, MDPP_EINVAL, "bad delay / reward_every_n_steps");
  if (cfg->n_term_boxes < 0 || cfg->n_term_boxes > MDPP_MAX_TERM_BOXES)
    return fail(ctx, MDPP_EINVAL, "at most 8 terminal boxes");
  if (cfg->image_mode && !std::isfinite(cfg->state_space_max))
    return fail(ctx, MDPP_EINVAL, "image observations need a bounded space");
  if (cfg->inertia_mode < 0 || cfg->inertia_mode > 2)
    return fail(ctx, MDPP_EINVAL, "bad inertia_mode");
  if (cfg->reward_kind != MDPP_REWARD_POINT && cfg->reward_kind != MDPP_REWARD_LINE)
    return fail(ctx, MDPP_EINVAL, "unknown reward_kind");
  if (cfg->reward_kind == MDPP_REWARD_LINE &&
      (cfg->sequence_length < 1 || cfg->sequence_length > kLineMaxSeq))
    return fail(ctx, MDPP_EINVAL, "move_along_a_line: sequence_length must be in 1..128");
  return MDPP_OK;
}

extern "C" int mdpp_set_continuous_config(mdpp_ctx* ctx,
                                          const mdpp_continuous_config* cfg) {
  if (!ctx) return MDPP_EINVAL;
  int rc = check_config(ctx, cfg);
  if (rc) return rc;
  release_groups(ctx->c_set);
  ctx->c_group_ranges.clear();
  ctx->c_cfg = *cfg;
  ctx->have_continuous = true;
  return MDPP_OK;
}

extern "C" int mdpp_set_continuous_groups(mdpp_ctx* ctx,
                                          const mdpp_continuous_group* groups,
                                          int32_t n_groups) {
  if (!ctx) return MDPP_EINVAL;
  int rc = validate_groups(ctx, __func__, groups, n_groups, /*env_map=*/false);
  if (rc) return rc;
  std::vector<ContinuousGroupDev> dev(n_groups);
  const mdpp_continuous_config& c0 = groups[0].cfg;
  // the launch-wide view: flags any group has (replay arrays, ring depth)
  mdpp_continuous_config view = c0;
  for (int g = 0; g < n_groups; ++g) {
    const mdpp_continuous_config& c = groups[g].cfg;
    rc = check_config(ctx, &c);
    if (rc) return rc;
    // the groups share everything that shapes the state arrays and the I/O rows
    // (the order may differ: derivative planes are addressed independently of it)
    if (c.dim != c0.dim || c.n_relevant != c0.n_relevant ||
        c.is_f64 != c0.is_f64 || c.image_mode != c0.image_mode ||
        c.reward_kind != c0.reward_kind ||
        (c.reward_kind == MDPP_REWARD_LINE && c.sequence_length != c0.sequence_length) ||
        std::memcmp(c.relevant_indices, c0.relevant_indices, sizeof c.relevant_indices) != 0)
      return fail(ctx, MDPP_EINVAL,
                  "continuous groups must agree on dim, relevant_indices, dtype, "
                  "reward function (and its sequence_length) and image mode");
    std::memset(&dev[g], 0, sizeof dev[g]);
    dev[g].cfg = c;
    for (int j = 0; j < MDPP_MAX_ORDER; ++j) dev[g].tu_pow[j] = std::pow(c.time_unit, j + 1);
    dev[g].env_begin = groups[g].env_begin;
    dev[g].env_count = groups[g].env_count;
    dev[g].gid_base = groups[g].global_id_base;
    view.has_transition_noise |= c.has_transition_noise;
    view.has_reward_noise |= c.has_reward_noise;
    if (c.delay > view.delay) view.delay = c.delay;
  }
  rc = install_groups(ctx, ctx->c_set, dev.data(), n_groups, kCBlock);
  if (rc) return rc;
  ctx->c_group_ranges.clear();
  for (int g = 0; g < n_groups; ++g)
    ctx->c_group_ranges.insert(ctx->c_group_ranges.end(),
                               {groups[g].env_begin, groups[g].env_count,
                                groups[g].global_id_base});
  ctx->c_cfg = view;
  ctx->have_continuous = true;
  return MDPP_OK;
}

int mdpp::fill_continuous_params(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                                   const mdpp_step_opts* opts, ContinuousParams* p) {
  if (!ctx) return MDPP_EINVAL;
  if (!ctx->have_continuous)
    return fail(ctx, MDPP_EINVAL, "mdpp_set_continuous_config was not called");
  if (!st || !st->derivs || !st->emitted || !st->t_episode || !st->episode ||
      !st->reached || st->n_envs < 1)
    return fail(ctx, MDPP_EINVAL, "continuous state has NULL arrays");
  if (ctx->c_cfg.delay > 0 && !st->ring)
    return fail(ctx, MDPP_EINVAL, "delay ring missing");
  if (ctx->c_cfg.reward_kind == MDPP_REWARD_LINE && !st->hist)
    return fail(ctx, MDPP_EINVAL, "move_along_a_line: state.hist is NULL");
  if (!opts) return fail(ctx, MDPP_EINVAL, "opts is NULL");
  std::memset(p, 0, sizeof(*p));
  p->cfg = ctx->c_cfg;
  for (int j = 0; j < MDPP_MAX_ORDER; ++j)
    p->tu_pow[j] = std::pow(ctx->c_cfg.time_unit, j + 1);
  p->st = *st;
  p->T = opts->n_steps;
  p->autoreset = opts->autoreset;
  p->horizon = opts->horizon;
  p->noise_mode = opts->noise_mode;
  p->normal_mode = opts->normal_mode;
  p->k0 = (uint32_t)opts->seed;
  p->k1 = (uint32_t)(opts->seed >> 32);
  philox_round_keys(p->k0, p->k1, p->rk);
  p->zig = ctx->d_zig;
  p->step_index = opts->step_index;
  p->step_index_dev = opts->step_index_dev;
  p->env_id_offset = opts->env_id_offset;
  if (ctx->c_set.n_groups > 0) {
    int rc = bind_groups(ctx, ctx->c_set, "continuous launch", st->n_envs);
    if (rc) return rc;
    p->groups = static_cast<const ContinuousGroupDev*>(ctx->c_set.groups);
    p->cta_map = ctx->c_set.cta_map;
    p->n_groups = ctx->c_set.n_groups;
  }
  return MDPP_OK;
}

template <typename R>
static int launch_groups(mdpp_ctx* ctx, const ContinuousParams& p, cudaStream_t s) {
  const unsigned grid = (unsigned)ctx->c_set.n_ctas;
  switch (p.noise_mode) {
    case MDPP_NOISE_OFF:
      continuous_rollout_kernel<R, MDPP_NOISE_OFF, true><<<grid, kCBlock, 0, s>>>(p);
      break;
    case MDPP_NOISE_REPLAY:
      continuous_rollout_kernel<R, MDPP_NOISE_REPLAY, true><<<grid, kCBlock, 0, s>>>(p);
      break;
    default:
      continuous_rollout_kernel<R, MDPP_NOISE_PHILOX, true><<<grid, kCBlock, 0, s>>>(p);
  }
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

template <typename R>
static int launch_aot(mdpp_ctx* ctx, const ContinuousParams& p, cudaStream_t s) {
  const unsigned grid = (unsigned)((p.st.n_envs + kCBlock - 1) / kCBlock);
  switch (p.noise_mode) {
    case MDPP_NOISE_OFF:
      continuous_rollout_kernel<R, MDPP_NOISE_OFF><<<grid, kCBlock, 0, s>>>(p);
      break;
    case MDPP_NOISE_REPLAY:
      continuous_rollout_kernel<R, MDPP_NOISE_REPLAY><<<grid, kCBlock, 0, s>>>(p);
      break;
    default:
      continuous_rollout_kernel<R, MDPP_NOISE_PHILOX><<<grid, kCBlock, 0, s>>>(p);
  }
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

extern "C" int mdpp_continuous_rollout(mdpp_ctx* ctx,
                                       const mdpp_continuous_state* st,
                                       const mdpp_continuous_io* io,
                                       const mdpp_step_opts* opts,
                                       void* cuda_stream) {
  ContinuousParams p;
  int rc = fill_continuous_params(ctx, st, opts, &p);
  if (rc) return rc;
  if (!io || !io->actions || opts->n_steps < 1)
    return fail(ctx, MDPP_EINVAL, "continuous rollout needs actions and T >= 1");
  if (opts->noise_mode < MDPP_NOISE_OFF || opts->noise_mode > MDPP_NOISE_PHILOX)
    return fail(ctx, MDPP_EINVAL, "unknown noise_mode");
  if (opts->noise_mode == MDPP_NOISE_REPLAY) {
    if ((ctx->c_cfg.has_transition_noise && !io->replay_state_noise) ||
        (ctx->c_cfg.has_reward_noise && !io->replay_reward_noise) ||
        (opts->autoreset && !io->replay_reset_state))
      return fail(ctx, MDPP_EINVAL, "replay mode: missing replay array");
  }
  // rows move as 8- / 16-byte vectors in the specialised kernels
  if (((uintptr_t)io->actions | (uintptr_t)io->obs | (uintptr_t)io->final_obs) & 15)
    return fail(ctx, MDPP_EINVAL, "actions / obs / final_obs must be 16-byte aligned");
  p.io = *io;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (p.groups)  // heterogeneous launch: every CTA under its own group's scalars
    return ctx->c_cfg.is_f64 ? launch_groups<double>(ctx, p, s)
                             : launch_groups<float>(ctx, p, s);
  rc = jit_try_continuous(ctx, p, s);
  if (rc != 0) return rc < 0 ? rc : MDPP_OK;
  return ctx->c_cfg.is_f64 ? launch_aot<double>(ctx, p, s)
                           : launch_aot<float>(ctx, p, s);
}

extern "C" int mdpp_continuous_reset(mdpp_ctx* ctx,
                                     const mdpp_continuous_state* st,
                                     const uint8_t* mask,
                                     const void* init_states, void* obs,
                                     const mdpp_step_opts* opts,
                                     void* cuda_stream) {
  ContinuousParams p;
  int rc = fill_continuous_params(ctx, st, opts, &p);
  if (rc) return rc;
  if (!init_states && opts->noise_mode == MDPP_NOISE_REPLAY)
    return fail(ctx, MDPP_EINVAL, "replay reset needs init_states");
  p.mask = mask;
  p.init_states = init_states;
  p.reset_obs = obs;
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned grid = p.groups ? (unsigned)ctx->c_set.n_ctas
                                 : (unsigned)((p.st.n_envs + kCBlock - 1) / kCBlock);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (p.groups && ctx->c_cfg.is_f64)
    continuous_reset_kernel<double, true><<<grid, kCBlock, 0, s>>>(p);
  else if (p.groups)
    continuous_reset_kernel<float, true><<<grid, kCBlock, 0, s>>>(p);
  else if (ctx->c_cfg.is_f64)
    continuous_reset_kernel<double><<<grid, kCBlock, 0, s>>>(p);
  else
    continuous_reset_kernel<float><<<grid, kCBlock, 0, s>>>(p);
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}
