// Internal declarations shared by the translation units of libmdpp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>


#include "device_types.h"

// A config-group set: descriptors of contiguous env ranges covering [0, N) in
// order, one group per configuration, and the map its kernels find their group by.
struct GroupSet {
  void* groups = nullptr;                // device copy of the descriptors
  mdpp::CtaMapEntry* cta_map = nullptr;  // [n_ctas] CTA -> (group, chunk): step kinds
  uint16_t* env_group = nullptr;         // [n_envs] env -> group: renderers
  int32_t n_groups = 0;
  int64_t n_ctas = 0, n_envs = 0;
};

struct mdpp_ctx {
  int device = 0;
  int sm_count = 0;
  int max_smem_optin = 0;
  std::string error;
  // discrete tables
  GroupSet d_set;  // DiscreteGroupDev (mdpp_set_discrete_groups)
  std::vector<mdpp::DiscreteGroupDev> d_groups_host;
  uint8_t* d_blob = nullptr;
  size_t d_blob_bytes = 0;
  int max_group_blob = 0;
  int max_delay = 0;
  int d_irr = 0;  // groups carry an irrelevant sub-MDP
  uint8_t* d_zig = nullptr;  // ziggurat tables (ziggurat.cuh layout), per context
  // continuous configuration (one per context): a single one, or the
  // launch-wide view of a group set (ContinuousGroupDev)
  bool have_continuous = false;
  mdpp_continuous_config c_cfg;
  GroupSet c_set;
  // (env_begin, env_count, global_id_base) of each group of c_set: the host
  // side of the ARS update (ars.cu); empty for a single configuration
  std::vector<int64_t> c_group_ranges;
  bool have_grid = false;
  mdpp_grid_config g_cfg;
  GroupSet g_set;  // GridGroupDev
  int64_t g_states = 0;  // most cells prod_k (shape_k + 1) of a grid group (capped at 2^31)
  // per-group image renderers: the ABI descriptors as given, with an
  // env -> group map (one load per image); the first-group views hold what
  // the groups share
  GroupSet img_d_set;  // mdpp_image_discrete_group
  mdpp_image_discrete_tables img_d_first;  // group 0's (shared sizes), any-rotate
  GroupSet img_c_set;  // mdpp_image_continuous_group
  mdpp_image_continuous_config img_c_first;
  // runtime-specialised kernels (jit.cu), keyed by their define string
  std::map<std::string, void*> jit_functions;   // CUfunction
  std::vector<void*> jit_modules;               // CUmodule
  // last launch's (signature -> function): step()-granularity callers repeat
  // the same launch shape, and building the -D list (the cache key of
  // jit_functions) costs more than the T = 1 kernel itself
  long long jit_sig_discrete[10] = {-1, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  void* jit_fn_discrete = nullptr;
  unsigned char jit_sig_continuous[sizeof(mdpp_continuous_config) + 64] = {0};
  void* jit_fn_continuous = nullptr;
  long long d_groups_version = 0;  // bumped by mdpp_set_discrete_groups
  int jit_enabled = 1;      // MDPP_JIT=0 in the environment disables it
  int jit_last_used = 0;    // 1 if the last rollout ran a JIT kernel
  std::string jit_log;      // why JIT was not used (informational)
};

namespace mdpp {
// jit.cu: try to run the rollout through a kernel compiled for exactly this
// configuration.  Returns 1 if it launched, 0 if JIT is unavailable (caller
// falls back to the ahead-of-time kernels), < 0 on a launch error.
int jit_try_rollout(mdpp_ctx* ctx, RolloutParams& p, int noise_mode,
                    int normal_mode, cudaStream_t stream);
struct ContinuousParams;
int jit_try_continuous(mdpp_ctx* ctx, ContinuousParams& p, cudaStream_t stream);
void jit_release(mdpp_ctx* ctx);
int smem_min_steps();  // MDPP_SMEM_MIN_T (default 1): shorter launches skip the smem staging
int fail(mdpp_ctx* ctx, int code, const std::string& msg);
// discrete.cu: validate a discrete launch and fill its parameters
int prepare_rollout(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                    const mdpp_discrete_io* io, const mdpp_step_opts* opts,
                    RolloutParams& p);
int cuda_fail(mdpp_ctx* ctx, cudaError_t e, const char* what);
// qlearn.cu: the checks of mdpp_qlearn_params that every learner shares (NULL
// arrays, a table smaller than n_states x n_actions, alpha / gamma / epsilon
// outside [0, 1]), then its device view
// continuous.cu: the checks and launch parameters every continuous step
// launch shares (state arrays, configuration, options, group binding)
struct ContinuousParams;
int fill_continuous_params(mdpp_ctx* ctx, const mdpp_continuous_state* st,
                           const mdpp_step_opts* opts, ContinuousParams* p);
int check_qlearn_params(mdpp_ctx* ctx, const mdpp_qlearn_params* qp, int64_t n_states,
                        int64_t n_actions, QlearnDev* d);
// The checks of the evaluation entry points (mdpp_discrete_qeval,
// mdpp_grid_qeval, mdpp_continuous_ars_eval): the launch options, the episode
// count and the output arrays, and the Q-table against the groups' S / A
// (n_states >= 0) or theta (n_states < 0); then the outputs' device view
int check_eval_params(mdpp_ctx* ctx, const char* who, bool has_actions,
                      const mdpp_step_opts* opts, const mdpp_eval_params* ep,
                      int64_t n_states, int64_t n_actions, EvalDev* d);

// Checks that groups[0..n) cover [0, N) contiguously, in order, with N >= 1, and
// that a set with an env -> group map has at most 65 535 groups (uint16).
// `setter` is the entry point named in the error.
template <typename G>
int validate_groups(mdpp_ctx* ctx, const char* setter, const G* groups, int32_t n,
                    bool env_map) {
  if (!groups || n < 1)
    return fail(ctx, MDPP_EINVAL, std::string(setter) + ": need at least one group");
  if (env_map && n > 65535)
    return fail(ctx, MDPP_EINVAL, std::string(setter) + ": at most 65535 groups");
  int64_t next = 0;
  for (int32_t g = 0; g < n; ++g) {
    if (groups[g].env_begin != next || groups[g].env_count < 0)
      return fail(ctx, MDPP_EINVAL, std::string(setter) + ": group " + std::to_string(g) +
                  " breaks the tiling (groups must tile the env range [0, N) "
                  "contiguously, in order)");
    next += groups[g].env_count;
  }
  if (next < 1) return fail(ctx, MDPP_EINVAL, std::string(setter) + ": no environments");
  return MDPP_OK;
}

inline void release_groups(GroupSet& set) {
  if (set.groups) cudaFree(set.groups);
  if (set.cta_map) cudaFree(set.cta_map);
  if (set.env_group) cudaFree(set.env_group);
  set = GroupSet();
}

// Replaces `set` with device copies of the n descriptors `groups` (tiling
// validated) and of its map: CTA -> (group, chunk) for CTAs of `block` envs
// when block > 0, else env -> group.  On failure `set` is left as it was.
template <typename D>
int install_groups(mdpp_ctx* ctx, GroupSet& set, const D* groups, int32_t n, int block) {
  std::vector<CtaMapEntry> cta_map;
  std::vector<uint16_t> env_group;
  GroupSet s;
  s.n_groups = n;
  for (int32_t g = 0; g < n; ++g) {
    if (block > 0)
      for (int32_t c = 0; (int64_t)c * block < groups[g].env_count; ++c)
        cta_map.push_back(CtaMapEntry{g, c});
    else
      env_group.insert(env_group.end(), (size_t)groups[g].env_count, (uint16_t)g);
    s.n_envs += groups[g].env_count;
  }
  s.n_ctas = (int64_t)cta_map.size();
  cudaError_t e = cudaSetDevice(ctx->device);
  auto upload = [&](void** dst, const void* src, size_t bytes) {
    if (e == cudaSuccess && bytes) e = cudaMalloc(dst, bytes);
    if (e == cudaSuccess && bytes) e = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
  };
  upload(&s.groups, groups, (size_t)n * sizeof(D));
  upload((void**)&s.cta_map, cta_map.data(), cta_map.size() * sizeof(CtaMapEntry));
  upload((void**)&s.env_group, env_group.data(), env_group.size() * sizeof(uint16_t));
  if (e != cudaSuccess) {
    release_groups(s);
    return cuda_fail(ctx, e, "group set upload");
  }
  release_groups(set);
  set = s;
  return MDPP_OK;
}

// A grouped launch's binding to its set: its n_envs must be the set's total.
// The launch then takes set.groups, the map and set.n_ctas.  Costs a compare
// on success (step() is launch-bound).
inline int bind_groups(mdpp_ctx* ctx, const GroupSet& set, const char* entry,
                       int64_t n_envs) {
  if (n_envs == set.n_envs) return MDPP_OK;
  return fail(ctx, MDPP_EINVAL, std::string(entry) + ": n_envs = " +
              std::to_string(n_envs) + " differs from the groups' total of " +
              std::to_string(set.n_envs) + " envs");
}
}  // namespace mdpp

#define MDPP_CUDA(ctx, call)                                      \
  do {                                                            \
    cudaError_t e_ = (call);                                      \
    if (e_ != cudaSuccess) return mdpp::cuda_fail(ctx, e_, #call); \
  } while (0)
