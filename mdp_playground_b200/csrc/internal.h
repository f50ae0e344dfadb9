// Internal declarations shared by the translation units of libmdpp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>


#include "device_types.h"


struct mdpp_ctx {
  int device = 0;
  int sm_count = 0;
  int max_smem_optin = 0;
  std::string error;
  // discrete tables
  std::vector<mdpp::DiscreteGroupDev> d_groups_host;
  mdpp::DiscreteGroupDev* d_groups = nullptr;
  uint8_t* d_blob = nullptr;
  size_t d_blob_bytes = 0;
  int max_group_blob = 0;
  int max_delay = 0;
  int64_t d_total_envs = 0;
  int d_irr = 0;  // groups carry an irrelevant sub-MDP
  uint8_t* d_zig = nullptr;  // ziggurat tables (ziggurat.cuh layout), per context
  // CTA -> (group, chunk) map, one per supported block size
  mdpp::CtaMapEntry* d_cta_map = nullptr;
  int cta_map_block = 0;
  int64_t n_ctas = 0;
  // continuous configuration (one per context)
  bool have_continuous = false;
  mdpp_continuous_config c_cfg;
  // heterogeneous continuous launches (mdpp_set_continuous_groups)
  void* c_groups = nullptr;   // ContinuousGroupDev[n]
  void* c_cta_map = nullptr;  // CtaMapEntry[c_n_ctas]
  int c_n_groups = 0;
  int64_t c_n_ctas = 0, c_total_envs = 0;
  bool have_grid = false;
  mdpp_grid_config g_cfg;
  // heterogeneous grid launches (mdpp_set_grid_groups)
  void* g_groups = nullptr;   // GridGroupDev[n]
  void* g_cta_map = nullptr;  // CtaMapEntry[g_n_ctas]
  int g_n_groups = 0;
  int64_t g_n_ctas = 0, g_total_envs = 0;
  // per-group image renderers (mdpp_set_image_discrete_groups /
  // mdpp_set_image_continuous_groups): the group descriptors and an
  // env -> group map, one load per image
  mdpp_image_discrete_group* img_d_groups = nullptr;  // [img_d_n_groups]
  uint16_t* img_d_env_group = nullptr;                // [img_d_total_envs]
  mdpp_image_discrete_tables img_d_first;  // group 0's (shared sizes), any-rotate
  int img_d_n_groups = 0;
  int64_t img_d_total_envs = 0;
  mdpp_image_continuous_group* img_c_groups = nullptr;
  uint16_t* img_c_env_group = nullptr;
  mdpp_image_continuous_config img_c_first;
  int img_c_n_groups = 0;
  int64_t img_c_total_envs = 0;
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
void render_release(mdpp_ctx* ctx);  // render.cu: the per-group image descriptors
int smem_min_steps();  // MDPP_SMEM_MIN_T (default 1): shorter launches skip the smem staging
int fail(mdpp_ctx* ctx, int code, const std::string& msg);
// discrete.cu: validate a discrete launch and fill its parameters
int prepare_rollout(mdpp_ctx* ctx, const mdpp_discrete_state* st,
                    const mdpp_discrete_io* io, const mdpp_step_opts* opts,
                    RolloutParams& p);
int cuda_fail(mdpp_ctx* ctx, cudaError_t e, const char* what);
}  // namespace mdpp

#define MDPP_CUDA(ctx, call)                                      \
  do {                                                            \
    cudaError_t e_ = (call);                                      \
    if (e_ != cudaSuccess) return mdpp::cuda_fail(ctx, e_, #call); \
  } while (0)
