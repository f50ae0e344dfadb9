// Host-side selection and launch of the ahead-of-time rollout kernels.
#pragma once
#include "discrete_kernels.cuh"
#include "internal.h"

namespace mdpp {

// Ring of delayed rewards lives in shared memory when it is small enough.
constexpr int kRingSmemMaxDelay = 16;

// Launch `kern` with argument `kp` for configuration C.  `p` is the rollout
// part of `kp` (kp itself for the rollout kernels): its shared-memory sizes
// are set here, before the launch copies `kp`.
template <typename C, typename KP>
inline int launch_kernel(mdpp_ctx* ctx, RolloutParams& p, int smem_tab,
                         cudaStream_t stream, void (*kern)(KP), const KP& kp) {
  p.ring_smem_bytes = C::RING_SMEM ? ctx->max_delay * kBlock * 8 : 0;
  p.tab_smem_bytes = C::SMEM ? smem_tab : 0;
  const bool zig = C::NORMAL == MDPP_NORMAL_ZIGGURAT && C::NOISE == MDPP_NOISE_PHILOX;
  const int smem = p.ring_smem_bytes + p.tab_smem_bytes +
                   (zig && C::SMEM ? kZigBytes + zig_stage_bytes(kBlock) : 0);
  if (smem > 48 * 1024 - 512)
    MDPP_CUDA(ctx, cudaFuncSetAttribute(
                       kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  // programmatic dependent launch for step()-granularity launches: the table
  // staging overlaps the tail of the previous kernel of the stream
  // (rollout_body waits with griddepcontrol.wait before it touches anything
  // mutable).  Long rollouts gain nothing and measured 2-3 % slower with it.
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ctx->d_set.n_ctas);
  cfg.blockDim = dim3(kBlock);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = p.T < kChunk ? 1 : 0;
  MDPP_CUDA(ctx, cudaLaunchKernelEx(&cfg, kern, kp));
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

template <typename C>
inline int launch_one(mdpp_ctx* ctx, RolloutParams& p, int smem_tab,
                      cudaStream_t stream) {
  return launch_kernel<C>(ctx, p, smem_tab, stream, discrete_rollout_kernel<C>, p);
}

// Whether the group tables (and the delay ring) of a launch go to shared
// memory: `ring_ok` the ring, the return value the tables.
inline bool tables_in_smem(const mdpp_ctx* ctx, const RolloutParams& p, bool* ring_ok) {
  *ring_ok = ctx->max_delay <= kRingSmemMaxDelay;
  const int ring_bytes = *ring_ok ? ctx->max_delay * kBlock * 8 : 0;
  return p.T >= smem_min_steps() &&
         ctx->max_group_blob + ring_bytes + kZigBytes + zig_stage_bytes(kBlock) <=
             ctx->max_smem_optin - 1024;
}

// Kernel variants.  The FAST ones (standard signature, tables + ring in
// shared memory) exist for the throughput-relevant noise modes, with the cdf
// search unrolled for <= 8 states (the toy sizes of BASELINE.json) or looped;
// everything else (replay, huge tables, deep delay rings, optional outputs)
// takes the generic variants.
template <int NOISE, int NORMAL>
inline int launch_rollout(mdpp_ctx* ctx, RolloutParams& p, cudaStream_t stream) {
  const int smem_tab = ctx->max_group_blob;
  bool ring_ok;
  const bool smem_ok = tables_in_smem(ctx, p, &ring_ok);
  const bool fast_io = p.io.actions && p.io.obs && p.io.reward &&
                       p.io.terminated && p.io.truncated && !p.io.final_obs &&
                       !p.st.history && !p.irr;  // (FAST kernels: no sub-MDP)
  if constexpr (NOISE != MDPP_NOISE_REPLAY) {
    if (smem_ok && ring_ok && fast_io && ctx->d_groups_host.size() == 1) {
      return ctx->d_groups_host[0].cdf_log2 == 3
          ? launch_one<Cfg<NOISE, NORMAL, true, true, true, 3, true>>(ctx, p, smem_tab, stream)
          : launch_one<Cfg<NOISE, NORMAL, true, true, true, -1, true>>(ctx, p, smem_tab, stream);
    }
  }
  if (smem_ok && ring_ok)
    return launch_one<Cfg<NOISE, NORMAL, true, true, false, -1>>(ctx, p, smem_tab, stream);
  return launch_one<Cfg<NOISE, NORMAL, false, false, false, -1>>(ctx, p, smem_tab, stream);
}

}  // namespace mdpp
