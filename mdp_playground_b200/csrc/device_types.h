// Types shared by host and device code of libmdpp_b200.so.  Also compiled by
// NVRTC (jit.cu), so it only needs the fixed-width integer types.
#pragma once
#include "mdpp_b200.h"

namespace mdpp {

// Device-side descriptor of one discrete configuration group.  The tables of
// the group live in one contiguous, 16-byte aligned blob so that a CTA can
// stage them into shared memory with 128-bit copies.
struct DiscreteGroupDev {
  int32_t S, A, L, delay, every_n, custom_reward, n_seq, key_bits;
  int32_t has_pnoise, has_rnoise, lookup_kind, hash_shift;  // kind: 0 LUT 1 hash 2 R
  uint32_t hash_mask;
  int32_t cdf_log2;    // cdf rows hold 2^cdf_log2 entries (sentinel padded)
  int32_t cdf_stride;  // = 2^cdf_log2
  int32_t has_guide;
  uint64_t key_mask;
  double p_noise, r_std, scale, shift, term_reward_scaled;
  // byte offsets inside the blob
  int32_t off_P, off_term, off_init_cdf, off_noise_cdf;
  int32_t off_lut, off_hash_keys, off_hash_vals, off_values, off_R, off_guide;
  int32_t blob_bytes;
  // Philox-mode transition noise in closed form (context.cu, noise_params):
  // noisy iff w < pn_T; then k = (w * pn_M) >> (32 + pn_shift) in [0, S-2] and
  // the noisy state is (P[s,a] + 1 + k) mod S: uniform over the S-1 others
  uint32_t pn_M;
  int32_t pn_shift;
  uint64_t pn_T;
  uint64_t term_mask;  // bit s = terminal(s); valid when S <= 64
  int64_t blob_offset;  // of this group's blob inside the context blob buffer
  int64_t env_begin, env_count;
  int64_t gid_base;  // global Philox id of the group's first env
  // irrelevant sub-MDP (S1 == 0: none): u16 table, padded cdfs like above
  int32_t S1, A1, irr_cdf_log2, irr_cdf_stride;
  int32_t off_P_irr, off_init_cdf_irr, off_noise_cdf_irr;
  int32_t irr_pn_shift;
  uint32_t irr_pn_M;  // noisy iff w < pn_T (same p); index among the S1-1 others
  // transition tables stored as u8 (S, S1 <= 256: one LEA + LDS.U8 per lookup)
  // instead of u16
  uint32_t p_is_u8;
};

struct CtaMapEntry {
  int32_t group;
  int32_t chunk;  // chunk index inside the group (units of block size)
};

// LUT: fp64 rewards indexed by the key; LUT8: one byte per key indexing the
// (<= 255) distinct reward values -- 8x smaller, for keys of 10-12 bits;
// HASH: open addressing on the 64-bit key; MATRIX: custom R[s, a].
enum { LOOKUP_LUT = 0, LOOKUP_HASH = 1, LOOKUP_MATRIX = 2, LOOKUP_LUT8 = 3 };
constexpr int kLutF64MaxBytes = 4096;
constexpr int kLutMaxBits = 12;
constexpr uint64_t kHashEmpty = ~0ull;
constexpr int kGuideBits = 12;
constexpr int kGuideEntries = 1 << kGuideBits;
constexpr uint8_t kGuideMiss = 0xFF;


struct RolloutParams {
  DiscreteGroupDev group0;  // copy of groups[0]: FAST kernels (single group)
                            // read it from the constant bank / uniform regs
  const DiscreteGroupDev* groups;
  const uint8_t* blob;
  const CtaMapEntry* cta_map;
  mdpp_discrete_state st;
  mdpp_discrete_io io;
  int32_t T, autoreset, horizon;
  int32_t ring_smem_bytes;
  int32_t tab_smem_bytes;  // shared-memory bytes reserved for the group tables
  uint32_t k0, k1;
  uint32_t rk[20];  // Philox round keys expanded from (k0, k1) by the host
  uint64_t step_index;
  const uint64_t* step_index_dev;  // optional device counter added to step_index
  int64_t env_id_offset;
  int32_t irr;  // every group has an irrelevant sub-MDP: I/O rows of 2
  int32_t n_groups;
  const uint8_t* zig;  // ziggurat tables (ziggurat.cuh), MDPP_NORMAL_ZIGGURAT
};

// What a learner riding along a rollout kernel sees of one step
// (discrete_kernels.cuh rollout_body, grid.cu grid_rollout_kernel).
struct StepOut {
  double r;      // the returned reward
  int32_t nxt;   // state (grid: cell index) before any auto-reset (final_obs)
  bool done, trunc;
};

// The per-env episode returns every learner keeps: the running episode's,
// and the sum / count of the returns of those that ended in an auto-reset.
struct ReturnsDev {
  double* ep_return;
  double* ret_sum;
  int32_t* ret_count;
};

// Device view of the outputs of mdpp_eval_params (qlearn.cu check_eval_params):
// per env, the return sum, count and length sum of the first `episodes`
// episodes of an evaluation launch.
struct EvalDev {
  double* ret_sum;
  int32_t* ret_count;
  int64_t* len_sum;
  int32_t episodes;
};

// One env's evaluation episodes, kept in registers over the launch.  The env
// starts a fresh episode at the launch's first step (the caller resets it);
// an episode ends on terminated or truncated (auto-reset), and only the
// first `episodes` are added.
struct EvalEpisodes {
  double ret, sum;   // running episode's return; sum over the counted ones
  int64_t len_sum;
  int32_t len, count;

  __device__ __forceinline__ void begin() {
    ret = sum = 0.0;
    len_sum = 0;
    len = count = 0;
  }
  __device__ __forceinline__ void step(const EvalDev& d, double r, bool ended) {
    if (count < d.episodes) {
      ret = __dadd_rn(ret, r);
      len += 1;
      if (ended) {
        sum = __dadd_rn(sum, ret);
        len_sum += len;
        count += 1;
        ret = 0.0;
        len = 0;
      }
    }
  }
  __device__ __forceinline__ void end(const EvalDev& d, int64_t env) const {
    d.ret_sum[env] = sum;
    d.ret_count[env] = count;
    d.len_sum[env] = len_sum;
  }
};

// Device view of mdpp_eval_params for the greedy tabular agents.
struct QevalDev {
  const double* q;
  int32_t q_states, q_actions;
  EvalDev ev;
};

// Device view of mdpp_qlearn_params (qlearn.cu check_qlearn_params).
struct QlearnDev {
  double* q;
  int32_t q_states, q_actions;
  double alpha, gamma;
  uint64_t explore_below;  // explore iff the exploring word < ceil(epsilon * 2^32)
  ReturnsDev ret;
  int32_t* actions_taken;
};

struct ResetParams {
  const DiscreteGroupDev* groups;
  const uint8_t* blob;
  const CtaMapEntry* cta_map;
  mdpp_discrete_state st;
  const uint8_t* mask;
  const int32_t* init_states;
  const double* replay_reset_u;
  int64_t* obs;
  int32_t noise_mode;
  uint32_t k0, k1;
  uint64_t step_index;
  int64_t env_id_offset;
  int32_t irr;
  int32_t n_groups;
};

}  // namespace mdpp
