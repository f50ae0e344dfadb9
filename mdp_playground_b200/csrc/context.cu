// Context lifetime, error reporting and host-side packing of the discrete
// tables into the device blob (LUT / open-addressing hash of sequence keys).
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "discrete_kernels.cuh"  // kBlock: the rollout's CTA size
#include "internal.h"
#include "ziggurat.cuh"
#include "ziggurat_tables.h"

namespace {
thread_local std::string g_create_error;
}

namespace mdpp {
int fail(mdpp_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->error = msg; else g_create_error = msg;
  return code;
}
int cuda_fail(mdpp_ctx* ctx, cudaError_t e, const char* what) {
  return fail(ctx, MDPP_ECUDA,
              std::string(what) + ": " + cudaGetErrorName(e) + " (" +
                  cudaGetErrorString(e) + ")");
}
}  // namespace mdpp

using namespace mdpp;

extern "C" int mdpp_abi_version(void) { return MDPP_ABI_VERSION; }

extern "C" const char* mdpp_last_error(const mdpp_ctx* ctx) {
  return ctx ? ctx->error.c_str() : g_create_error.c_str();
}

extern "C" void mdpp_ziggurat_tables(const uint64_t** ki, const uint64_t** wi_bits,
                                     const uint64_t** fi_bits) {
  if (ki) *ki = kZigKi;
  if (wi_bits) *wi_bits = kZigWiBits;
  if (fi_bits) *fi_bits = kZigFiBits;
}

extern "C" int mdpp_create(int device, mdpp_ctx** out_ctx) {
  if (!out_ctx) return fail(nullptr, MDPP_EINVAL, "out_ctx is NULL");
  *out_ctx = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceCount");
  if (device < 0 || device >= n)
    return fail(nullptr, MDPP_EINVAL, "no such CUDA device");
  mdpp_ctx* ctx = new mdpp_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    delete ctx;
    return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
  }
  const char* jit_env = std::getenv("MDPP_JIT");
  ctx->jit_enabled = !(jit_env && jit_env[0] == '0');
  ctx->sm_count = prop.multiProcessorCount;
  ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  {  // ziggurat tables: {wi, (double)ki}[256] for the fast path, then fi[256]
    std::vector<uint64_t> z(kZigBytes / 8);
    for (int i = 0; i < kZigLayers; ++i) {
      z[kZigOffFast / 8 + 2 * i] = kZigWiBits[i];
      const double kid = (double)kZigKi[i];  // exact: ki < 2^52
      std::memcpy(&z[kZigOffFast / 8 + 2 * i + 1], &kid, 8);
      z[kZigOffFi / 8 + i] = kZigFiBits[i];
    }
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_zig, kZigBytes);
    if (e == cudaSuccess)
      e = cudaMemcpy(ctx->d_zig, z.data(), kZigBytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      delete ctx;
      return cuda_fail(nullptr, e, "ziggurat table upload");
    }
  }
  *out_ctx = ctx;
  return MDPP_OK;
}

extern "C" void mdpp_destroy(mdpp_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  jit_release(ctx);
  if (ctx->d_blob) cudaFree(ctx->d_blob);
  if (ctx->d_zig) cudaFree(ctx->d_zig);
  for (GroupSet* set : {&ctx->d_set, &ctx->c_set, &ctx->g_set, &ctx->img_d_set,
                        &ctx->img_c_set})
    release_groups(*set);
  delete ctx;
}

namespace {

inline int align_up(int x, int a) { return (x + a - 1) / a * a; }

inline int bits_for(int n_states) {
  int b = 1;
  while ((1 << b) < n_states) ++b;
  return b;
}

inline uint32_t hash_slot(uint64_t key, int shift, uint32_t mask) {
  return (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> shift) & mask;
}

}  // namespace

extern "C" int mdpp_set_discrete_groups(mdpp_ctx* ctx,
                                        const mdpp_discrete_group* groups,
                                        int32_t n_groups) {
  if (!ctx) return MDPP_EINVAL;
  int rc = validate_groups(ctx, __func__, groups, n_groups, /*env_map=*/false);
  if (rc) return rc;
  std::vector<DiscreteGroupDev> dev(n_groups);
  std::vector<uint8_t> blob;
  int max_group_blob = 0, max_delay = 0;
  const int irr = groups[0].n_states_irr > 0;
  for (int g = 0; g < n_groups; ++g) {
    const mdpp_discrete_group& in = groups[g];
    DiscreteGroupDev& d = dev[g];
    std::memset(&d, 0, sizeof(d));
    const int S = in.n_states, A = in.n_actions, L = in.sequence_length;
    if (S < 1 || S > 65535 || A < 1 || L < 1 || in.delay < 0 ||
        in.reward_every_n_steps < 1)
      return fail(ctx, MDPP_EINVAL, "discrete group: bad sizes");
    if (!in.transition || !in.terminal || !in.init_cdf)
      return fail(ctx, MDPP_EINVAL, "discrete group: missing table");
    if (in.has_transition_noise && !in.noise_cdf)
      return fail(ctx, MDPP_EINVAL, "transition noise needs noise_cdf");
    if ((in.n_states_irr > 0) != (irr != 0))
      return fail(ctx, MDPP_EINVAL,
                  "all groups must agree on having an irrelevant sub-MDP");
    if (in.n_states_irr > 0 &&
        (in.n_states_irr > 65535 || in.n_actions_irr < 1 || !in.transition_irr ||
         !in.init_cdf_irr || (in.has_transition_noise && !in.noise_cdf_irr)))
      return fail(ctx, MDPP_EINVAL, "discrete group: bad irrelevant sub-MDP");
    const int b = bits_for(S);
    if ((int64_t)b * L > 63)
      return fail(ctx, MDPP_EINVAL,
                  "sequence key does not fit 63 bits (bits(S)*L > 63)");
    d.S = S; d.A = A; d.L = L; d.delay = in.delay;
    d.every_n = in.reward_every_n_steps;
    d.custom_reward = in.custom_reward;
    d.n_seq = in.n_sequences;
    d.key_bits = b;
    d.key_mask = (b * L == 64) ? ~0ull : ((1ull << (b * L)) - 1ull);
    d.has_pnoise = in.has_transition_noise;
    d.has_rnoise = in.has_reward_noise;
    d.p_noise = in.transition_noise;
    d.r_std = in.reward_noise_std;
    d.scale = in.reward_scale;
    d.shift = in.reward_shift;
    // rl_toy_env.py:2107-2109: reward += term_state_reward * reward_scale
    d.term_reward_scaled = in.term_state_reward * in.reward_scale;
    d.env_begin = in.env_begin;
    d.gid_base = in.global_id_base;
    d.env_count = in.env_count;
    if (in.delay > max_delay) max_delay = in.delay;

    // ---- pack the blob -------------------------------------------------
    std::vector<uint8_t> gb;
    auto reserve = [&](int bytes, int align) {
      int off = align_up((int)gb.size(), align);
      gb.resize(off + bytes, 0);
      return off;
    };
    for (int i = 0; i < S * A; ++i)
      if (in.transition[i] < 0 || in.transition[i] >= S)
        return fail(ctx, MDPP_EINVAL, "transition table entry out of range");
    d.p_is_u8 = S <= 256 && in.n_states_irr <= 256;
    d.off_P = reserve(S * A * (d.p_is_u8 ? 1 : 2), 16);
    if (d.p_is_u8) {
      for (int i = 0; i < S * A; ++i) gb[d.off_P + i] = (uint8_t)in.transition[i];
    } else {
      uint16_t* P = reinterpret_cast<uint16_t*>(gb.data() + d.off_P);
      for (int i = 0; i < S * A; ++i) P[i] = (uint16_t)in.transition[i];
    }
    d.off_term = reserve(S, 16);
    std::memcpy(gb.data() + d.off_term, in.terminal, S);
    // cdf rows are padded to a power of two with a sentinel (2.0 > any u) so
    // that the device can run a fixed-trip, branch-free binary search
    int log2pad = 0;
    while ((1 << log2pad) < S) ++log2pad;
    const int Sp = 1 << log2pad;
    d.cdf_log2 = log2pad;
    d.cdf_stride = Sp;
    auto put_row = [&](double* dst, const double* src) {
      for (int k = 0; k < Sp; ++k) dst[k] = k < S ? src[k] : 2.0;
    };
    d.off_init_cdf = reserve(Sp * 8, 16);
    put_row(reinterpret_cast<double*>(gb.data() + d.off_init_cdf), in.init_cdf);
    if (in.has_transition_noise) {
      d.off_noise_cdf = reserve(S * Sp * 8, 16);
      for (int r = 0; r < S; ++r)
        put_row(reinterpret_cast<double*>(gb.data() + d.off_noise_cdf) + (size_t)r * Sp,
                in.noise_cdf + (size_t)r * S);
    }
    // Philox-mode transition noise in closed form.  The reference's noisy
    // distribution (rl_toy_env.py:1606-1617) is P(P[s,a]) = 1 - p and p / (S-1)
    // for each other state, so a 32-bit word w decides: noisy iff w < T with
    // T = round(p 2^32); given that, w is uniform on [0, T) and
    // k = floor(w M / 2^sh), M = floor((S-1) 2^sh / T), is uniform on [0, S-2]
    // (every value within 2^-32 of its probability; k <= S-2 because M is
    // rounded down).  The noisy state is (P[s,a] + 1 + k) mod S, i.e. one of
    // the S-1 other states.  Only that last add depends on the env state; the
    // rest is drawn ahead.
    auto noise_params = [&](int n_states, uint32_t* pn_M, int32_t* pn_shift) {
      double t = std::floor(in.transition_noise * 4294967296.0 + 0.5);
      uint64_t T = t <= 0.0 ? 0ull : t >= 4294967296.0 ? (1ull << 32) : (uint64_t)t;
      d.pn_T = T;
      if (T > 0) {
        int sh = 63;
        unsigned __int128 M;
        while (((M = (((unsigned __int128)(n_states - 1)) << sh) / T) >> 32) && sh > 32) --sh;
        // T < S-1 (p below ~S 2^-32) cannot be uniform over the others anyway
        *pn_M = (M >> 32) ? 0xFFFFFFFFu : (uint32_t)M;
        *pn_shift = sh - 32;
      }
    };
    if (in.has_transition_noise && S >= 2) noise_params(S, &d.pn_M, &d.pn_shift);
    if (in.n_states_irr > 0) {  // the irrelevant sub-MDP's tables, same formats
      const int S1 = in.n_states_irr, A1 = in.n_actions_irr;
      d.S1 = S1; d.A1 = A1;
      for (int i = 0; i < S1 * A1; ++i)
        if (in.transition_irr[i] < 0 || in.transition_irr[i] >= S1)
          return fail(ctx, MDPP_EINVAL, "irrelevant transition entry out of range");
      d.off_P_irr = reserve(S1 * A1 * (d.p_is_u8 ? 1 : 2), 16);
      if (d.p_is_u8) {
        for (int i = 0; i < S1 * A1; ++i)
          gb[d.off_P_irr + i] = (uint8_t)in.transition_irr[i];
      } else {
        uint16_t* P = reinterpret_cast<uint16_t*>(gb.data() + d.off_P_irr);
        for (int i = 0; i < S1 * A1; ++i) P[i] = (uint16_t)in.transition_irr[i];
      }
      int lg = 0;
      while ((1 << lg) < S1) ++lg;
      const int S1p = 1 << lg;
      d.irr_cdf_log2 = lg;
      d.irr_cdf_stride = S1p;
      auto put_row1 = [&](double* dst, const double* src) {
        for (int k = 0; k < S1p; ++k) dst[k] = k < S1 ? src[k] : 2.0;
      };
      d.off_init_cdf_irr = reserve(S1p * 8, 16);
      put_row1(reinterpret_cast<double*>(gb.data() + d.off_init_cdf_irr), in.init_cdf_irr);
      if (in.has_transition_noise) {
        d.off_noise_cdf_irr = reserve(S1 * S1p * 8, 16);
        for (int r = 0; r < S1; ++r)
          put_row1(reinterpret_cast<double*>(gb.data() + d.off_noise_cdf_irr) + (size_t)r * S1p,
                   in.noise_cdf_irr + (size_t)r * S1);
        if (S1 >= 2) noise_params(S1, &d.irr_pn_M, &d.irr_pn_shift);
      }
    }
    if (S <= 64)
      for (int k = 0; k < S; ++k)
        if (in.terminal[k]) d.term_mask |= 1ull << k;
    // Guide table of the auto-reset draw: bucket b = top 12 bits of the 32-bit
    // Philox word w (u = (w + 0.5) 2^-32).  If every w of the bucket maps to
    // the same initial state the entry holds it, else kGuideMiss (the device
    // then runs the search).  Exact: the bucket's extreme u values are
    // representable, and searchsorted is monotone in u.
    if (S <= 254) {
      d.has_guide = 1;
      d.off_guide = reserve(kGuideEntries, 16);
      uint8_t* guide = gb.data() + d.off_guide;
      auto search = [&](double u) {
        int n = 0;
        for (int k = 0; k < S; ++k) n += in.init_cdf[k] <= u;
        return n < S ? n : S - 1;
      };
      for (int b = 0; b < kGuideEntries; ++b) {
        const uint64_t w_lo = (uint64_t)b << (32 - kGuideBits);
        const uint64_t w_hi = (((uint64_t)b + 1) << (32 - kGuideBits)) - 1;
        const int s_lo = search(((double)w_lo + 0.5) * (1.0 / 4294967296.0));
        const int s_hi = search(((double)w_hi + 0.5) * (1.0 / 4294967296.0));
        guide[b] = s_lo == s_hi ? (uint8_t)s_lo : kGuideMiss;
      }
    }
    if (in.custom_reward) {
      if (!in.reward_matrix)
        return fail(ctx, MDPP_EINVAL, "custom_reward needs reward_matrix");
      d.lookup_kind = LOOKUP_MATRIX;
      d.off_R = reserve(S * A * 8, 16);
      // "+ 0.0" maps a -0.0 entry to +0.0 (same for the value tables below):
      // with no negative zero entering the reward arithmetic the kernels may
      // drop `* 1.0` and `+ 0.0` without changing a single result bit
      double* R = reinterpret_cast<double*>(gb.data() + d.off_R);
      for (int i = 0; i < S * A; ++i) R[i] = in.reward_matrix[i] + 0.0;
    } else {
      if (in.n_sequences < 0 || (in.n_sequences > 0 &&
                                 (!in.sequences || !in.sequence_rewards)))
        return fail(ctx, MDPP_EINVAL, "missing rewardable sequences");
      const int n = in.n_sequences;
      std::vector<uint64_t> keys(n);
      for (int i = 0; i < n; ++i) {
        uint64_t k = 0;
        for (int j = 0; j < L; ++j) {
          int s = in.sequences[(size_t)i * L + j];
          if (s < 0 || s >= S)
            return fail(ctx, MDPP_EINVAL, "sequence state out of range");
          k = (k << b) | (uint64_t)s;  // oldest state highest, newest lowest
        }
        keys[i] = k;
      }
      // distinct reward values (by bit pattern), 0.0 first
      std::vector<double> uniq = {0.0};
      std::vector<int> uidx(n);
      for (int i = 0; i < n; ++i) {
        const double r = in.sequence_rewards[i] + 0.0;
        size_t k = 0;
        while (k < uniq.size() && std::memcmp(&uniq[k], &r, 8) != 0) ++k;
        if (k == uniq.size()) uniq.push_back(r);
        uidx[i] = (int)k;
      }
      const int entries = b * L <= kLutMaxBits ? 1 << (b * L) : 0;
      if (entries && entries * 8 <= kLutF64MaxBytes) {
        d.lookup_kind = LOOKUP_LUT;
        d.off_lut = reserve(entries * 8, 16);  // rewards stored directly
        double* lut = reinterpret_cast<double*>(gb.data() + d.off_lut);
        for (int i = 0; i < n; ++i) lut[keys[i]] = in.sequence_rewards[i] + 0.0;
      } else if (entries && uniq.size() <= 255) {
        // a big fp64 table per CTA would cap the occupancy of multi-group
        // launches (every CTA gets the largest group's shared memory)
        d.lookup_kind = LOOKUP_LUT8;
        d.off_values = reserve((int)uniq.size() * 8, 16);  // replaces the per-sequence list
        std::memcpy(gb.data() + d.off_values, uniq.data(), uniq.size() * 8);
        d.off_lut = reserve(entries, 16);
        uint8_t* lut = gb.data() + d.off_lut;
        for (int i = 0; i < n; ++i) lut[keys[i]] = (uint8_t)uidx[i];
      } else {
        d.lookup_kind = LOOKUP_HASH;
        d.off_values = reserve((n + 1) * 8, 16);
        {
          double* v = reinterpret_cast<double*>(gb.data() + d.off_values);
          v[0] = 0.0;
          for (int i = 0; i < n; ++i) v[i + 1] = in.sequence_rewards[i] + 0.0;
        }
        int log2cap = 4;
        while ((1 << log2cap) < 2 * n) ++log2cap;
        const uint32_t cap = 1u << log2cap;
        d.hash_mask = cap - 1;
        d.hash_shift = 64 - log2cap;
        d.off_hash_keys = reserve(cap * 8, 16);
        d.off_hash_vals = reserve(cap * 4, 16);
        uint64_t* hk = reinterpret_cast<uint64_t*>(gb.data() + d.off_hash_keys);
        uint32_t* hv = reinterpret_cast<uint32_t*>(gb.data() + d.off_hash_vals);
        for (uint32_t i = 0; i < cap; ++i) hk[i] = kHashEmpty;
        for (int i = 0; i < n; ++i) {
          uint32_t slot = hash_slot(keys[i], d.hash_shift, d.hash_mask);
          while (hk[slot] != kHashEmpty && hk[slot] != keys[i])
            slot = (slot + 1) & d.hash_mask;
          hk[slot] = keys[i];
          hv[slot] = (uint32_t)(i + 1);  // later duplicates win, like a dict
        }
      }
    }
    d.blob_bytes = align_up((int)gb.size(), 16);
    gb.resize(d.blob_bytes, 0);
    d.blob_offset = (int64_t)blob.size();
    blob.insert(blob.end(), gb.begin(), gb.end());
    if (d.blob_bytes > max_group_blob) max_group_blob = d.blob_bytes;
  }
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  uint8_t* d_blob = nullptr;
  cudaError_t e = cudaMalloc(&d_blob, blob.size());
  if (e == cudaSuccess)
    e = cudaMemcpy(d_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice);
  rc = e == cudaSuccess ? install_groups(ctx, ctx->d_set, dev.data(), n_groups, kBlock)
                        : cuda_fail(ctx, e, "discrete table upload");
  if (rc) {
    if (d_blob) cudaFree(d_blob);
    return rc;
  }
  if (ctx->d_blob) cudaFree(ctx->d_blob);
  ctx->d_blob = d_blob;
  ctx->d_blob_bytes = blob.size();
  ctx->d_groups_host = dev;
  ctx->max_group_blob = max_group_blob;
  ctx->max_delay = max_delay;
  ctx->d_irr = irr;
  ctx->d_groups_version += 1;
  return MDPP_OK;
}
