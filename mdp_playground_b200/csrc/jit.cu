// Runtime specialisation of the discrete rollout kernel (NVRTC).
//
// The ahead-of-time kernels read every group scalar (S, A, L, delay, noise
// flags, scale, ...) at run time, which costs ~290 issued instructions per
// env-step on a path that is issue-bound at 65 536 envs.  For single-group
// launches the same hand-written source (discrete_kernels.cuh, embedded in
// the library at build time) is compiled once per configuration with those
// scalars as literals (-DMDPP_JIT -DMDPP_S=8 ...): searches unroll, dead
// features vanish, ~160 instructions per env-step remain.  The cubin is
// loaded through the driver API and cached in the context.
//
// libnvrtc / libcuda are dlopen()ed lazily so the library still loads on
// machines without a driver (the CPU-side ABI tests).  If either is missing,
// or MDPP_JIT=0 is set, the caller falls back to the AOT kernels.
#include <cuda.h>  // driver API types only; the symbols are dlsym()ed
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "continuous_kernels.cuh"
#include "discrete_kernels.cuh"
#include "embedded_sources.inc"
#include "internal.h"

namespace mdpp {
namespace {

typedef int nvrtcResult;
typedef struct _nvrtcProgram* nvrtcProgram;

struct Api {
  bool tried = false, ok = false;
  std::string why;
  nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int,
                               const char* const*, const char* const*);
  nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*);
  nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*);
  nvrtcResult (*GetCUBIN)(nvrtcProgram, char*);
  nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*);
  nvrtcResult (*GetProgramLog)(nvrtcProgram, char*);
  nvrtcResult (*DestroyProgram)(nvrtcProgram*);
  CUresult (*ModuleLoadData)(CUmodule*, const void*);
  CUresult (*ModuleUnload)(CUmodule);
  CUresult (*ModuleGetFunction)(CUfunction*, CUmodule, const char*);
  CUresult (*FuncSetAttribute)(CUfunction, int, int);
  CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned,
                           unsigned, unsigned, unsigned, CUstream, void**,
                           void**);
  CUresult (*LaunchKernelEx)(const CUlaunchConfig*, CUfunction, void**, void**);
};

Api& api() {
  static Api a;
  if (a.tried) return a;
  a.tried = true;
  void* rtc = nullptr;
  for (const char* n : {"libnvrtc.so.12", "libnvrtc.so",
                        "/usr/local/cuda/lib64/libnvrtc.so.12"}) {
    rtc = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (rtc) break;
  }
  if (!rtc) { a.why = "libnvrtc not found"; return a; }
  void* drv = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
  if (!drv) { a.why = "libcuda.so.1 not found"; return a; }
#define LOAD(lib, field, sym)                                   \
  *(void**)(&a.field) = dlsym(lib, sym);                        \
  if (!a.field) { a.why = std::string("missing ") + sym; return a; }
  LOAD(rtc, CreateProgram, "nvrtcCreateProgram")
  LOAD(rtc, CompileProgram, "nvrtcCompileProgram")
  LOAD(rtc, GetCUBINSize, "nvrtcGetCUBINSize")
  LOAD(rtc, GetCUBIN, "nvrtcGetCUBIN")
  LOAD(rtc, GetProgramLogSize, "nvrtcGetProgramLogSize")
  LOAD(rtc, GetProgramLog, "nvrtcGetProgramLog")
  LOAD(rtc, DestroyProgram, "nvrtcDestroyProgram")
  LOAD(drv, ModuleLoadData, "cuModuleLoadData")
  LOAD(drv, ModuleUnload, "cuModuleUnload")
  LOAD(drv, ModuleGetFunction, "cuModuleGetFunction")
  LOAD(drv, FuncSetAttribute, "cuFuncSetAttribute")
  LOAD(drv, LaunchKernel, "cuLaunchKernel")
  LOAD(drv, LaunchKernelEx, "cuLaunchKernelEx")
#undef LOAD
  a.ok = true;
  return a;
}

std::string hexf(double x) {
  char buf[64];
  std::snprintf(buf, sizeof buf, "%a", x);
  return buf;
}

// The -D list that makes one specialisation; also its cache key.  A group
// scalar becomes a literal only if every group of the launch agrees on it.
std::vector<std::string> defines_for(const std::vector<DiscreteGroupDev>& groups,
                                     const RolloutParams& p, int noise,
                                     int normal, bool fast, bool ring_smem,
                                     int cdf_log2_tpl, bool smem = true,
                                     bool stage = true) {
  auto D = [](const char* k, const std::string& v) {
    return std::string("-DMDPP_") + k + "=" + v;
  };
  auto I = [](long long v) { return std::to_string(v); };
  const DiscreteGroupDev& g = groups[0];
  std::vector<std::string> d = {"-DMDPP_JIT"};
#define UNIFORM(field)                                                    \
  [&] {                                                                   \
    for (auto& h : groups)                                                \
      if (std::memcmp(&h.field, &g.field, sizeof(g.field)) != 0) return false; \
    return true;                                                          \
  }()
  if (UNIFORM(S)) d.push_back(D("S", I(g.S)));
  if (UNIFORM(A)) d.push_back(D("A", I(g.A)));
  if (UNIFORM(L)) d.push_back(D("L", I(g.L)));
  if (UNIFORM(delay)) d.push_back(D("DELAY", I(g.delay)));
  if (UNIFORM(every_n)) d.push_back(D("EVERY_N", I(g.every_n)));
  if (UNIFORM(lookup_kind)) d.push_back(D("LOOKUP", I(g.lookup_kind)));
  if (UNIFORM(key_bits)) d.push_back(D("KEY_BITS", I(g.key_bits)));
  if (UNIFORM(hash_shift)) d.push_back(D("HASH_SHIFT", I(g.hash_shift)));
  if (UNIFORM(hash_mask)) d.push_back(D("HASH_MASK", I(g.hash_mask) + "u"));
  if (UNIFORM(key_mask))
    d.push_back(D("KEY_MASK", std::to_string((unsigned long long)g.key_mask) + "ull"));
  if (UNIFORM(has_pnoise)) d.push_back(D("PNOISE", g.has_pnoise ? "true" : "false"));
  if (UNIFORM(has_rnoise)) d.push_back(D("RNOISE", g.has_rnoise ? "true" : "false"));
  if (UNIFORM(cdf_log2)) d.push_back(D("CDF_LOG2", I(g.cdf_log2)));
  if (UNIFORM(has_guide)) d.push_back(D("HAS_GUIDE", g.has_guide ? "true" : "false"));
  if (UNIFORM(p_is_u8)) d.push_back(D("P8", g.p_is_u8 ? "true" : "false"));
  if (UNIFORM(r_std)) d.push_back(D("R_STD", hexf(g.r_std)));
  if (UNIFORM(scale)) d.push_back(D("SCALE", hexf(g.scale)));
  if (UNIFORM(shift)) d.push_back(D("SHIFT", hexf(g.shift)));
  if (UNIFORM(term_reward_scaled)) d.push_back(D("TERM_REWARD", hexf(g.term_reward_scaled)));
  if (UNIFORM(shift)) d.push_back(D("SHIFT_NEGZERO", std::signbit(g.shift) && g.shift == 0.0 ? "1" : "0"));
  if (UNIFORM(term_reward_scaled))
    d.push_back(D("TERM_NEGZERO",
                  std::signbit(g.term_reward_scaled) && g.term_reward_scaled == 0.0 ? "1" : "0"));
  if (UNIFORM(pn_T) && UNIFORM(pn_M) && UNIFORM(pn_shift)) {
    d.push_back(D("PN_T", std::to_string((unsigned long long)g.pn_T) + "ull"));
    d.push_back(D("PN_M", std::to_string(g.pn_M) + "u"));
    d.push_back(D("PN_SHIFT", I(g.pn_shift)));
  }
  // delay FIFO in registers when every group has the same small delay
  d.push_back(D("CFG_RING_REGS",
                I(UNIFORM(delay) && g.delay >= 1 && g.delay <= kMaxRingRegs ? g.delay : 0)));
#undef UNIFORM
  d.push_back(D("IRR", I(p.irr)));
  d.push_back(D("OBS_DTYPE", I(p.io.obs_dtype)));
  d.push_back(D("N_ENVS", I(p.st.n_envs) + "ll"));
  d.push_back(D("AUTORESET", I(p.autoreset)));
  d.push_back(D("HORIZON", I(p.horizon)));
  d.push_back(D("CFG_NOISE", I(noise)));
  d.push_back(D("CFG_NORMAL", I(normal)));
  d.push_back(D("CFG_FAST", fast ? "true" : "false"));
  d.push_back(D("CFG_RING", ring_smem ? "true" : "false"));
  d.push_back(D("CFG_SMEM", smem ? "true" : "false"));
  d.push_back(D("CFG_STAGE", stage ? "true" : "false"));
  d.push_back(D("CFG_CDF", I(cdf_log2_tpl)));
  d.push_back(D("CFG_SINGLE", groups.size() == 1 ? "true" : "false"));
  return d;
}

const char* kEntrySource = R"SRC(
#include "discrete_kernels.cuh"
using JitCfg = mdpp::Cfg<MDPP_CFG_NOISE, MDPP_CFG_NORMAL, MDPP_CFG_SMEM, MDPP_CFG_RING,
                         MDPP_CFG_FAST, MDPP_CFG_CDF, MDPP_CFG_SINGLE,
                         MDPP_CFG_RING_REGS>;
extern "C" __global__ void __launch_bounds__(mdpp::kBlock, mdpp::kMinBlocksPerSM)
mdpp_jit_rollout(const __grid_constant__ mdpp::RolloutParams p) {
  mdpp::rollout_body<JitCfg>(p);
}
)SRC";

const char* kStdintShim = R"SRC(
#pragma once
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef short int16_t;
typedef unsigned short uint16_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
)SRC";

const char* kHeaderNames[] = {"discrete_kernels.cuh", "continuous_kernels.cuh",
                              "device_types.h", "philox.cuh", "mdpp_b200.h",
                              "stdint.h", "ziggurat.cuh"};
const char* kHeaderSources[] = {kSrc_discrete_kernels_cuh,
                                kSrc_continuous_kernels_cuh, kSrc_device_types_h,
                                kSrc_philox_cuh, kSrc_mdpp_b200_h, kStdintShim,
                                kSrc_ziggurat_cuh};
constexpr int kNumHeaders = 7;

void* compile(mdpp_ctx* ctx, const char* entry_source, const char* entry_name,
              const std::vector<std::string>& defs, void** module_out) {
  Api& a = api();
  nvrtcProgram prog = nullptr;
  if (a.CreateProgram(&prog, entry_source, "mdpp_jit_entry.cu", kNumHeaders,
                      kHeaderSources, kHeaderNames)) {
    ctx->jit_log = "nvrtcCreateProgram failed";
    return nullptr;
  }
  std::vector<std::string> opts = {"--gpu-architecture=sm_100a", "-std=c++17",
                                   "-lineinfo"};
  opts.insert(opts.end(), defs.begin(), defs.end());
  std::vector<const char*> copts;
  for (auto& o : opts) copts.push_back(o.c_str());
  nvrtcResult rc = a.CompileProgram(prog, (int)copts.size(), copts.data());
  if (rc != 0) {
    size_t n = 0;
    a.GetProgramLogSize(prog, &n);
    std::string log(n, '\0');
    if (n) a.GetProgramLog(prog, &log[0]);
    ctx->jit_log = "nvrtc compile failed: " + log;
    a.DestroyProgram(&prog);
    return nullptr;
  }
  size_t size = 0;
  a.GetCUBINSize(prog, &size);
  std::vector<char> cubin(size);
  a.GetCUBIN(prog, cubin.data());
  a.DestroyProgram(&prog);
  CUmodule mod = nullptr;
  if (a.ModuleLoadData(&mod, cubin.data())) {
    ctx->jit_log = "cuModuleLoadData failed";
    return nullptr;
  }
  CUfunction fn = nullptr;
  if (a.ModuleGetFunction(&fn, mod, entry_name)) {
    ctx->jit_log = "cuModuleGetFunction failed";
    a.ModuleUnload(mod);
    return nullptr;
  }
  *module_out = mod;
  return fn;
}

const char* kContinuousEntrySource = R"SRC(
#include "continuous_kernels.cuh"
#ifndef MDPP_C_MINBLOCKS
#define MDPP_C_MINBLOCKS 6  // measured best of 1/5/6/8 on C3 (rollout and T = 1)
#endif
extern "C" __global__ void __launch_bounds__(mdpp::kCBlock, MDPP_C_MINBLOCKS)
mdpp_jit_continuous(const __grid_constant__ mdpp::ContinuousParams p) {
  mdpp::continuous_body<MDPP_C_REAL, MDPP_C_NOISE>(p);
}
)SRC";

// Cached lookup: returns the CUfunction of (entry, defines), compiling it on
// first use; nullptr if NVRTC / the driver API is unavailable or it failed.
void* get_function(mdpp_ctx* ctx, const char* entry_source,
                   const char* entry_name,
                   const std::vector<std::string>& defs) {
  Api& a = api();
  if (!a.ok) { ctx->jit_log = a.why; return nullptr; }
  std::string key = entry_name;
  for (auto& d : defs) { key += ' '; key += d; }
  auto it = ctx->jit_functions.find(key);
  if (it != ctx->jit_functions.end()) return it->second;
  void* mod = nullptr;
  void* fn = compile(ctx, entry_source, entry_name, defs, &mod);
  ctx->jit_functions[key] = fn;  // failures are cached too: no retry per call
  if (fn) ctx->jit_modules.push_back(mod);
  return fn;
}

int launch(mdpp_ctx* ctx, void* fn, unsigned grid, unsigned block, int smem,
           cudaStream_t stream, void* param, bool pdl = false) {
  Api& a = api();
  if (smem > 48 * 1024 - 512) {
    // CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES = 8
    if (a.FuncSetAttribute((CUfunction)fn, 8, smem))
      return fail(ctx, MDPP_ECUDA, "cuFuncSetAttribute(max dynamic smem) failed");
  }
  void* args[] = {param};
  // programmatic dependent launch: the kernel may start while the previous
  // kernel of the stream drains; everything it does before its
  // griddepcontrol.wait touches only immutable tables (rollout_body)
  CUlaunchAttribute attr;
  std::memset(&attr, 0, sizeof attr);
  attr.id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
  attr.value.programmaticStreamSerializationAllowed = 1;
  CUlaunchConfig cfg;
  std::memset(&cfg, 0, sizeof cfg);
  cfg.gridDimX = grid; cfg.gridDimY = 1; cfg.gridDimZ = 1;
  cfg.blockDimX = block; cfg.blockDimY = 1; cfg.blockDimZ = 1;
  cfg.sharedMemBytes = (unsigned)smem;
  cfg.hStream = (CUstream)stream;
  cfg.attrs = &attr;
  cfg.numAttrs = pdl ? 1 : 0;
  CUresult rc = a.LaunchKernelEx(&cfg, (CUfunction)fn, args, nullptr);
  if (rc != 0)
    return fail(ctx, MDPP_ECUDA, "cuLaunchKernel(jit) failed: " + std::to_string(rc));
  ctx->jit_last_used = 1;
  return 1;
}

}  // namespace

int jit_try_continuous(mdpp_ctx* ctx, ContinuousParams& p, cudaStream_t stream) {
  ctx->jit_last_used = 0;
  if (!ctx->jit_enabled) return 0;
  const mdpp_continuous_config& c = p.cfg;
  // signature of the -D list: the whole configuration + the launch shape
  unsigned char sig[sizeof ctx->jit_sig_continuous];
  std::memset(sig, 0, sizeof sig);
  std::memcpy(sig, &c, sizeof c);
  {
    const long long extra[8] = {p.noise_mode, p.normal_mode, p.horizon, p.autoreset,
                                (long long)p.st.n_envs,
                                p.io.obs && p.io.reward && p.io.terminated &&
                                    p.io.truncated && !p.io.final_obs, 1, 0};
    std::memcpy(sig + sizeof c, extra, sizeof extra);
  }
  const unsigned grid0 = (unsigned)((p.st.n_envs + kCBlock - 1) / kCBlock);
  if (std::memcmp(sig, ctx->jit_sig_continuous, sizeof sig) == 0) {
    if (!ctx->jit_fn_continuous) return 0;
    return launch(ctx, ctx->jit_fn_continuous, grid0, kCBlock, 0, stream, &p);
  }
  auto D = [](const char* k, const std::string& v) {
    return std::string("-DMDPP_C_") + k + "=" + v;
  };
  auto I = [](long long v) { return std::to_string(v); };
  auto B = [](bool v) { return std::string(v ? "true" : "false"); };
  std::vector<std::string> defs = {
      "-DMDPP_JIT", D("REAL", c.is_f64 ? "double" : "float"),
      D("NOISE", I(p.noise_mode)), D("DIM", I(c.dim)), D("ORDER", I(c.order)),
      D("NREL", I(c.n_relevant)), D("DELAY", I(c.delay)),
      D("EVERY_N", I(c.reward_every_n_steps)), D("DENSE", B(c.dense)),
      D("PNOISE", B(c.has_transition_noise)), D("RNOISE", B(c.has_reward_noise)),
      D("IMAGE", B(c.image_mode)), D("TARGET64", B(c.target_is_f64)),
      D("NORMAL", I(p.normal_mode)), D("IMODE", I(c.inertia_mode)),
      D("LINE", B(c.reward_kind == MDPP_REWARD_LINE)), D("SEQ", I(c.sequence_length)),
      D("NBOX", I(c.n_term_boxes)), D("HORIZON", I(p.horizon)),
      D("AUTORESET", B(p.autoreset != 0)), D("N_ENVS", I(p.st.n_envs) + "ll"),
      D("FAST", B(p.io.obs && p.io.reward && p.io.terminated && p.io.truncated &&
                  !p.io.final_obs)),
  };
  auto F = [&](const char* k, double v) {
    unsigned long long bits;
    std::memcpy(&bits, &v, 8);
    char buf[40];
    std::snprintf(buf, sizeof buf, "0x%llxll", bits);
    defs.push_back(D((std::string(k) + "_BITS").c_str(), buf));
  };
  F("AMAX", c.action_space_max); F("SMAX", c.state_space_max);
  F("INERTIA", c.inertia); F("RADIUS", c.target_radius);
  F("ALW", c.action_loss_weight); F("SCALE", c.reward_scale);
  F("SHIFT", c.reward_shift);
  F("TERM_ADD", c.term_state_reward * c.reward_scale);
  F("P_STD", c.transition_noise_std); F("R_STD", c.reward_noise_std);
  F("TU1", p.tu_pow[0]); F("TU2", p.tu_pow[1]); F("TU3", p.tu_pow[2]);
  F("TU4", p.tu_pow[3]);
  for (int k = 0; k < MDPP_MAX_DIM; ++k)
    defs.push_back(D(("REL" + std::to_string(k)).c_str(),
                     I(k < c.n_relevant ? c.relevant_indices[k] : 0)));
  if (const char* mb = std::getenv("MDPP_JIT_C_MINBLOCKS"))  // tuning knob
    defs.push_back(std::string("-DMDPP_C_MINBLOCKS=") + mb);
  if (const char* pf = std::getenv("MDPP_JIT_C_PREFETCH"))   // tuning knob
    defs.push_back(std::string("-DMDPP_C_PREFETCH=") + pf);
  void* fn = get_function(ctx, kContinuousEntrySource, "mdpp_jit_continuous", defs);
  std::memcpy(ctx->jit_sig_continuous, sig, sizeof sig);
  ctx->jit_fn_continuous = fn;
  if (!fn) return 0;
  const unsigned grid = (unsigned)((p.st.n_envs + kCBlock - 1) / kCBlock);
  return launch(ctx, fn, grid, kCBlock, 0, stream, &p);
}

int smem_min_steps() {
  static const int v = [] {
    const char* e = std::getenv("MDPP_SMEM_MIN_T");
    return e ? std::atoi(e) : 1;
  }();
  return v;
}

int jit_try_rollout(mdpp_ctx* ctx, RolloutParams& p, int noise_mode,
                    int normal_mode, cudaStream_t stream) {
  ctx->jit_last_used = 0;
  if (!ctx->jit_enabled) return 0;
  if (noise_mode == MDPP_NOISE_REPLAY) { ctx->jit_log = "replay mode"; return 0; }
  const auto& groups = ctx->d_groups_host;
  constexpr int kRingSmemMaxDelay = 16;
  const bool ring_ok = ctx->max_delay <= kRingSmemMaxDelay;
  // (the delay FIFO lives in registers when every group has the same small
  // delay -- MDPP_CFG_RING_REGS in defines_for -- and needs no shared memory)
  bool ring_in_regs = groups[0].delay >= 1 && groups[0].delay <= kMaxRingRegs;
  for (auto& g : groups) ring_in_regs &= g.delay == groups[0].delay;
  const int ring_bytes =
      ring_ok && !ring_in_regs ? ctx->max_delay * kBlock * 8 : 0;
  // staged ziggurat window: 32 steps (16 KB per CTA) unless that costs a CTA per
  // SM below the 7 the register file allows anyway -- then 16 steps (measured
  // on the 1000-group launch: 6 -> 7 CTAs / SM)
  const bool zig = noise_mode == MDPP_NOISE_PHILOX && normal_mode == MDPP_NORMAL_ZIGGURAT;
  int zig_window = 32;
  if (zig) {
    auto ctas = [&](int window) {
      const int per_cta = ring_bytes + ctx->max_group_blob + kZigBytes +
                          zig_stage_bytes(kBlock, window) + 1024 + 256;
      return (228 * 1024) / per_cta;
    };
    if (ctas(32) < 7 && ctas(16) > ctas(32)) zig_window = 16;
    if (const char* w = std::getenv("MDPP_ZIG_WINDOW")) zig_window = std::atoi(w);  // tuning knob
  }
  const int zig_bytes = zig ? kZigBytes + zig_stage_bytes(kBlock, zig_window) : 0;
  if (!ring_ok ||
      ctx->max_group_blob + ring_bytes + zig_bytes > ctx->max_smem_optin - 1024) {
    ctx->jit_log = "tables or delay ring do not fit shared memory";
    return 0;
  }
  const bool fast = p.io.actions && p.io.obs && p.io.reward && p.io.terminated &&
                    p.io.truncated && !p.io.final_obs && !p.st.history;
  // everything the -D list depends on besides the (versioned) group tables
  const long long sig[10] = {ctx->d_groups_version, noise_mode, normal_mode, fast,
                             (long long)p.st.n_envs, p.autoreset, p.horizon, p.irr,
                             p.io.obs_dtype,
                             (p.T >= smem_min_steps()) + 2 * (p.T >= zig_window) +
                                 4 * zig_window + 8 * (zig && p.T < 8 * zig_window)};
  // tables staged in shared memory (always, unless MDPP_SMEM_MIN_T says that
  // launches shorter than that read them from global memory: measured slower,
  // the staging overlaps the previous kernel under programmatic launch)
  const bool smem = p.T >= smem_min_steps();
  void* fn = nullptr;
  if (std::memcmp(sig, ctx->jit_sig_discrete, sizeof sig) == 0) {
    fn = ctx->jit_fn_discrete;
  } else {
    int cdf_tpl = groups[0].cdf_log2 <= 6 ? groups[0].cdf_log2 : -1;
    for (auto& g : groups)
      if (g.cdf_log2 != groups[0].cdf_log2) cdf_tpl = -1;
    std::vector<std::string> defs =
        defines_for(groups, p, noise_mode, normal_mode, fast, true, cdf_tpl, smem,
                    p.T >= zig_window);
    defs.push_back("-DMDPP_ZIG_WINDOW=" + std::to_string(zig_window));
    // launches of a few windows: the last window is drawn only as far as it is
    // read (C5 at 100 steps per launch: +1.6 %); long launches keep the
    // compile-time trip count (the headline loses 9 % without it)
    if (zig && p.T < 8 * zig_window) defs.push_back("-DMDPP_ZIG_FILL_DYN");
    if (const char* ch = std::getenv("MDPP_JIT_CHUNK"))  // tuning knob (4/8/16)
      defs.push_back(std::string("-DMDPP_JIT_CHUNK=") + ch);
    else if (groups.size() > 1)
      // multi-group builds keep L / delay / noise flags run-time: a chunk of 4
      // halves the hot loop's code (ncu: no_instruction 2.4 stalls per issue
      // with chunks of 8 and fp64 normals); measured +6 % (fast) / +9 % (fp64)
      defs.push_back("-DMDPP_JIT_CHUNK=4");
    if (const char* mb = std::getenv("MDPP_JIT_MINBLOCKS"))  // tuning knob
      defs.push_back(std::string("-DMDPP_JIT_MINBLOCKS=") + mb);
    if (const char* ex = std::getenv("MDPP_JIT_EXTRA")) {  // experiments: "-DX=1 -DY"
      std::string all(ex), tok;
      for (size_t i = 0; i <= all.size(); ++i) {
        if (i == all.size() || all[i] == ' ') {
          if (!tok.empty()) defs.push_back(tok);
          tok.clear();
        } else {
          tok += all[i];
        }
      }
    }
    fn = get_function(ctx, kEntrySource, "mdpp_jit_rollout", defs);
    std::memcpy(ctx->jit_sig_discrete, sig, sizeof sig);
    ctx->jit_fn_discrete = fn;
  }
  if (!fn) return 0;
  p.ring_smem_bytes = ring_bytes;
  p.tab_smem_bytes = smem ? ctx->max_group_blob : 0;
  return launch(ctx, fn, (unsigned)ctx->d_set.n_ctas, kBlock,
                ring_bytes + (smem ? ctx->max_group_blob + zig_bytes : 0), stream, &p,
                /*pdl=*/p.T < kChunk);
}

void jit_release(mdpp_ctx* ctx) {
  Api& a = api();
  if (a.ok)
    for (void* m : ctx->jit_modules) a.ModuleUnload((CUmodule)m);
  ctx->jit_modules.clear();
  ctx->jit_functions.clear();
}

}  // namespace mdpp

// Compile (not load) the specialisation of the BASELINE config #2 shape with
// NVRTC only -- usable without a GPU; returns 0 on success and copies the
// compiler log into `log` (may be NULL).
extern "C" int mdpp_jit_selftest(char* log, int log_bytes) {
  using namespace mdpp;
  mdpp_ctx tmp;
  DiscreteGroupDev g;
  std::memset(&g, 0, sizeof g);
  g.S = 8; g.A = 8; g.L = 3; g.delay = 2; g.every_n = 1; g.key_bits = 3;
  g.key_mask = 511; g.has_pnoise = 1; g.has_rnoise = 1; g.cdf_log2 = 3;
  g.has_guide = 1; g.r_std = 0.25; g.scale = 1.0; g.p_is_u8 = 1;
  g.pn_T = 429496730ull; g.pn_M = 2348810237u; g.pn_shift = 25;
  RolloutParams p;
  std::memset(&p, 0, sizeof p);
  p.st.n_envs = 65536; p.autoreset = 1; p.horizon = 100;
  std::vector<std::string> defs = defines_for(
      std::vector<DiscreteGroupDev>{g}, p, MDPP_NOISE_PHILOX, MDPP_NORMAL_FAST,
      true, true, 3);
  // compile() loads the module too, which needs a driver: stop after NVRTC
  void* rtc = dlopen("libnvrtc.so.12", RTLD_NOW | RTLD_GLOBAL);
  if (!rtc) rtc = dlopen("/usr/local/cuda/lib64/libnvrtc.so.12", RTLD_NOW | RTLD_GLOBAL);
  std::string msg;
  int rc = -1;
  if (!rtc) {
    msg = "libnvrtc not found";
  } else {
    auto Create = (nvrtcResult(*)(nvrtcProgram*, const char*, const char*, int,
                                  const char* const*, const char* const*))
        dlsym(rtc, "nvrtcCreateProgram");
    auto Compile = (nvrtcResult(*)(nvrtcProgram, int, const char* const*))
        dlsym(rtc, "nvrtcCompileProgram");
    auto LogSize = (nvrtcResult(*)(nvrtcProgram, size_t*))
        dlsym(rtc, "nvrtcGetProgramLogSize");
    auto Log = (nvrtcResult(*)(nvrtcProgram, char*)) dlsym(rtc, "nvrtcGetProgramLog");
    auto Destroy = (nvrtcResult(*)(nvrtcProgram*)) dlsym(rtc, "nvrtcDestroyProgram");
    // BASELINE config #3 shape for the continuous kernel
    std::vector<std::string> cdefs = {
        "-DMDPP_JIT", "-DMDPP_C_REAL=float", "-DMDPP_C_NOISE=2", "-DMDPP_C_DIM=6",
        "-DMDPP_C_ORDER=2", "-DMDPP_C_NREL=2", "-DMDPP_C_DELAY=0",
        "-DMDPP_C_EVERY_N=1", "-DMDPP_C_DENSE=true", "-DMDPP_C_PNOISE=false",
        "-DMDPP_C_RNOISE=false", "-DMDPP_C_IMAGE=false", "-DMDPP_C_TARGET64=false",
        "-DMDPP_C_NORMAL=0", "-DMDPP_C_IMODE=0", "-DMDPP_C_LINE=false", "-DMDPP_C_SEQ=1", "-DMDPP_C_NBOX=0", "-DMDPP_C_HORIZON=100", "-DMDPP_C_AUTORESET=true",
        "-DMDPP_C_N_ENVS=1048576ll", "-DMDPP_C_FAST=true",
        "-DMDPP_C_REL0=0", "-DMDPP_C_REL1=1"};
    for (int k = 2; k < MDPP_MAX_DIM; ++k)
      cdefs.push_back("-DMDPP_C_REL" + std::to_string(k) + "=0");
    for (const char* k : {"AMAX", "SMAX", "INERTIA", "RADIUS", "ALW", "SCALE",
                          "SHIFT", "TERM_ADD", "P_STD", "R_STD", "TU1", "TU2",
                          "TU3", "TU4"})
      cdefs.push_back(std::string("-DMDPP_C_") + k + "_BITS=0x3ff0000000000000ll");
    rc = 0;
    for (int which = 0; which < 2 && rc == 0; ++which) {
      nvrtcProgram prog = nullptr;
      Create(&prog, which == 1 ? kContinuousEntrySource : kEntrySource,
             "mdpp_jit_entry.cu", kNumHeaders, kHeaderSources, kHeaderNames);
      std::vector<std::string> opts = {"--gpu-architecture=sm_100a",
                                       "-std=c++17", "-lineinfo"};
      auto& dd = which == 1 ? cdefs : defs;
      opts.insert(opts.end(), dd.begin(), dd.end());
      std::vector<const char*> copts;
      for (auto& o : opts) copts.push_back(o.c_str());
      rc = Compile(prog, (int)copts.size(), copts.data());
      size_t n = 0;
      LogSize(prog, &n);
      std::string part(n, '\0');
      if (n) Log(prog, &part[0]);
      msg += part;
      Destroy(&prog);
    }
  }
  if (log && log_bytes > 0) {
    std::strncpy(log, msg.c_str(), log_bytes - 1);
    log[log_bytes - 1] = '\0';
  }
  return rc;
}

extern "C" int mdpp_jit_last_used(const mdpp_ctx* ctx) {
  return ctx ? ctx->jit_last_used : 0;
}

extern "C" const char* mdpp_jit_log(const mdpp_ctx* ctx) {
  return ctx ? ctx->jit_log.c_str() : "";
}

extern "C" void mdpp_set_jit(mdpp_ctx* ctx, int enabled) {
  if (ctx) ctx->jit_enabled = enabled;
}
