#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched RLToyEnv step path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N \
        --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1]): discrete toy MDP, 8 states x 8 actions,
sequence_length 3, delay 2, transition_noise 0.1, reward_noise 0.25,
65 536 envs per GPU, horizon 100 with auto-reset, native Philox noise with
the API-default fp64 reward normals (numpy's ziggurat on Philox words).
One bench "step" = one fused rollout launch of --inner (default 1000)
env-steps over all envs of the rank: actions [T,N] int32 are read from HBM,
obs i64 / reward f64 / terminated u8 / truncated u8 [T,N] are written
(22 B per env-step, 1.44 GB per launch: larger than the 126 MB L2, so no
flush is needed between launches).

Prints ONE JSON line (rank 0):
  value / roofline   K launches back to back, device resident (burst)
  sustained          the same launch repeated for >= 2 s, clocks sampled over
                     the whole leg
  parity             sampled rows of the TIMED output buffers recomputed by
                     the CPU oracle from a pre-timing state snapshot
  variants           the same launch with the other normal generators
  e2e                host buffers in, host buffers out (public API)
  step_api           the gym-style step() call itself, eager and graphed
  cpu_baseline       the reference's own RLToyEnv loop on one host core
`--dump-outputs DIR` writes what the last timed launch returned (rank 0) as
DIR/<name>.npy, every step of a fixed, seeded sample of envs, so that two
builds can be compared output for output (the inputs depend on the arguments
only).
`--impl reference` times the reference's RLToyEnv (oracle/_ref, vendored by
oracle/make_ref.py; else the CPU port oracle/scalar_env.py) on all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
ENVS_PER_GPU = 65536
ALGO_BYTES_ROLLOUT = 22   # SURVEY.md 8d (ii): action in + outputs out
ALGO_BYTES_STEP = 58      # SURVEY.md 8d table, config C2 single step
NORMAL_NAMES = {"fp64": "fp64 ziggurat (numpy's Generator.normal algorithm)",
                "boxmuller": "fp64 Box-Muller", "fast": "fp32 SFU Box-Muller"}
DUMP_BYTES = 48 << 20     # cap of what --dump-outputs writes


def workload_config():
    return dict(seed=0, state_space_type="discrete",
                action_space_type="discrete", state_space_size=8,
                action_space_size=8, sequence_length=3, delay=2,
                transition_noise=0.1, reward_noise=0.25, reward_density=0.25,
                terminal_state_density=0.25, generate_random_mdp=True,
                reward_every_n_steps=True)


WORKLOAD_NAME = ("discrete toy (dqn_p_r_noises/dqn_seq_del shape): 8 states, "
                 "8 actions, sequence_length=3, delay=2, transition_noise=0.1, "
                 "reward_noise=0.25, 65536 envs per GPU, horizon 100 auto-reset")

def bench_config(n_envs, inner, normal):
    """The `config` object of the JSON line -- identical for both arms."""
    return {"workload": WORKLOAD_NAME, "envs_per_gpu": n_envs,
            "env_steps_per_launch": inner,
            "noise": "transition_noise 0.1 + reward_noise N(0, 0.25) every step; "
                     "GPU arm: philox4x32-10, reward normals " + NORMAL_NAMES[normal]
                     + (" (API default)" if normal == "fp64" else "")
                     + "; reference arm: numpy PCG64",
            "autoreset": "on terminated or after 100 steps",
            "l2_policy": f"inputs+outputs {inner * n_envs * 22 / 1e6:.0f} MB per "
                         "launch > 126 MB L2 (no flush needed)"}


C1_CONFIG = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
                 state_space_size=8, action_space_size=8, reward_density=0.25,
                 terminal_state_density=0.25, sequence_length=1, delay=0)
C3_CONFIG = dict(seed=0, state_space_type="continuous", state_space_dim=6,
                 relevant_indices=[0, 1], irrelevant_features=True,
                 transition_dynamics_order=2, inertia=1.0, time_unit=0.5,
                 target_radius=0.05, target_point=[0.0, 0.0],
                 state_space_max=10.0, action_space_max=1.0)
C4_CONFIG = dict(C1_CONFIG, image_representations=True, image_transforms="shift",
                 image_sh_quant=4, image_width=100, image_height=100)


# --------------------------------------------------------------------------
# CPU legs: the reference's own loop (BASELINE.md section 3)
# --------------------------------------------------------------------------
def reference_kind():
    from oracle import ref_loader
    return "reference" if ref_loader.reference_available() else "port"


def _make_cpu_env(config, kind):
    if kind == "reference":
        from oracle.ref_loader import make_reference_env
        return make_reference_env(config)
    from oracle.scalar_env import ScalarRLToyEnv
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ScalarRLToyEnv(**config)


def _cpu_loop(n_steps, seed=0, horizon=100, config=None, kind="port",
              max_seconds=None):
    """for t: env.step(a_t); reset on done or every `horizon` steps.  Returns
    (steps done, seconds)."""
    import numpy as np
    cfg = dict(workload_config() if config is None else config, seed=seed)
    env = _make_cpu_env(cfg, kind)
    rng = np.random.default_rng(0xC0FFEE + seed)
    if cfg["state_space_type"] == "continuous":
        acts = rng.uniform(-1, 1, size=(n_steps, cfg["state_space_dim"])).astype(
            np.float32)
    else:
        acts = rng.integers(0, 8, size=n_steps).tolist()
    t0 = time.perf_counter()
    since = done_steps = 0
    for a in acts:
        _, _, done, _, _ = env.step(a)
        since += 1
        done_steps += 1
        if done or since == horizon:
            env.reset()
            since = 0
        if max_seconds and (done_steps & 255) == 0 and \
                time.perf_counter() - t0 > max_seconds:
            break
    return done_steps, time.perf_counter() - t0


def _cpu_worker(args):
    n_steps, seed, kind = args
    return _cpu_loop(n_steps, seed, kind=kind)


def cpu_throughput(n_steps, procs, kind):
    """Aggregate steps/s of `procs` independent scalar envs (1 = in-process)."""
    if procs == 1:
        n, dt = _cpu_loop(n_steps, kind=kind)
        return n / dt
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(n_steps, s, kind) for s in range(procs)])
        wall = time.perf_counter() - t0
    return procs * n_steps / wall


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind = reference_kind()
    cores = len(os.sched_getaffinity(0))
    per_proc = args.ref_sample if kind == "port" else max(args.ref_sample // 8, 2000)
    _cpu_loop(2000, kind=kind)  # import + warm caches
    for _ in range(args.warmup):
        cpu_throughput(max(per_proc // 10, 1000), cores, kind)
    t0 = time.perf_counter()
    vals = [cpu_throughput(per_proc, cores, kind) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    value = sum(vals) / len(vals)
    what = ("the UNMODIFIED reference RLToyEnv (oracle/_ref, gymnasium stand-in)"
            if kind == "reference" else
            "the scalar CPU port of the reference loop (oracle/scalar_env.py)")
    sample = (f"{cores} processes x {per_proc} env-steps of {what} per bench "
              f"step, reset on done or every 100 steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64",
        "data": "synthetic",
        "config": bench_config(args.envs, args.inner, args.normal),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores,
                         "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML,
    every 2 ms; nvidia-smi polling is too coarse for a 20-50 ms region)."""
    HW_SLOWDOWN, SW_POWER_CAP = 0x8, 0x4
    HW_THERMAL, SW_THERMAL = 0x40, 0x20

    def __init__(self, index, period=0.002):
        self.index, self.sm, self.reasons = index, [], 0
        self.power = []
        self.period = period
        self.stop_flag, self.thread, self.max_mhz = False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(
                self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.reasons |= nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1e3)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        sm = sorted(self.sm)
        names = [(self.HW_SLOWDOWN, "hw_slowdown"),
                 (self.HW_THERMAL, "hw_thermal_slowdown"),
                 (self.SW_THERMAL, "sw_thermal_slowdown"),
                 (self.SW_POWER_CAP, "sw_power_cap")]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": self.max_mhz,
                "reasons": [n for bit, n in names if self.reasons & bit],
                "samples": len(sm),
                "power_w_max": max(self.power) if self.power else None}


# --------------------------------------------------------------------------
def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(n_envs, n_steps, normal):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant
    kernel, from the committed `ncu --set full` capture (profiles/), when the
    launch shape matches the captured one; else null."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            k = json.load(f)["mdpp_jit_rollout"][normal]
        if k["envs"] == n_envs and k["steps_per_launch"] == n_steps:
            return k["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def bind_to_gpu_numa(torch, index):
    """Pin this process (and the pinned buffers it allocates from now on) to
    the CPUs of the GPU's NUMA node.  Returns a description for the JSON."""
    info = {"numa_node": None, "cpus": len(os.sched_getaffinity(0))}
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        info["pci"] = bdf
        info["numa_node"] = node
        if node >= 0:
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                a, _, b = part.partition("-")
                cpus |= set(range(int(a), int(b or a) + 1))
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                info["cpus"] = len(cpus)
    except Exception as e:  # not fatal: the probe below records what we got
        info["error"] = str(e)[:80]
    return info


def _time_launches(torch, fn, n, barrier, max_over_ranks):
    for _ in range(3):
        fn()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    barrier()
    return max_over_ranks(e0.elapsed_time(e1)) / n


def cpu_reference_leg(config, seconds=2.5):
    """steps/s of the reference's own loop for one of the other configs (one
    process, bounded by wall time)."""
    kind = reference_kind()
    try:
        _cpu_loop(200, config=config, kind=kind)
        n, dt = _cpu_loop(1 << 22, config=config, kind=kind, max_seconds=seconds)
        return {"value": n / dt, "unit": UNIT, "cores": 1, "kind": kind,
                "sample": f"{n} env-steps in {dt:.1f} s"}
    except Exception as e:
        return {"error": str(e)[:120], "kind": kind}


def other_configs(torch, Env, dev, rank, world, barrier, max_over_ranks, peak,
                  with_cpu):
    """The other BASELINE.json shapes, device-resident, one line each:
    env-steps/s (all ranks) and fraction of the HBM roofline with the
    algorithmic bytes of SURVEY.md 8d."""
    import numpy as np
    res = {}
    base = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
                state_space_size=8, action_space_size=8, reward_density=0.25,
                terminal_state_density=0.25)

    def line(name, n_envs, steps_per_launch, ms, bytes_per_step, note):
        sps = world * n_envs * steps_per_launch / (ms * 1e-3)
        res[name] = {"value": sps, "unit": UNIT, "envs_per_gpu": n_envs,
                     "env_steps_per_launch": steps_per_launch,
                     "ms_per_launch": ms,
                     "algorithmic_bytes_per_env_step": bytes_per_step,
                     "roofline_frac": sps / world * bytes_per_step / 1e9 / peak,
                     "what": note}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        # C1: seq 1, delay 0, no noise
        N, T = 65536, 1000
        env = Env(N, device=dev, autoreset=True, horizon=100,
                  env_id_offset=rank * N, sequence_length=1, delay=0, **base)
        acts = torch.randint(0, 8, (T, N), dtype=torch.int32, device=dev)
        out = env.rollout(T, actions=acts, want_final_obs=False)
        ms = _time_launches(torch, lambda: env.rollout(T, actions=acts, out=out),
                            10, barrier, max_over_ranks)
        line("C1_discrete_seq1_rollout", N, T, ms, 22,
             "fused rollout, noise off")
        if with_cpu:
            res["C1_discrete_seq1_rollout"]["cpu_reference"] = cpu_reference_leg(C1_CONFIG)
        del env, acts, out
        # N2 (SURVEY.md 8f): discrete irrelevant_features, dqn_irr_dims.py
        # shape; rows (relevant, irrelevant): 8 B actions in, 16 B obs out
        env = Env(N, device=dev, autoreset=True, horizon=100,
                  env_id_offset=rank * N, sequence_length=1, delay=0,
                  irrelevant_features=True, transition_noise=0.1,
                  **dict(base, state_space_size=[8, 8], action_space_size=[8, 8]))
        acts = torch.randint(0, 8, (T, N, 2), dtype=torch.int32, device=dev)
        out = env.rollout(T, actions=acts, want_final_obs=False)
        ms = _time_launches(torch, lambda: env.rollout(T, actions=acts, out=out),
                            10, barrier, max_over_ranks)
        line("N2_discrete_irrelevant_features_rollout", N, T, ms, 34,
             "fused rollout, two sub-MDPs per env, transition noise 0.1")
        del env, acts, out
        # N1 (SURVEY.md 8f): grid env, tests/test_mdp_playground.py:1057 shape;
        # int64 rows: 16 B action in, 16 B cell + 8 B reward + 2 B flags out
        Ng, Tg = 1 << 20, 100
        env = Env(Ng, device=dev, autoreset=True, horizon=100,
                  env_id_offset=rank * Ng, seed=0, state_space_type="grid",
                  grid_shape=(8, 8), delay=0, sequence_length=1,
                  reward_function="move_to_a_point", target_point=[5, 5],
                  make_denser=True, transition_noise=0.1)
        acts = torch.zeros((Tg, Ng, 2), dtype=torch.int64, device=dev)
        acts[..., 0] = torch.randint(-1, 2, (Tg, Ng), device=dev)
        out = env.rollout(Tg, actions=acts, want_final_obs=False)
        ms = _time_launches(torch, lambda: env.rollout(Tg, actions=acts, out=out),
                            5, barrier, max_over_ranks)
        line("N1_grid_rollout", Ng, Tg, ms, 42,
             "fused rollout, 8x8 grid, dense reward, transition noise 0.1")
        del env, acts, out
        # N3: GymEnvWrapper's post-processing tail for EXTERNAL vector envs
        # (gym_env_wrapper.py:350-439, :523-618), one call pair per step
        from mdp_playground_b200 import VectorGymEnvTail
        Nt, side, pad = 8192, 84, 20
        tail = VectorGymEnvTail(Nt, device=dev, seed=0, env_id_offset=rank * Nt,
                                n_actions=18, state_space_type="discrete", delay=2,
                                transition_noise=0.1, reward_noise=0.5, reward_scale=2.0,
                                image_transforms="shift", image_side=side,
                                image_padding=pad, image_sh_quant=2)
        a = torch.randint(0, 18, (Nt,), dtype=torch.int32, device=dev)
        frames = torch.randint(0, 256, (Nt, side, side, 3), dtype=torch.uint8, device=dev)
        r = torch.rand(Nt, dtype=torch.float64, device=dev)
        d = torch.zeros(Nt, dtype=torch.uint8, device=dev)

        def atari_like():
            tail.actions(a)
            return tail.post(frames, r, d)
        ms = _time_launches(torch, atari_like, 10, barrier, max_over_ranks)
        tot = side + 2 * pad
        line("N3_wrapper_tail[atari-like: 84x84x3 frames, shift into 124x124x3]", Nt, 1, ms,
             8 + 17 + side * side * 3 + tot * tot * 3,
             "VectorGymEnvTail.actions + .post per step: action noise, reward delay 2 "
             "+ noise + scale, padded canvas with a random quantised shift")
        del tail, frames
        Nm = 1 << 20
        tail = VectorGymEnvTail(Nm, device=dev, seed=0, env_id_offset=rank * Nm,
                                obs_dim=17, state_space_type="continuous", delay=1,
                                transition_noise=0.05, reward_noise=0.1)
        obs = torch.rand((Nm, 17), device=dev)
        r = torch.rand(Nm, dtype=torch.float64, device=dev)
        d = torch.zeros(Nm, dtype=torch.uint8, device=dev)
        ms = _time_launches(torch, lambda: tail.post(obs, r, d), 20, barrier,
                            max_over_ranks)
        line("N3_wrapper_tail[mujoco-like: 17-dim fp32 observations]", Nm, 1, ms,
             17 * 4 * 2 + 17 + 16,
             "VectorGymEnvTail.post per step: observation noise, reward delay 1 + noise "
             "(bytes: obs in + out, reward in + out, done, FIFO slot read + write); "
             "fp64 Box-Muller normals (18 per env-step)")
        del tail
        tail = VectorGymEnvTail(Nm, device=dev, seed=0, env_id_offset=rank * Nm,
                                obs_dim=17, state_space_type="continuous", delay=1,
                                transition_noise=0.05, reward_noise=0.1,
                                normal_precision="fast")
        ms = _time_launches(torch, lambda: tail.post(obs, r, d), 20, barrier,
                            max_over_ranks)
        line("N3_wrapper_tail[mujoco-like, fast normals]", Nm, 1, ms, 17 * 4 * 2 + 17 + 16,
             "the same with normal_precision='fast' (fp32 SFU Box-Muller)")
        del tail, obs, r, d
        # C3: continuous move_to_a_point, 1M envs
        N, T = 1 << 20, 100
        env = Env(N, device=dev, autoreset=True, horizon=100,
                  env_id_offset=rank * N, **C3_CONFIG)
        acts = torch.rand((T, N, 6), device=dev) * 2 - 1
        out = env.rollout(T, actions=acts, want_final_obs=False)
        ms = _time_launches(torch, lambda: env.rollout(T, actions=acts, out=out),
                            5, barrier, max_over_ranks)
        line("C3_continuous_rollout", N, T, ms, 54, "fused rollout, fp32")
        if with_cpu:
            res["C3_continuous_rollout"]["cpu_reference"] = cpu_reference_leg(C3_CONFIG)
        a1, o1 = acts[:1], {k: v[:1] for k, v in out.items()}
        ms = _time_launches(torch, lambda: env.rollout(1, actions=a1, out=o1),
                            50, barrier, max_over_ranks)
        line("C3_continuous_single_step", N, 1, ms, 256,
             "rollout(1) into caller-owned buffers: one launch per step")
        gstep = env.make_graphed_step()
        gstep.actions.copy_(a1[0])  # actions resident in the graph's input buffer
        ms = _time_launches(torch, lambda: gstep(gstep.actions), 50, barrier,
                            max_over_ranks)
        line("C3_continuous_single_step_cuda_graph", N, 1, ms, 256,
             "step() replayed from a CUDA graph")
        del gstep
        del env, acts, out
        # C4: 100x100 image observations, 16384 envs
        N = 16384
        for tr, extra in (("shift", dict(image_sh_quant=4)),
                          ("shift,scale,rotate", dict(image_sh_quant=1,
                                                      image_ro_quant=1,
                                                      image_scale_range=(0.5, 1.5)))):
            env = Env(N, device=dev, autoreset=True, horizon=100,
                      env_id_offset=rank * N, sequence_length=1, delay=0,
                      image_representations=True, image_transforms=tr,
                      image_width=100, image_height=100, **extra, **base)
            a = torch.randint(0, 8, (N,), dtype=torch.int32, device=dev)
            ms = _time_launches(torch, lambda: env.step(a), 30, barrier,
                                max_over_ranks)
            line(f"C4_image_step[{tr}]", N, 1, ms, 10034,
                 "step() + render, two launches per step")
            if with_cpu and tr == "shift":
                res[f"C4_image_step[{tr}]"]["cpu_reference"] = cpu_reference_leg(C4_CONFIG)
            gstep = env.make_graphed_step()
            gstep.actions.copy_(a)  # (resident in the graph's input buffer)
            ms = _time_launches(torch, lambda: gstep(gstep.actions), 30, barrier,
                                max_over_ranks)
            line(f"C4_image_step_cuda_graph[{tr}]", N, 1, ms, 10034,
                 "step() + render replayed from a CUDA graph")
            # fused form (SURVEY.md 8d ii): T steps in one rollout launch, all
            # T x N observations rendered by one launch
            Tr = 8
            acts = torch.randint(0, 8, (Tr, N), dtype=torch.int32, device=dev)
            out = env.rollout(Tr, actions=acts, want_final_obs=False)

            def rollout_and_render():
                env.rollout(Tr, actions=acts, out=out)
                return env.render_observation(out["obs"],
                                              step_index=env._step_index - Tr)
            ms = _time_launches(torch, rollout_and_render, 10, barrier,
                                max_over_ranks)
            line(f"C4_image_rollout[{tr}]", N, Tr, ms, 10014,
                 "rollout(8) + one render launch for the 8 x N observations")
            del env, gstep, acts, out
        # C5: 1000-cell heterogeneous grid, 1M envs per GPU
        cfgs = [dict(base, delay=d, sequence_length=L, transition_noise=pn,
                     reward_noise=rn, make_denser=md, reward_every_n_steps=True)
                for d in (0, 1, 2, 4, 8) for L in (1, 2, 3, 4)
                for pn in (0, 0.01, 0.02, 0.1, 0.25) for rn in (0, 1, 5, 10, 25)
                for md in (False, True)]
        N = 1 << 20
        # 100 steps per launch (round 1's shape, 2.3 GB of I/O buffers) and the
        # 1000 steps per launch SURVEY.md 8d specifies (23 GB: prologue and the
        # last partial ziggurat window amortised over ten times the steps)
        for T in (100, 1000):
            for prec in ("fp64", "fast"):
                env = Env(N, device=dev, autoreset=True, horizon=100, config_groups=cfgs,
                          shard=(rank, world), normal_precision=prec)
                acts = torch.randint(0, 8, (T, N), dtype=torch.int32, device=dev)
                out = env.rollout(T, actions=acts, want_final_obs=False)
                ms = _time_launches(torch, lambda: env.rollout(T, actions=acts, out=out),
                                    5, barrier, max_over_ranks)
                name = "C5_heterogeneous_1000_groups_rollout" + (
                    "" if prec == "fp64" else "[fast normals]") + (
                    "" if T == 100 else "[1000 steps per launch]")
                line(name, N, T, ms, 22,
                     "fused rollout, one multi-group launch (scalars shared by all "
                     "groups specialised); reward normals: " + NORMAL_NAMES[prec])
                if prec == "fp64" and T == 100:
                    s5 = env.episode_stats(reduce=True)
                    res[name]["stats_allreduce"] = {
                        "groups": len(cfgs),
                        "episode_len_mean_min_max": [float(np.min(s5["episode_len_mean"])),
                                                     float(np.max(s5["episode_len_mean"]))]}
                del env, acts, out
                torch.cuda.empty_cache()
    return res


def parity_check(env, snap, actions, out_rows, idx, n_launches, T, rank, N):
    """Recompute the sampled envs `idx` with the CPU oracle from the state
    snapshot taken before the timed region, through all `n_launches` timed
    launches, and compare the LAST launch with the rows copied out of the timed
    output buffers.  States / flags bit-exact, fp64 rewards 1e-12."""
    import numpy as np
    from oracle.scalar_env import ScalarRLToyEnv
    from oracle.vector_oracle import VectorDiscreteOracle
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        scalar = ScalarRLToyEnv(**workload_config())
    ora = VectorDiscreteOracle(
        scalar, len(idx), autoreset=True, horizon=100, seed=env.philox_seed,
        gids=rank * N + idx, fast_normal=env.normal_precision == "fast",
        normal="boxmuller" if env.normal_precision == "boxmuller" else "ziggurat")
    ora.load_state(snap["cur"][idx], snap["t"][idx], snap["episode"][idx],
                   snap["key"][idx], snap["ring"][:, idx], snap["step_index"], 3)
    a = actions[:, idx]
    t0 = time.perf_counter()
    for _ in range(n_launches):
        want = ora.rollout(T, actions=a)
    ok = all(np.array_equal(out_rows[k], want[k])
             for k in ("obs", "terminated", "truncated"))
    tol = 1e-5 if env.normal_precision == "fast" else 1e-12
    err = float(np.abs(out_rows["reward"] - want["reward"]).max())
    return {"parity_checked": bool(ok and err <= tol),
            "what": f"{len(idx)} sampled envs x {T} steps of the last timed launch "
                    f"(after {n_launches} launches from the snapshot) vs "
                    "oracle/vector_oracle.py: obs / terminated / truncated "
                    f"bit-exact = {bool(ok)}, max |reward error| = {err:.2e} "
                    f"(tolerance {tol:g})",
            "oracle_seconds": round(time.perf_counter() - t0, 1)}


def dump_outputs(path, out):
    """Write the [T, N] arrays of one rollout as path/<name>.npy: obs and
    reward as float64, the flags as float32, restricted to a seeded sample of
    envs (and of steps, should one env's column alone exceed DUMP_BYTES)."""
    import numpy as np
    import torch
    T, N = out["obs"].shape
    per_step = 8 + 8 + 4 + 4
    n_envs = max(1, min(N, DUMP_BYTES // (T * per_step)))
    n_steps = min(T, DUMP_BYTES // (n_envs * per_step))

    def sample(n, k, seed):
        if k >= n:
            return np.arange(n)
        return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
    dev = out["obs"].device
    rows = torch.as_tensor(sample(T, n_steps, 1), device=dev)
    cols = torch.as_tensor(sample(N, n_envs, 0), device=dev)
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        a = v.index_select(0, rows).index_select(1, cols).cpu().numpy()
        dt = np.float64 if k in ("obs", "reward") else np.float32
        np.save(os.path.join(path, k + ".npy"), a.astype(dt))


def run_gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from mdp_playground_b200 import VectorRLToyEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner (and any NCCL_DEBUG output) to the
        # process's stdout from C: keep file descriptor 1 for the ONE JSON
        # line of the bench contract and send everything else to stderr
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa(torch, local_rank)
    N, T = args.envs, args.inner

    def make_env(normal):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            e = VectorRLToyEnv(N, device=dev, autoreset=True, horizon=100,
                               env_id_offset=rank * N, normal_precision=normal,
                               **workload_config())
        e.set_jit(not args.no_jit)
        return e
    env = make_env(args.normal)
    # synthetic actions: Philox, seed 0xC0FFEE + rank (SURVEY.md 8d)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xC0FFEE + rank)
    actions = torch.randint(0, 8, (T, N), dtype=torch.int32, device=dev,
                            generator=gen)
    out = {
        "obs": torch.empty((T, N), dtype=torch.int64, device=dev),
        "reward": torch.empty((T, N), dtype=torch.float64, device=dev),
        "terminated": torch.empty((T, N), dtype=torch.bool, device=dev),
        "truncated": torch.empty((T, N), dtype=torch.bool, device=dev),
    }

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peak, peak_src = measured_peak_gbs()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)

    # ---- device-resident leg: `value` and the roofline --------------------
    for _ in range(args.warmup):
        env.rollout(T, actions=actions, out=out)
    torch.cuda.synchronize(dev)
    # state snapshot for the parity check of the timed buffers (rank 0)
    snap = None
    if rank == 0 and not args.no_parity:
        snap = {"cur": env._cur.cpu().numpy(), "t": env._t.cpu().numpy(),
                "episode": env._episode.cpu().numpy(),
                "key": env._key.cpu().numpy(), "ring": env._ring.cpu().numpy(),
                "step_index": env._step_index}
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    e0.record()
    for _ in range(args.steps):
        env.rollout(T, actions=actions, out=out)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms_total / args.steps
    value = world * N * T * args.steps / (ms_total * 1e-3)
    per_gpu_steps_per_s = N * T / (ms_per_step * 1e-3)
    achieved = per_gpu_steps_per_s * ALGO_BYTES_ROLLOUT / 1e9
    jit_used = env.jit_last_used
    # the legs below reuse `out`: save the last timed launch's outputs first
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    # rows of the timed output buffers, for the oracle comparison below
    parity = None
    if snap is not None:
        budget = 640_000  # oracle env-steps (~20 s of Python)
        n_s = int(min(64, max(8, budget // (args.steps * T))))
        idx = np.unique(np.linspace(0, N - 1, n_s).astype(np.int64))
        sel = torch.as_tensor(idx, device=dev)
        out_rows = {k: v.index_select(1, sel).cpu().numpy() for k, v in out.items()}

    # ---- sustained leg: the same launch for >= args.sustain seconds -------
    sustained = None
    if args.sustain > 0:
        n_sus = max(args.steps, int(args.sustain * 1e3 / ms_per_step) + 1)
        sampler = ClockSampler(local_rank, period=0.01)
        barrier()
        if rank == 0:
            sampler.start()
        e0.record()
        for _ in range(n_sus):
            env.rollout(T, actions=actions, out=out)
        e1.record()
        barrier()
        sus_ms = max_over_ranks(e0.elapsed_time(e1))
        sus_clocks = sampler.stop() if rank == 0 else None
        sus_value = world * N * T * n_sus / (sus_ms * 1e-3)
        sustained = {"value": sus_value, "unit": UNIT, "launches": n_sus,
                     "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus,
                     "roofline_frac": sus_value / world * ALGO_BYTES_ROLLOUT / 1e9 / peak,
                     "clocks": sus_clocks}

    # ---- the same launch with the other normal generators -----------------
    variants = {}
    for normal in ("fp64", "boxmuller", "fast"):
        if normal == args.normal or args.no_variants:
            continue
        ev = make_env(normal)
        ms = _time_launches(torch, lambda: ev.rollout(T, actions=actions, out=out),
                            args.steps, barrier, max_over_ranks)
        sps = world * N * T / (ms * 1e-3)
        variants[normal] = {"reward_normals": NORMAL_NAMES[normal], "value": sps,
                            "unit": UNIT, "ms_per_step": ms,
                            "roofline_frac": sps / world * ALGO_BYTES_ROLLOUT / 1e9 / peak}
        del ev

    # ---- gym-style step() calls (launch-bound; reported, SURVEY 8d) -------
    n_single = 200
    a1 = actions[0]

    def timed(fn, n=n_single):
        for _ in range(10):
            fn()
        barrier()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / n
        sps = world * N / (ms * 1e-3)
        return {"value": sps, "unit": UNIT, "us_per_call": ms * 1e3,
                "roofline_frac": sps / world * ALGO_BYTES_STEP / 1e9 / peak}
    step_api = {"step": dict(timed(lambda: env.step(a1)),
                             what="env.step(actions): the gym-style call itself "
                                  "(rotating pre-marshalled output sets, returns "
                                  "final_obs; step_buffers=2)")}
    a1r = actions[0:1]
    o1 = {k: v[0:1] for k, v in out.items()}
    step_api["rollout_1"] = dict(
        timed(lambda: env.rollout(1, actions=a1r, out=o1)),
        what="env.rollout(1, actions, out=...) into caller-owned buffers")
    gstep = env.make_graphed_step()
    gstep.actions.copy_(actions[0])  # actions resident in the graph's input buffer
    step_api["cuda_graph"] = dict(
        timed(lambda: gstep(gstep.actions)),
        what="step() replayed from a CUDA graph (make_graphed_step)")
    del gstep

    # ---- end-to-end leg: host buffers through the public API --------------
    h_act = torch.empty((T, N), dtype=torch.int32).pin_memory()
    h_act.copy_(actions.cpu())
    h_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory()
             for k, v in out.items()}

    def e2e_step():  # public host-buffer API: pipelined H2D / kernel / D2H
        env.rollout_host(T, h_act, h_out, chunk_steps=50)

    e2e_steps = max(1, min(args.steps, 5))
    e2e_step()
    barrier()
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * N * T * e2e_steps / (e2e_ms * 1e-3)
    h2d = T * N * 4
    d2h = T * N * (8 + 8 + 1 + 1)
    # the same leg with compact observations (dtype_o=uint8: 3-bit states)
    e2e_compact = None
    if hasattr(env, "set_obs_dtype"):
        envc = make_env(args.normal)
        envc.set_obs_dtype(torch.uint8)
        h_out_c = dict(h_out, obs=torch.empty((T, N), dtype=torch.uint8).pin_memory())
        envc.rollout_host(T, h_act, h_out_c, chunk_steps=50)
        barrier()
        e0.record()
        for _ in range(e2e_steps):
            envc.rollout_host(T, h_act, h_out_c, chunk_steps=50)
        e1.record()
        barrier()
        ms_c = max_over_ranks(e0.elapsed_time(e1))
        e2e_compact = {"value": world * N * T * e2e_steps / (ms_c * 1e-3),
                       "unit": UNIT, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": T * N * (1 + 8 + 1 + 1),
                       "what": "dtype_o=uint8 observations (rl_toy_env.py:611-614)"}
        del envc, h_out_c
    # pinned-memory copy bandwidth of every rank AT THE SAME TIME: the ceiling
    # of the host-buffer leg on this box (all ranks share the host's PCIe /
    # memory path)
    probe_bytes = 256 << 20
    hb = torch.empty(probe_bytes, dtype=torch.uint8).pin_memory()
    db = torch.empty(probe_bytes, dtype=torch.uint8, device=dev)
    probe = {}
    s2 = torch.cuda.Stream(dev)
    for name in ("h2d", "d2h", "both"):
        def go():
            if name in ("h2d", "both"):
                db.copy_(hb, non_blocking=True)
            if name == "both":
                with torch.cuda.stream(s2):
                    hb2.copy_(db2, non_blocking=True)
            elif name == "d2h":
                hb.copy_(db, non_blocking=True)
        if name == "both":
            hb2 = torch.empty(probe_bytes, dtype=torch.uint8).pin_memory()
            db2 = torch.empty(probe_bytes, dtype=torch.uint8, device=dev)
        go()
        barrier()
        t0 = time.perf_counter()
        for _ in range(4):
            go()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        gbs = 4 * probe_bytes * (2 if name == "both" else 1) / dt / 1e9
        if world > 1:
            t = torch.tensor([gbs], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            lo = float(t.item())
            t = torch.tensor([gbs], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            probe[name + "_gbs_per_rank_min"] = lo
            probe[name + "_gbs_all_ranks"] = float(t.item())
        else:
            probe[name + "_gbs_per_rank_min"] = gbs
            probe[name + "_gbs_all_ranks"] = gbs
        barrier()
    probe["bytes_per_env_step"] = 22
    probe["e2e_ceiling_env_steps_per_s"] = probe["both_gbs_all_ranks"] * 1e9 / 22
    # the job ends with its slowest rank (max over ranks), and 18 of the 22
    # bytes of an env-step travel device -> host: what the slowest rank's D2H
    # rate allows, all ranks copying at once
    probe["e2e_ceiling_slowest_rank_d2h"] = world * probe["d2h_gbs_per_rank_min"] * 1e9 / 18
    probe["e2e_frac_of_slowest_rank_d2h"] = e2e_value / probe["e2e_ceiling_slowest_rank_d2h"]
    probe["what"] = ("pinned 256 MiB copies, every rank at once; 'both' = H2D and "
                     "D2H on two streams (sum of directions)")
    del hb, db

    # ---- end-of-run episode statistics: ONE all-reduce (NCCL) -------------
    summ = env.episode_stats(reduce=True)
    stats = {"episodes": float(summ["episodes"][0]),
             "transitions": float(summ["transitions"][0]),
             "episode_reward_mean": float(summ["episode_reward_mean"][0]),
             "episode_len_mean": float(summ["episode_len_mean"][0]),
             "noisy_transition_frac": float(summ["noisy_transitions"][0]
                                            / max(summ["transitions"][0], 1))}
    others = None if args.no_other_configs else other_configs(
        torch, VectorRLToyEnv, dev, rank, world, barrier, max_over_ranks, peak,
        with_cpu=(rank == 0 and world == 1 and not args.no_cpu_baseline))

    if rank == 0:
        if snap is not None:
            parity = parity_check(env, snap, actions.cpu().numpy(), out_rows, idx,
                                  args.steps, T, rank, N)
        # ---- CPU baseline: the reference loop, one core, bounded sample ----
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            kind = reference_kind()
            n_cpu = args.cpu_sample if kind == "reference" else 6 * args.cpu_sample
            _cpu_loop(2000, kind=kind)
            v = cpu_throughput(n_cpu, 1, kind)
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
                   "sample": f"{n_cpu} env-steps of "
                             + ("the unmodified reference RLToyEnv (oracle/_ref)"
                                if kind == "reference" else
                                "oracle/scalar_env.py (CPU port of the reference loop)")
                             + ", one process, reset on done or every 100 steps"}
            if kind == "reference":
                _cpu_loop(2000, kind="port")
                cpu["port_value"] = cpu_throughput(6 * args.cpu_sample // 2, 1, "port")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32+f64",
            "data": "synthetic",
            "config": bench_config(N, T, args.normal),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(N, T, args.normal),
                         "peak_source": peak_src,
                         "kernel": "mdpp_jit_rollout" if jit_used
                         else "discrete_rollout_kernel<PHILOX,smem>",
                         "kernel_build": "nvrtc-specialised" if jit_used
                         else "ahead-of-time",
                         "algorithmic_bytes_per_env_step": ALGO_BYTES_ROLLOUT,
                         "env_steps_per_launch": N * T},
            "sustained": sustained,
            "parity": parity,
            "variants": variants,
            "step_api": step_api,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "e2e_compact_obs": e2e_compact,
            "host_copy_probe": probe,
            "numa": numa,
            "gpu_launches": args.steps,
            "clocks": clocks,
            "episode_stats_allreduced": stats,
            "other_configs": others,
        }
        sys.stdout.flush()
        if world > 1:
            os.write(json_fd, (json.dumps(line) + "\n").encode())
        else:
            print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU,
                    help="envs per GPU")
    ap.add_argument("--inner", type=int, default=1000,
                    help="env-steps fused into one launch (one bench step)")
    ap.add_argument("--cpu-sample", type=int, default=50000)
    ap.add_argument("--ref-sample", type=int, default=100000)
    ap.add_argument("--sustain", type=float, default=2.0,
                    help="seconds of the sustained leg (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the extra BASELINE.json shapes (C1/C3/C4/C5)")
    ap.add_argument("--normal", default="fp64", choices=["fp64", "boxmuller", "fast"],
                    help="reward-noise normals: fp64 ziggurat (API default), "
                         "fp64 Box-Muller, or fp32 SFU Box-Muller")
    ap.add_argument("--no-jit", action="store_true",
                    help="use the ahead-of-time kernels instead of the "
                         "NVRTC-specialised one")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed launch (a "
                         "seeded sample of envs, every step) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.gpus > 1 and world == 1:
            # convenience: re-launch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                   "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
            sys.exit(subprocess.call(cmd))
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
