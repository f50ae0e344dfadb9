"""Device time of the grouped image renderers against the single-config ones.

    python tools/time_render_groups.py [N] [K] [rounds]

N images of 100 x 100 (default 16 384, the C4 shape).  Discrete transforms
none / shift / shift+scale+rotate; arms: the single-config renderer, the
grouped renderer with G = 1, 64 and 1000 identical configurations, and with
6 distinct ones.  The same for the continuous renderer at 2-D and 4-D.  Each
arm is K launches (default 200) captured in one CUDA graph, timed with CUDA
events after a warm-up replay; the arms alternate over `rounds` rounds and
the median per launch is reported, with the grouped / single ratio and the
card's name and power limit.
"""
import ctypes as C
import statistics
import subprocess
import sys
import warnings

import numpy as np
import torch

sys.path.insert(0, ".")
from mdp_playground_b200 import VectorRLToyEnv, _lib  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
K = int(sys.argv[2]) if len(sys.argv) > 2 else 200
ROUNDS = int(sys.argv[3]) if len(sys.argv) > 3 else 7
LIB = _lib.load()

DISCRETE = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
                state_space_size=8, action_space_size=8, sequence_length=1, delay=0,
                reward_density=0.25, terminal_state_density=0.25,
                image_representations=True, image_width=100, image_height=100)
CONTINUOUS = dict(seed=0, state_space_type="continuous",
                  action_space_type="continuous", transition_dynamics_order=1,
                  target_point=[3.0, -3.0], target_radius=0.05, state_space_max=5.0,
                  action_space_max=1.0, reward_function="move_to_a_point",
                  image_representations=True, image_width=100, image_height=100,
                  terminal_states=[[1.0, 1.0], [-2.0, 0.5]], term_state_edge=1.5)
TRANSFORMS = {
    "none": [dict(image_transforms="none", state_space_size=8 + k) for k in range(6)],
    "shift": [dict(image_transforms="shift", image_sh_quant=1 + k) for k in range(6)],
    "shift,scale,rotate": [dict(image_transforms="shift,scale,rotate",
                                image_sh_quant=1 + k % 2, image_ro_quant=1 + k,
                                image_scale_range=(0.5 + 0.05 * k, 1.5))
                           for k in range(6)],
}


def make_env(n, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return VectorRLToyEnv(n, **kw)


def new_ctx():
    ctx = C.c_void_p()
    _lib.check(LIB, None, LIB.mdpp_create(torch.cuda.current_device(), C.byref(ctx)))
    return ctx


def even_layout(G):
    sizes = [N // G + (1 if g < N % G else 0) for g in range(G)]
    begin = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    return [(int(b), int(s)) for b, s in zip(begin, sizes)]


def capture(launch):
    """K launches of `launch(stream)` in one CUDA graph."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch(C.c_void_p(side.cuda_stream))
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for _ in range(K):
            launch(s)
    g.replay()  # warm-up
    torch.cuda.synchronize()
    return g


def time_graph(g):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / K  # us per launch


def discrete_arms(tr):
    """(name, graph) of every arm of one transform family."""
    cfgs = TRANSFORMS[tr]
    env = make_env(N, philox_seed=1, **{**DISCRETE, **cfgs[0]})
    st = torch.randint(0, 8, (N,), device="cuda")
    out = torch.empty((N, 100, 100), dtype=torch.uint8, device="cuda")
    prm = torch.empty((N, 5), dtype=torch.int32, device="cuda")
    opts = _lib.StepOpts()
    opts.seed = 1
    keep = [env, st, out, prm, opts]

    def single(s):
        _lib.check(LIB, env._ctx, LIB.mdpp_render_discrete(
            env._ctx, C.byref(env._img_cfg), st.data_ptr(), None, prm.data_ptr(),
            out.data_ptr(), N, N, 3, C.byref(opts), s))

    def grouped(ctx):
        def launch(s):
            _lib.check(LIB, ctx, LIB.mdpp_render_discrete_groups(
                ctx, st.data_ptr(), None, prm.data_ptr(), out.data_ptr(), N, N, 3,
                C.byref(opts), s))
        return launch
    arms = [("single", capture(single))]
    for G in (1, 64, 1000):
        ctx = new_ctx()
        groups = (_lib.ImageDiscreteGroup * G)()
        for g, (b, n) in zip(groups, even_layout(G)):
            g.tb = env._img_cfg
            g.env_begin, g.env_count, g.global_id_base = b, n, b
        _lib.check(LIB, ctx, LIB.mdpp_set_image_discrete_groups(ctx, groups, G))
        keep.append(ctx)
        arms.append((f"grouped G={G}", capture(grouped(ctx))))
    # ("none": the 6 configurations differ in the state count only, and
    # share one table set)
    het = make_env(N, philox_seed=1, config_groups=cfgs, **DISCRETE)
    keep.append(het)
    arms.append((f"grouped 6 distinct ({len(het.image_table_sets)} table sets)",
                 capture(grouped(het._ctx))))
    return arms, keep


def continuous_arms(D):
    base = dict(CONTINUOUS, state_space_dim=D, action_space_dim=D,
                relevant_indices=[0, 1], irrelevant_features=D == 4)
    env = make_env(N, philox_seed=1, **base)
    st = (torch.rand((N, D), device="cuda") * 10 - 5).contiguous()
    out = torch.empty((N,) + env.obs_shape, dtype=torch.uint8, device="cuda")
    keep = [env, st, out]

    def single(s):
        _lib.check(LIB, env._ctx, LIB.mdpp_render_continuous(
            env._ctx, C.byref(env._img_cfg), st.data_ptr(), out.data_ptr(), N, s))

    def grouped(ctx):
        def launch(s):
            _lib.check(LIB, ctx, LIB.mdpp_render_continuous_groups(
                ctx, st.data_ptr(), out.data_ptr(), N, N, s))
        return launch
    arms = [("single", capture(single))]
    for G in (1, 64, 1000):
        ctx = new_ctx()
        groups = (_lib.ImageContinuousGroup * G)()
        for g, (b, n) in zip(groups, even_layout(G)):
            g.cfg = env._img_cfg
            g.env_begin, g.env_count = b, n
        _lib.check(LIB, ctx, LIB.mdpp_set_image_continuous_groups(ctx, groups, G))
        keep.append(ctx)
        arms.append((f"grouped G={G}", capture(grouped(ctx))))
    cells = [dict(target_point=[-3.0 + k, 1.0], state_space_max=5.0 + k,
                  terminal_states=[[0.5 * k, -1.0]]) for k in range(6)]
    het = make_env(N, philox_seed=1, config_groups=cells, **base)
    keep.append(het)
    arms.append(("grouped 6 distinct", capture(grouped(het._ctx))))
    return arms, keep


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    name, power = card()
    print(f"# {name}, power limit {power}; N = {N} images, {K} launches per graph, "
          f"median of {ROUNDS} alternating rounds", flush=True)
    families = [(f"discrete[{tr}]", *discrete_arms(tr)) for tr in TRANSFORMS]
    families += [(f"continuous[{D}-D]", *continuous_arms(D)) for D in (2, 4)]
    times = {(f, a): [] for f, arms, _ in families for a, _ in arms}
    for _ in range(ROUNDS):
        for f, arms, _ in families:
            for a, g in arms:
                times[(f, a)].append(time_graph(g))
    for f, arms, _ in families:
        single = statistics.median(times[(f, "single")])
        for a, _ in arms:
            t = times[(f, a)]
            med = statistics.median(t)
            print(f"{f:28s} {a:36s} {med:8.2f} us/launch  (min {min(t):7.2f}, "
                  f"max {max(t):7.2f})  x{med / single:.3f} of single", flush=True)


if __name__ == "__main__":
    main()
