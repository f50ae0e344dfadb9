"""GPU tests of augmented random search in the continuous rollout kernel
(mdpp_continuous_ars*, mdp_playground_b200/ars.py, Sweep.train_continuous)."""
import ctypes as C
import os
import types
import warnings
from collections import OrderedDict

import numpy as np
import pytest
import torch

from tests import ars_oracle as ao

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "fixtures", "ddpg_move_to_a_point_like.py")


def quiet(f, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return f(*a, **k)


def make_env(*a, **k):
    from mdp_playground_b200 import VectorRLToyEnv
    return quiet(VectorRLToyEnv, *a, **k)


def cont(D=2, **kw):
    rel = [0] if D == 1 else [0, 1]
    c = dict(seed=0, state_space_type="continuous", action_space_type="continuous",
             state_space_dim=D, action_space_dim=D, relevant_indices=rel,
             irrelevant_features=D > len(rel), transition_dynamics_order=1,
             inertia=1.0, time_unit=0.5, target_radius=0.05,
             target_point=[0.0] * len(rel), state_space_max=4.0,
             action_space_max=1.0, reward_function="move_to_a_point",
             make_denser=True)
    c.update(kw)
    return c


def np_(t):
    return t.cpu().numpy()


def group_of_env(env):
    return np.repeat(np.arange(env.n_groups), env._group_sizes)


def host_actions(env, ag, obs, noise_std):
    """The section-1 action of every env from the state it last saw."""
    theta, delta = np_(ag.theta), np_(ag.perturbations())
    g = group_of_env(env)
    w = ao.env_weights(np.zeros_like(theta[0]), delta, 0.0)  # (shape only)
    for i in range(0, env.num_envs, 2):
        p = i // 2
        w[i] = theta[g[i]] + noise_std * delta[p]
        w[i + 1] = theta[g[i]] + (-noise_std) * delta[p]
    out = np.empty(obs.shape, dtype=obs.dtype)
    for gi, s_ in enumerate(env._group_specs):
        sel = g == gi
        out[sel] = ao.policy_actions(w[sel], obs[sel], obs.dtype.type,
                                     float(s_.action_space_max))
    return out


# (config, extra env kwargs)
CASES = {
    "f32_order1_D2": (cont(), {}),
    "f64_order2_D6": (cont(6, transition_dynamics_order=2, dtype_s=np.float64), {}),
    "f32_order3_D1": (cont(1, transition_dynamics_order=3, time_unit=0.3), {}),
    "f32_order4_D16": (cont(16, transition_dynamics_order=4, time_unit=0.2,
                            state_space_max=8.0), {}),
    "unbounded": ({k: v for k, v in cont(3).items()
                   if k not in ("state_space_max", "action_space_max")}, {}),
    "delay": (cont(2, delay=2, transition_dynamics_order=2), {}),
    "noise_fp64": (cont(2, transition_noise=0.05, reward_noise=0.1), {}),
    "noise_ziggurat": (cont(2, transition_noise=0.05, reward_noise=0.1),
                       {"normal_precision": "ziggurat"}),
    "noise_fast": (cont(2, transition_noise=0.05, reward_noise=0.1),
                   {"normal_precision": "fast"}),
    "f64_noise": (cont(4, transition_noise=0.05, reward_noise=0.1, dtype_s=np.float64), {}),
    "line": ({k: v for k, v in cont(2, sequence_length=4,
                                    reward_function="move_along_a_line").items()
              if k not in ("target_point", "target_radius", "make_denser")}, {}),
    "three_groups": (cont(2), {"config_groups": [
        {"transition_dynamics_order": 1}, {"transition_dynamics_order": 2},
        {"transition_dynamics_order": 3, "action_space_max": 0.5}],
        "group_sizes": [64, 96, 96]}),
}


def case_env(name, n=256, seed=3):
    cfg, kw = CASES[name]
    return make_env(n, autoreset=True, horizon=25, philox_seed=seed, **cfg, **kw)


def learner(env, **k):
    from mdp_playground_b200 import LinearARS
    return LinearARS(env, **k)


def random_theta(ag, scale=0.4, seed=0):
    g = torch.Generator().manual_seed(seed)
    ag.theta.copy_(torch.randn(ag.theta.shape, generator=g, dtype=torch.float64) * scale)


# -- 1. the recorded actions are the policy's ----------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_actions_are_the_policy(name):
    env = case_env(name)
    ag = learner(env, noise_std=0.5)
    random_theta(ag)
    obs = np_(env.get_augmented_state()["curr_state"])
    for T in (37, 20):  # two consecutive learn calls
        got = ag.learn(T, record=True)
        acts, o = np_(got["actions"]), np_(got["obs"])
        assert acts.dtype == obs.dtype and acts.shape == (T, env.num_envs, obs.shape[1])
        for t in range(T):
            want = host_actions(env, ag, obs, 0.5)
            assert np.array_equal(acts[t].view(np.uint8), want.view(np.uint8)), (name, T, t)
            obs = o[t]


# -- 2. replay --------------------------------------------------------------------
@pytest.mark.parametrize("name", ["noise_fp64", "delay", "three_groups", "f64_order2_D6"])
def test_recorded_actions_replay_as_a_rollout(name):
    a, b = case_env(name), case_env(name)
    ag = learner(a, noise_std=0.5)
    random_theta(ag)
    for T in (37, 64, 1):
        got = ag.learn(T, record=True)
        want = b.rollout(T, actions=got["actions"])
        for k in ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(got[k], want[k]), (T, k)
    sa, sb = a.get_augmented_state(), b.get_augmented_state()
    for k in ("curr_state", "state_derivatives"):
        assert torch.equal(sa[k], sb[k]), k
    assert a._step_index == b._step_index == 102
    sta, stb = a.episode_stats(), b.episode_stats()
    for k in sta:
        assert np.array_equal(sta[k], stb[k]), k


# -- 3. perturbations ---------------------------------------------------------------
def test_perturbations_match_the_oracle():
    env = case_env("three_groups", seed=11)
    ag = learner(env)
    d0 = np_(ag.perturbations())
    gid = np.arange(0, env.num_envs, 2)  # global ids of the + members
    want = ao.perturbations(env.philox_seed, gid, 0, 2)
    np.testing.assert_allclose(d0, want, rtol=1e-14, atol=1e-14)
    assert len({d0[p].tobytes() for p in range(len(d0))}) == len(d0)  # pairs differ
    ag.update()
    d1 = np_(ag.perturbations())
    np.testing.assert_allclose(d1, ao.perturbations(env.philox_seed, gid, 1, 2),
                               rtol=1e-14, atol=1e-14)
    assert not np.any(d0 == d1)  # iterations differ
    assert not np.array_equal(d0[:32], d0[32:64])  # groups differ


def test_perturbation_moments():
    env = make_env(48000, autoreset=True, horizon=10, philox_seed=5, **cont(6))
    d = np_(learner(env).perturbations()).reshape(-1)
    n = d.size
    assert n >= 10**6
    assert abs(d.mean()) < 5 / np.sqrt(n)
    assert abs(d.var() - 1.0) < 5 * np.sqrt(2.0 / n)


# -- 4. fitness -----------------------------------------------------------------------
def test_fitness_is_the_sequential_reward_sum():
    env = case_env("noise_fp64")
    ag = learner(env, noise_std=0.3)
    random_theta(ag)
    f = np.zeros(env.num_envs)
    for T in (30, 1, 45):
        r = np_(ag.learn(T, record=True)["reward"]).astype(np.float64)
        for t in range(T):
            f = f + r[t]
    assert np.array_equal(np_(ag.fitness), f)


# -- 5. update -------------------------------------------------------------------------
@pytest.mark.parametrize("top", [None, 5])
def test_update_matches_the_oracle(top):
    env = case_env("three_groups")
    ag = learner(env, step_size=0.05, noise_std=0.2, top_directions=top)
    random_theta(ag, 0.2)
    ag.learn(60)
    theta, fit, delta = np_(ag.theta), np_(ag.fitness), np_(ag.perturbations())
    res = ag.update()
    begin = np.cumsum([0] + env._group_sizes)
    for g in range(env.n_groups):
        lo, hi = begin[g], begin[g + 1]
        b = ag.top_directions
        want, m, sigma, upd = ao.update(theta[g], fit[lo:hi], delta[lo // 2:hi // 2], b, 0.05)
        assert upd and res["updated"][g]
        assert np.array_equal(np_(ag.theta)[g], want), g
        assert res["fitness_mean"][g] == m and res["sigma_R"][g] == sigma
    assert ag.iteration == 1 and not ag.fitness.any()


def test_equal_fitness_leaves_the_group_unchanged():
    # group 1: sparse reward at an unreachable target: every return is 0
    env = make_env(128, autoreset=True, horizon=20, philox_seed=2, **cont(2),
                   config_groups=[{}, {"make_denser": False, "target_point": [3.9, 3.9],
                                       "target_radius": 1e-6}], group_sizes=[64, 64])
    ag = learner(env, step_size=0.05, noise_std=0.1)
    random_theta(ag, 0.1)
    before = ag.theta.clone()
    ag.learn(40)
    res = ag.update()
    assert list(res["updated"]) == [True, False] and res["sigma_R"][1] == 0.0
    assert torch.equal(ag.theta[1], before[1]) and not torch.equal(ag.theta[0], before[0])
    assert ag.iteration == 1 and not ag.fitness.any()


# -- 6. noise_std = 0 ---------------------------------------------------------------------
def test_zero_noise_acts_with_theta():
    env = make_env(128, autoreset=True, horizon=0, philox_seed=9, **cont(3))
    st = env.get_augmented_state()["curr_state"].clone()
    st[1::2] = st[0::2]  # both members of each pair start in the same state
    env.set_augmented_state(st)
    ag = learner(env)
    random_theta(ag, 0.3)
    got = ag.learn(10, record=True, noise_std=0.0)
    a = got["actions"]
    assert torch.equal(a[:, 0::2], a[:, 1::2])
    assert torch.equal(got["obs"][:, 0::2], got["obs"][:, 1::2])


# -- 7. it learns ------------------------------------------------------------------------
def test_it_learns_move_to_a_point():
    """tests/test_ars_oracle.py::test_ars_learns_on_the_oracle improved the
    order-1 cells' mean return by 9.1 over 10 iterations; the device run
    must reach at least half of that."""
    from mdp_playground_b200 import sweep
    sw = quiet(sweep.Sweep, FIXTURE, envs_per_cell=16)
    assert len(sw.envs) == 1 and sw.env.n_groups == sw.n_cells
    res = sw.train_continuous(10, 100)
    order1 = np.array([c["transition_dynamics_order"] == 1 for c in sw.cell_configs])
    first = np.nanmean(res[0]["episode_reward_mean"][order1])
    last = np.nanmean(res[-1]["episode_reward_mean"][order1])
    assert last - first >= 0.5 * 9.1, (first, last)


# -- 8. Sweep -------------------------------------------------------------------------------
def check_csv(sw, path, iterations, steps):
    lines = open(sw.write_csv(path)).read().splitlines()
    rows = [ln.split(" ") for ln in lines[1:]]
    assert len(rows) == iterations * sw.n_cells
    assert {r[1] for r in rows} == {"ARS"}
    ts = np.array([int(r[-3]) for r in rows]).reshape(iterations, sw.n_cells)
    assert (np.diff(ts, axis=0) > 0).all()
    assert (ts[0] == steps * sw.envs_per_cell).all()


def test_sweep_train_continuous_on_the_grouped_fixture(tmp_path):
    from mdp_playground_b200 import sweep
    sw = quiet(sweep.Sweep, FIXTURE, envs_per_cell=8)
    sw.train_continuous(3, 100, chunk=64)
    check_csv(sw, str(tmp_path / "g.csv"), 3, 100)


DIM_EXPERIMENT = types.ModuleType("cont_dims_like")
DIM_EXPERIMENT.var_env_configs = OrderedDict({
    "state_space_dim": [2, 3], "time_unit": [0.5, 1.0]})
DIM_EXPERIMENT.env_config = {
    "env": "RLToy-v0", "horizon": 30,
    "env_config": {"seed": 0, "state_space_type": "continuous",
                   "action_space_type": "continuous", "relevant_indices": [0, 1],
                   "target_point": [0.0, 0.0], "target_radius": 0.3,
                   "state_space_max": 4.0, "action_space_max": 1.0,
                   "transition_dynamics_order": 1, "inertia": 1.0,
                   "reward_function": "move_to_a_point", "make_denser": True}}


def test_sweep_train_continuous_one_learner_per_cell(tmp_path):
    from mdp_playground_b200 import LinearARS, VectorRLToyEnv, sweep
    sw = quiet(sweep.Sweep, DIM_EXPERIMENT, envs_per_cell=32)
    assert len(sw.envs) == sw.n_cells == 4 and not getattr(sw, "grouped", False)
    res = sw.train_continuous(2, 100, step_size=0.05, noise_std=0.1, chunk=64)
    check_csv(sw, str(tmp_path / "c.csv"), 2, 100)
    for i, cfg in enumerate(sw.cell_configs):
        env = quiet(VectorRLToyEnv, 32, autoreset=True, horizon=30,
                    env_id_offset=i * 32, **cfg)
        ag = LinearARS(env, step_size=0.05, noise_std=0.1)
        for it in range(2):
            ag.episode_returns(clear=True)
            for T in (64, 36):
                ag.learn(T)
            ret = ag.episode_returns()
            ag.update()
            np.testing.assert_array_equal(res[it]["episode_reward_mean"][i],
                                          ret["episode_reward_mean"][0])
            assert res[it]["timesteps_total"][i] == env.episode_stats()["transitions"][0]
        assert torch.equal(sw.agents[i].theta, ag.theta)


def test_sweep_train_continuous_rejects_the_other_kinds():
    from mdp_playground_b200 import sweep
    for fixture in ("grid_noises_like.py", "dqn_seq_del_like.py"):
        sw = quiet(sweep.Sweep, os.path.join(HERE, "fixtures", fixture), envs_per_cell=4)
        with pytest.raises(NotImplementedError, match="continuous experiments only"):
            sw.train_continuous(1, 10)
    sw = quiet(sweep.Sweep, FIXTURE, envs_per_cell=4, shard=(0, 2))
    with pytest.raises(NotImplementedError, match="sharded"):
        sw.train_continuous(1, 10)
    # Sweep.train still runs discrete experiments only
    with pytest.raises(NotImplementedError):
        quiet(sweep.Sweep, FIXTURE, envs_per_cell=4).train(1, 10)


# -- 9. rejections ------------------------------------------------------------------------------
def test_python_rejections():
    from mdp_playground_b200 import LinearARS
    with pytest.raises(ValueError, match="continuous env"):
        LinearARS(make_env(8, state_space_type="discrete", action_space_type="discrete",
                           state_space_size=4, action_space_size=4, seed=0))
    with pytest.raises(ValueError, match="philox"):
        LinearARS(make_env(8, noise="numpy", **cont(2)))
    with pytest.raises(ValueError, match="image_representations"):
        LinearARS(make_env(8, **dict(cont(4), image_representations=True,
                                     state_space_max=5.0)))
    with pytest.raises(ValueError, match="even number"):
        LinearARS(make_env(7, **cont(2)))
    with pytest.raises(ValueError, match="even number"):
        LinearARS(make_env(12, **cont(2), config_groups=[{}, {}], group_sizes=[5, 7]))
    env = make_env(16, autoreset=True, **cont(2))
    for kw in ({"step_size": 0.0}, {"step_size": float("nan")}, {"noise_std": -0.1},
               {"noise_std": float("inf")}, {"top_directions": 0},
               {"top_directions": 9}):
        with pytest.raises(ValueError):
            LinearARS(env, **kw)
    with pytest.raises(ValueError):
        LinearARS(env).learn(4, noise_std=-1.0)


def test_c_abi_rejections():
    from mdp_playground_b200 import _lib
    env = make_env(16, autoreset=True, philox_seed=2, **cont(2))
    ag = learner(env)
    lib = env._lib

    def learn(ap, io=None, opts=None):
        rc = lib.mdpp_continuous_ars(env._ctx, C.byref(env._state),
                                     C.byref(io or _lib.ContinuousIO()), C.byref(ap),
                                     C.byref(opts or env._opts(8, _lib.MDPP_NOISE_PHILOX)),
                                     env._stream())
        return rc, lib.mdpp_last_error(env._ctx).decode()

    def update(ap):
        rc = lib.mdpp_continuous_ars_update(env._ctx, env.num_envs, C.byref(ap),
                                            env._stream())
        return rc, lib.mdpp_last_error(env._ctx).decode()

    def params(**kw):
        ap = ag._params()
        for k, v in kw.items():
            setattr(ap, k, v)
        return ap

    acts = torch.zeros((8, 16, 2), dtype=torch.float32, device=env.device)
    io = _lib.ContinuousIO()
    io.actions = acts.data_ptr()
    assert learn(params(), io=io) == (
        -1, "ars: io->actions must be NULL (the policy acts)")
    for mode in (_lib.MDPP_NOISE_OFF, _lib.MDPP_NOISE_REPLAY):
        assert learn(params(), opts=env._opts(8, mode)) == (-1, "ars: Philox noise only")
    null = (-1, "ars: theta, fitness, ep_return, ret_sum or ret_count is NULL")
    for k in ("theta", "fitness", "ep_return", "ret_sum", "ret_count"):
        assert learn(params(**{k: None})) == null, k
    for k in ("theta", "fitness"):
        assert update(params(**{k: None})) == null, k
    top = (-1, "ars: top_directions must lie in [1, the smallest group's pairs]")
    for v in (0, 9):
        assert learn(params(top_directions=v)) == top
        assert update(params(top_directions=v)) == top
    for v in (0.0, -1.0, float("nan"), float("inf")):
        assert update(params(step_size=v)) == (-1, "ars: step_size must be finite and > 0")
    for v in (-0.5, float("nan"), float("inf")):
        assert learn(params(noise_std=v)) == (-1, "ars: noise_std must be finite and >= 0")
    assert learn(params(), opts=env._opts(0, _lib.MDPP_NOISE_PHILOX)) == (
        -1, "ars: T must be >= 1")
    odd = make_env(15, autoreset=True, **cont(2))
    ap = params()
    ap.top_directions = 1
    rc = lib.mdpp_continuous_ars_update(odd._ctx, 15, C.byref(ap), odd._stream())
    assert (rc, lib.mdpp_last_error(odd._ctx).decode()) == (
        -1, "ars: every group needs an even number (>= 2) of envs")
    img = make_env(16, **dict(cont(4), image_representations=True, state_space_max=5.0))
    rc = lib.mdpp_continuous_ars_update(img._ctx, 16, C.byref(params()), img._stream())
    assert (rc, lib.mdpp_last_error(img._ctx).decode()) == (
        -1, "ars: image observations are not supported")
    # nothing ran
    assert ag.iteration == 0 and not ag.fitness.any() and not ag.theta.any()
