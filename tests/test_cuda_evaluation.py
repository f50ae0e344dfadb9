"""GPU tests of the evaluation launches (mdpp_discrete_qeval, mdpp_grid_qeval,
mdpp_continuous_ars_eval; TabularQLearner / GridQLearner / LinearARS
.evaluate; Sweep's evaluation and write_eval_csv)."""
import ctypes as C
import os
import re
import warnings

import numpy as np
import pytest
import torch

from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_continuous_oracle import (VectorContinuousOracle,
                                             VectorGroupedContinuousOracle)
from oracle.vector_grid_oracle import VectorGridOracle, VectorGroupedGridOracle
from oracle.vector_oracle import VectorDiscreteOracle, VectorGroupedOracle
from tests import eval_oracle as eo
from tests import golden_util as gu

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def quiet(f, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return f(*a, **k)


def make_env(*a, **k):
    from mdp_playground_b200 import VectorRLToyEnv
    return quiet(VectorRLToyEnv, *a, **k)


def np_(t):
    return t.cpu().numpy()


def disc(**kw):
    c = dict(seed=7, state_space_type="discrete", action_space_type="discrete",
             state_space_size=8, action_space_size=5, sequence_length=1, delay=0,
             reward_density=0.25, terminal_state_density=0.25)
    c.update(kw)
    return c


def grid(**kw):
    c = dict(seed=0, state_space_type="grid", grid_shape=(5, 7), delay=0,
             sequence_length=1, reward_function="move_to_a_point",
             target_point=[3, 4], make_denser=True)
    c.update(kw)
    return c


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


# name -> (kind, env kwargs (one config or config_groups), horizon)
CASES = {
    "disc_zig_rnoise": ("discrete", dict(normal_precision="ziggurat",
                                         **disc(reward_noise=0.25, transition_noise=0.1)), 9),
    "disc_f64_seq3_delay2": ("discrete", dict(normal_precision="boxmuller",
                                              **disc(sequence_length=3, delay=2,
                                                     reward_noise=0.25,
                                                     reward_every_n_steps=True)), 12),
    "disc_fast_delay17": ("discrete", dict(normal_precision="fast",
                                           **disc(delay=17, reward_noise=0.25)), 25),
    "disc_generic_tables": ("discrete", dict(**disc(state_space_size=300,
                                                    action_space_size=4,
                                                    transition_noise=0.1)), 9),
    "disc_groups": ("discrete", dict(config_groups=[
        disc(), disc(state_space_size=6, action_space_size=4, delay=1),
        disc(sequence_length=2, reward_noise=0.5)], group_sizes=[24, 40, 32]), 10),
    "grid_2d": ("grid", dict(**grid(transition_noise=0.25, reward_noise=1.0)), 9),
    "grid_4d_irr": ("grid", dict(**grid(irrelevant_features=True, grid_shape=(3, 4),
                                        target_point=[1, 2], transition_noise=0.25)), 9),
    "grid_groups": ("grid", dict(config_groups=[
        grid(), grid(grid_shape=(8, 8), target_point=[5, 5], transition_noise=0.25),
        grid(grid_shape=(3, 3), target_point=[1, 1], make_denser=False)],
        group_sizes=[32, 32, 32]), 9),
    "cont_f32_o1_D2": ("continuous", dict(**cont(2)), 12),
    "cont_f64_o2_D1": ("continuous", dict(**cont(1, transition_dynamics_order=2,
                                                 dtype_s=np.float64)), 12),
    "cont_f32_o3_D6_unbounded": ("continuous", dict(**cont(
        6, transition_dynamics_order=3, action_space_max=np.inf,
        transition_noise=0.01, reward_noise=0.1)), 10),
    "cont_f64_o4_D16": ("continuous", dict(**cont(16, transition_dynamics_order=4,
                                                  dtype_s=np.float64)), 8),
    "cont_groups": ("continuous", dict(config_groups=[
        cont(2), cont(2, time_unit=1.0, transition_dynamics_order=2),
        cont(2, action_space_max=0.5, target_point=[1.0, -1.0])],
        group_sizes=[32, 32, 32]), 12),
}


def build(name, n=96):
    kind, kw, horizon = CASES[name]
    kw = dict(kw)
    if "config_groups" not in kw:
        kw.setdefault("num_envs", n)
    else:
        kw["num_envs"] = sum(kw["group_sizes"])
    N = kw.pop("num_envs")
    return kind, make_env(N, autoreset=True, horizon=horizon, **kw), horizon


def learner_of(kind, env):
    from mdp_playground_b200 import GridQLearner, LinearARS, TabularQLearner
    return {"discrete": TabularQLearner, "grid": GridQLearner,
            "continuous": LinearARS}[kind](env)


def fixed_policy(kind, ag, seed=0):
    """A fixed random policy: Q-tables with seeded exact ties, or theta."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    if kind == "continuous":
        ag.theta.copy_(torch.randn(ag.theta.shape, generator=g, dtype=torch.float64) * 0.5)
        return ag.theta
    ag.q.copy_(torch.randint(0, 3, ag.q.shape, generator=g).to(torch.float64))
    return ag.q


def oracle_of(kind, env, horizon):
    """The batched oracle of env, reset like its constructor did."""
    specs = env._group_specs
    if kind == "discrete":
        one, many = VectorDiscreteOracle, VectorGroupedOracle
        kw = {"normal": "boxmuller"} if env.normal_precision == "boxmuller" else \
            {"fast_normal": True} if env.normal_precision == "fast" else {}
    elif kind == "grid":
        one, many = VectorGridOracle, VectorGroupedGridOracle
        kw = {"normal": "ziggurat"} if env.normal_precision == "ziggurat" else \
            {"fast_normal": True} if env.normal_precision == "fast" else {}
    else:
        one, many = VectorContinuousOracle, VectorGroupedContinuousOracle
        kw = {}
    if env.n_groups == 1:
        o = one(quiet(ScalarRLToyEnv, **specs[0].config), env.num_envs, autoreset=True,
                horizon=horizon, seed=env.philox_seed, **kw)
    else:
        o = many([quiet(ScalarRLToyEnv, **s_.config) for s_ in specs], env._group_sizes,
                 autoreset=True, horizon=horizon, seed=env.philox_seed, **kw)
    o.reset()
    return o


def learn_as_evaluation(kind, name, policy, E):
    """The same evaluation through the learner: a second, identically built
    env, reset(), learn(E * H) with nothing learned and no exploration."""
    _, env, H = build(name)
    ag = learner_of(kind, env)
    if kind == "continuous":
        ag.theta.copy_(policy)
        env.reset()
        out = ag.learn(E * H, noise_std=0.0, record=True)
    else:
        ag.q.copy_(policy)
        env.reset()
        out = ag.learn(E * H, alpha=0.0, epsilon=0.0, record=True)
    return env, out


@pytest.mark.parametrize("name", list(CASES))
def test_evaluate_equals_the_learners_greedy_run(name):
    E = 3
    kind, env, H = build(name)
    ev_env = build(name)[1]
    ag = learner_of(kind, env)
    policy = fixed_policy(kind, ag)
    res = ag.evaluate(ev_env, E, per_env=True)
    ref_env, out = learn_as_evaluation(kind, name, policy, E)
    ended = np_(out["terminated"] | out["truncated"])
    ret_sum, count, len_sum = eo.first_episodes(np_(out["reward"]), ended, E)
    assert np.array_equal(np_(res["ret_sum"]), ret_sum)  # bit for bit
    assert np.array_equal(np_(res["ret_count"]), count)
    assert np.array_equal(np_(res["len_sum"]), len_sum)
    assert (count == E).all() and (len_sum <= E * H).all()
    # the env stepped exactly as the learner's greedy run: same end state
    # (the statistics are atomically added float sums: not compared bitwise)
    for a, b in zip(ev_env._state_tensors(), ref_env._state_tensors()):
        if a is ev_env._stats or b is ref_env._stats:
            continue
        if a.dtype.is_floating_point:
            a, b = a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8)
        assert torch.equal(a, b)
    assert ev_env._step_index == ref_env._step_index == E * H
    g = np.repeat(np.arange(ev_env.n_groups), ev_env._group_sizes)
    for k in range(ev_env.n_groups):
        assert res["episodes"][k] == E * (g == k).sum()
        np.testing.assert_allclose(res["episode_reward_mean"][k],
                                   ret_sum[g == k].sum() / (E * (g == k).sum()))
        np.testing.assert_allclose(res["episode_len_mean"][k],
                                   len_sum[g == k].sum() / (E * (g == k).sum()))


@pytest.mark.parametrize("name", ["disc_zig_rnoise", "disc_groups", "grid_4d_irr",
                                  "grid_groups", "cont_f32_o1_D2", "cont_groups"])
def test_evaluate_matches_the_oracle(name):
    E = 2
    kind, env, H = build(name, n=32)
    ev_env = build(name, n=32)[1]
    ora = oracle_of(kind, ev_env, H)
    ag = learner_of(kind, env)
    policy = np_(fixed_policy(kind, ag, seed=3))
    res = ag.evaluate(ev_env, E, per_env=True)
    ora.reset()  # evaluate's reset()
    want = eo.evaluate(ora, kind, policy, E, H)
    if kind == "continuous" and ev_env._real == torch.float32:
        np.testing.assert_allclose(np_(res["ret_sum"]), want["ret_sum"], rtol=1e-5,
                                   atol=1e-5)
    else:
        assert np.array_equal(np_(res["ret_sum"]), want["ret_sum"])
    assert np.array_equal(np_(res["ret_count"]), want["ret_count"])
    assert np.array_equal(np_(res["len_sum"]), want["len_sum"])


@pytest.mark.parametrize("name", ["disc_f64_seq3_delay2", "grid_groups", "cont_groups"])
def test_evaluate_leaves_training_state_untouched(name):
    kind, env, H = build(name)
    ev_env = build(name)[1]
    ag = learner_of(kind, env)
    fixed_policy(kind, ag)
    if kind == "continuous":
        ag.learn(17)
        ag.update()
        ag.learn(5)
        own = [ag.theta, ag.fitness]
    else:
        ag.learn(23)
        own = [ag.q]
    own += [ag.ep_return, ag.ret_sum, ag.ret_count]
    before = [t.clone() for t in own + [x for x in env._state_tensors() if x is not None]]
    meta = (env._step_index, getattr(ag, "iteration", None), env.episode_stats())
    res = ag.evaluate(ev_env, 4, per_env=True)
    after = own + [x for x in env._state_tensors() if x is not None]
    assert all(torch.equal(a, b) for a, b in zip(before, after))
    assert env._step_index == meta[0] and getattr(ag, "iteration", None) == meta[1]
    st = env.episode_stats()
    assert all(np.array_equal(np.asarray(st[k]), np.asarray(meta[2][k])) for k in st)
    assert (np_(res["ret_count"]) == 4).all() and (np_(res["len_sum"]) <= 4 * H).all()
    # a second evaluation starts from fresh initial states (reset() without a seed)
    res2 = ag.evaluate(ev_env, 4, per_env=True)
    assert (np_(res2["ret_count"]) == 4).all()
    assert ev_env._step_index == 8 * H


def test_python_rejections():
    from mdp_playground_b200 import GridQLearner, LinearARS, TabularQLearner
    N = 16
    ag = TabularQLearner(make_env(N, autoreset=True, horizon=9, **disc()))
    bad = {
        "GridEnv": make_env(N, autoreset=True, horizon=9, **grid()),
        "envs": make_env(2 * N, autoreset=True, horizon=9, **disc()),
        "groups": make_env(N, autoreset=True, horizon=9,
                           config_groups=[disc(), disc()], group_sizes=[8, 8]),
        "(S, A)": make_env(N, autoreset=True, horizon=9, **disc(action_space_size=4)),
        "irrelevant_features": make_env(N, autoreset=True, horizon=9,
                                        **gu.case_config("irr_8x5_det")),
        "philox": make_env(N, autoreset=True, horizon=9, noise="replay", **disc()),
        "image_representations": make_env(N, autoreset=True, horizon=9,
                                          **disc(image_representations=True)),
        "autoreset": make_env(N, autoreset=False, horizon=9, **disc()),
        "horizon": make_env(N, autoreset=True, horizon=0, **disc()),
    }
    for what, e in bad.items():
        with pytest.raises(ValueError, match=r"evaluate: .*" + re.escape(what)):
            ag.evaluate(e, 2)
    with pytest.raises(ValueError, match="episodes"):
        ag.evaluate(make_env(N, autoreset=True, horizon=9, **disc()), 0)
    gq = GridQLearner(make_env(N, autoreset=True, horizon=9, **grid()))
    with pytest.raises(ValueError, match="grid shapes"):
        gq.evaluate(make_env(N, autoreset=True, horizon=9, **grid(grid_shape=(5, 6))), 2)
    ars = LinearARS(make_env(N, autoreset=True, horizon=9, **cont(2)))
    with pytest.raises(ValueError, match="D = "):
        ars.evaluate(make_env(N, autoreset=True, horizon=9, **cont(1)), 2)
    with pytest.raises(ValueError, match="D = "):
        ars.evaluate(make_env(N, autoreset=True, horizon=9, **cont(2, dtype_s=np.float64)), 2)


def test_c_abi_rejections():
    from mdp_playground_b200 import _lib
    N, H = 64, 9
    cases = {
        "qeval": (make_env(N, autoreset=True, horizon=H, **disc()), "mdpp_discrete_qeval"),
        "grid qeval": (make_env(N, autoreset=True, horizon=H, **grid()), "mdpp_grid_qeval"),
        "ars eval": (make_env(N, autoreset=True, horizon=H, **cont(2)),
                     "mdpp_continuous_ars_eval"),
    }
    for who, (env, entry) in cases.items():
        lib, dev = env._lib, env.device
        q = torch.zeros((N, 64, 9), dtype=torch.float64, device=dev)
        th = torch.zeros((1, 2, 3), dtype=torch.float64, device=dev)
        rs = torch.zeros(N, dtype=torch.float64, device=dev)
        rc_ = torch.zeros(N, dtype=torch.int32, device=dev)
        ls = torch.zeros(N, dtype=torch.int64, device=dev)

        def params(**kw):
            p = _lib.EvalParams()
            p.q, p.q_states, p.q_actions = q.data_ptr(), 64, 9
            p.theta = th.data_ptr()
            p.episodes = 2
            p.ret_sum, p.ret_count, p.len_sum = rs.data_ptr(), rc_.data_ptr(), ls.data_ptr()
            for k, v in kw.items():
                setattr(p, k, v)
            return p

        def call(p=None, io=None, opts=None):
            rc = getattr(lib, entry)(env._ctx, C.byref(env._state),
                                     C.byref(io or env._IO()), C.byref(p or params()),
                                     C.byref(opts or env._opts(2 * H)), env._stream())
            return rc, lib.mdpp_last_error(env._ctx).decode()

        assert call()[0] == 0, call()
        torch.cuda.synchronize()
        assert (rc_ == 2).all()
        acts = torch.zeros((2 * H, N) + env._row, dtype=env._adt if hasattr(env, "_adt")
                           else torch.int32, device=dev)
        io = env._IO()
        io.actions = acts.data_ptr()
        assert call(io=io) == (-1, f"{who}: io->actions must be NULL (the policy acts)")
        o = env._opts(2 * H)
        o.noise_mode = _lib.MDPP_NOISE_OFF
        assert call(opts=o) == (-1, f"{who}: Philox noise only")
        o = env._opts(2 * H)
        o.autoreset = 0
        assert call(opts=o)[1].startswith(f"{who}: needs autoreset")
        o = env._opts(2 * H)
        o.horizon = 0
        assert call(opts=o) == (-1, f"{who}: horizon must be >= 1")
        assert call(p=params(episodes=0)) == (-1, f"{who}: episodes must be >= 1")
        assert call(opts=env._opts(2 * H - 1)) == (
            -1, f"{who}: n_steps must be >= episodes * horizon")
        keys = ("theta",) if who == "ars eval" else ("q",)
        for k in keys + ("ret_sum", "ret_count", "len_sum"):
            assert call(p=params(**{k: None}))[1].endswith(
                "ret_sum, ret_count or len_sum is NULL"), k
        if who != "ars eval":
            assert call(p=params(q_states=1)) == (
                -1, f"{who}: q_states / q_actions smaller than a group's S / A")
            assert call(p=params(q_actions=1)) == (
                -1, f"{who}: q_states / q_actions smaller than a group's S / A")
    irr = make_env(N, autoreset=True, horizon=H, **gu.case_config("irr_8x5_det"))
    p = _lib.EvalParams()
    q = torch.zeros((N, 64, 9), dtype=torch.float64, device=irr.device)
    p.q, p.q_states, p.q_actions, p.episodes = q.data_ptr(), 64, 9, 1
    rc = irr._lib.mdpp_discrete_qeval(irr._ctx, C.byref(irr._state), C.byref(irr._IO()),
                                      C.byref(p), C.byref(irr._opts(H)), irr._stream())
    assert (rc, irr._lib.mdpp_last_error(irr._ctx).decode()) == (
        -1, "qeval: irrelevant features are not supported")


# -- Sweep -----------------------------------------------------------------------
def _tables_equal(kind, a, b):
    if kind == "discrete":
        for x, y in zip(a.group_tables, b.group_tables):
            for k in ("transition", "terminal_states", "init_cdf", "init_state_dist",
                      "sequences", "sequence_rewards"):
                assert np.array_equal(getattr(x, k), getattr(y, k)), k
    else:
        for x, y in zip(a._group_specs, b._group_specs):
            for k in ("target_point", "terminal_states", "grid_shape", "state_space_dim",
                      "relevant_indices", "action_space_max", "state_space_max",
                      "time_unit", "transition_dynamics_order", "reward_scale"):
                if hasattr(x, k):
                    assert np.array_equal(np.asarray(getattr(x, k), dtype=object),
                                          np.asarray(getattr(y, k), dtype=object)), k
    assert a.num_envs == b.num_envs and a._group_sizes == b._group_sizes
    assert a.env_id_offset == b.env_id_offset and a.philox_seed == b.philox_seed


@pytest.mark.parametrize("fixture,method,kw", [
    ("dqn_seq_del_eval_like.py", "train", dict(alpha=0.2, gamma=0.9, epsilon=0.2)),
    ("grid_noises_like.py", "train_grid", dict(alpha=0.2, gamma=0.9, epsilon=0.2)),
    ("ddpg_move_to_a_point_like.py", "train_continuous", {}),
])
def test_sweep_evaluation(tmp_path, fixture, method, kw):
    from mdp_playground_b200 import sweep
    sw = quiet(sweep.Sweep, os.path.join(HERE, "fixtures", fixture), envs_per_cell=8)
    ev = {"evaluation_interval": 2, "evaluation_num_episodes": 3, "horizon": 20}
    if fixture != "dqn_seq_del_eval_like.py":
        ev["env_config"] = {"transition_noise": 0.0,
                            "reward_noise": lambda a: a.normal(0, 0)}
    getattr(sw, method)(3, 40, evaluation=ev, **kw)
    assert [r["training_iteration"] for r in sw.eval_results] == [2]
    getattr(sw, method)(2, 40, **kw)  # no evaluation: nothing appended
    assert len(sw.eval_results) == 1
    getattr(sw, method)(2, 40, evaluation=True, **kw)  # the first call's settings
    assert [r["training_iteration"] for r in sw.eval_results] == [2, 6]
    assert len(sw.eval_envs) == len(sw.envs)
    for a, b in zip(sw.envs, sw.eval_envs):
        _tables_equal(sw.kind, a, b)
        assert b.horizon == 20
        assert all(s_.reward_noise_std == 0.0 for s_ in b._group_specs)
        assert all(s_.transition_noise == 0.0 for s_ in b._group_specs)
    r = sw.eval_results[-1]
    assert np.array_equal(r["timesteps_total"], sw.train_results[5]["timesteps_total"])
    assert np.isfinite(r["episode_reward_mean"]).all()
    assert ((r["episode_len_mean"] >= 1) & (r["episode_len_mean"] <= 20)).all()
    path = sw.write_eval_csv(str(tmp_path / "eval.csv"))
    lines = open(path).read().splitlines()
    assert lines[0] == open(sw.write_csv(str(tmp_path / "t.csv"))).read().splitlines()[0]
    assert len(lines) == 1 + 2 * sw.n_cells
    it, algo = lines[1].split()[:2]
    assert it == "2" and algo == sw.algorithm
    assert lines[-1].split()[0] == "6"
    assert float(lines[-1].split()[-1]) == pytest.approx(r["episode_len_mean"][-1],
                                                         rel=1e-2)


def test_sweep_evaluation_per_cell_envs():
    import types
    from collections import OrderedDict
    from mdp_playground_b200 import sweep
    exp = types.ModuleType("grid_irrelevant_eval_like")
    exp.var_env_configs = OrderedDict({"irrelevant_features": [False, True],
                                       "transition_noise": [0, 0.25]})
    exp.env_config = {
        "env": "RLToy-v0", "horizon": 30,
        "env_config": {"seed": 0, "state_space_type": "grid", "grid_shape": (4, 4),
                       "target_point": [2, 2], "reward_function": "move_to_a_point",
                       "make_denser": True, "delay": 0, "sequence_length": 1}}
    exp.eval_config = {"evaluation_interval": 1,
                       "evaluation_config": {"explore": False, "evaluation_num_episodes": 2,
                                             "env_config": {"transition_noise": 0}}}
    sw = quiet(sweep.Sweep, exp, envs_per_cell=16)
    assert len(sw.envs) == 4
    sw.train_grid(2, 60, alpha=0.2, gamma=0.9, epsilon=0.2, evaluation=True)
    assert [r["training_iteration"] for r in sw.eval_results] == [1, 2]
    for a, b in zip(sw.envs, sw.eval_envs):
        _tables_equal("grid", a, b)
        assert b.horizon == 30 and b._group_specs[0].transition_noise == 0.0
    assert sw.eval_results[0]["episode_reward_mean"].shape == (4,)


# -- the evaluation measures a learned policy ----------------------------------
def _optimal_q(cfg, gamma):
    """Value iteration on a deterministic (L = 1, no noise) config: the
    one-step reward and successor of every (s, a) from the oracle's step."""
    one = VectorDiscreteOracle(quiet(ScalarRLToyEnv, **cfg), 1, seed=0)
    S, A = one.S, one.A
    probe = VectorDiscreteOracle(quiet(ScalarRLToyEnv, **cfg), S * A, seed=0)
    probe.reset()
    probe.set_state(np.repeat(np.arange(S), A))
    o = probe.rollout(1, actions=np.tile(np.arange(A), S)[None])
    r = o["reward"][0].reshape(S, A)
    nxt = o["final_obs"][0].reshape(S, A)
    done = o["terminated"][0].reshape(S, A)
    q = np.zeros((S, A))
    for _ in range(2000):
        q = r + gamma * np.where(done, 0.0, q[nxt].max(axis=2))
    return q


def test_greedy_evaluation_of_a_trained_learner_is_optimal():
    from mdp_playground_b200 import TabularQLearner
    cfg = disc(state_space_size=8, action_space_size=4, reward_density=0.25,
               terminal_state_density=0.25)
    N, H, E, gamma = 64, 20, 5, 0.9
    env = make_env(N, autoreset=True, horizon=H, **cfg)
    ev_env = make_env(N, autoreset=True, horizon=H, **cfg)
    ag = TabularQLearner(env, alpha=0.5, gamma=gamma, epsilon=0.5)
    for _ in range(40):
        ag.learn(500)
    got = ag.evaluate(ev_env, E, per_env=True)
    ora = VectorDiscreteOracle(quiet(ScalarRLToyEnv, **cfg), N, autoreset=True, horizon=H,
                               seed=ev_env.philox_seed)
    q_star = _optimal_q(cfg, gamma)
    assert q_star.shape == tuple(ag.q.shape[1:])
    ora.reset()
    ora.reset()  # the constructor's reset and evaluate's
    want = eo.evaluate(ora, "discrete", np.broadcast_to(q_star, tuple(ag.q.shape)), E, H)
    assert np.array_equal(np_(got["ret_sum"]), want["ret_sum"])
    assert np.array_equal(np_(got["len_sum"]), want["len_sum"])
