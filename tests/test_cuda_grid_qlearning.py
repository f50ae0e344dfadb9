"""GPU tests of tabular Q-learning in the grid rollout kernel
(mdpp_grid_qlearn, mdp_playground_b200/qlearning.py, Sweep.train on grid
experiments)."""
import ctypes as C
import os
import types
import warnings
from collections import OrderedDict

import numpy as np
import pytest
import torch

from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_grid_oracle import VectorGridOracle
from tests import golden_util as gu
from tests import grid_qlearn_oracle as gqo
from tests import qlearn_oracle as qo

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def quiet(f, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return f(*a, **k)


def make_env(*a, **k):
    from mdp_playground_b200 import VectorRLToyEnv
    return quiet(VectorRLToyEnv, *a, **k)


def learner(env, **k):
    from mdp_playground_b200 import GridQLearner
    return GridQLearner(env, **k)


def grid(**kw):
    c = dict(seed=0, state_space_type="grid", grid_shape=(5, 7), delay=0,
             sequence_length=1, reward_function="move_to_a_point",
             target_point=[3, 4], make_denser=True)
    c.update(kw)
    return c


def np_(t):
    return t.cpu().numpy()


# (config, normal_precision, oracle normal kwargs, autoreset horizon)
NORMALS = {"fp64": {}, "ziggurat": {"normal": "ziggurat"}, "fast": {"fast_normal": True}}
CASES = {
    "dense_5x7": (grid(), "fp64", 9),
    "sparse_pnoise25": (grid(make_denser=False, transition_noise=0.25), "fp64", 12),
    "pnoise1": (grid(transition_noise=1.0), "fp64", 9),
    "rnoise_f64": (grid(reward_noise=1.0, transition_noise=0.25), "fp64", 9),
    "rnoise_fast": (grid(reward_noise=1.0), "fast", 9),
    "rnoise_zig": (grid(reward_noise=1.0, make_denser=False), "ziggurat", 9),
    "every3": (grid(reward_every_n_steps=3), "fp64", 10),
    "scale_shift_term": (grid(reward_scale=2.5, reward_shift=-0.5,
                              term_state_reward=1.5, transition_noise=0.1), "fp64", 9),
    "horizon3_8x8": (grid(grid_shape=(8, 8), target_point=[5, 5]), "fp64", 3),
    "nd4": (grid(irrelevant_features=True, grid_shape=(3, 4), target_point=[1, 2],
                 transition_noise=0.25), "fp64", 9),
}


def pair(name, n):
    cfg, normal, horizon = CASES[name]
    env = make_env(n, autoreset=True, horizon=horizon, normal_precision=normal,
                   track_history=True, **cfg)
    ora = VectorGridOracle(quiet(ScalarRLToyEnv, **cfg), n, autoreset=True,
                           horizon=horizon, seed=env.philox_seed, **NORMALS[normal])
    ora.reset()  # mirrors the reset at the end of the env constructor
    assert np.array_equal(np_(env._pos.t()), ora.pos)
    return env, ora


def end_state(env):
    return {t: getattr(env, t).clone() for t in ("_pos", "_t", "_episode", "_reached", "_prev")}


# -- the recorded rows replay as a rollout ---------------------------------------
@pytest.mark.parametrize("epsilon", [0.0, 0.1, 1.0])
@pytest.mark.parametrize("name", ["sparse_pnoise25", "rnoise_f64", "rnoise_zig", "nd4"])
def test_recorded_actions_replay_as_a_rollout(name, epsilon):
    cfg, normal, horizon = CASES[name]
    n = 300
    a, b = (make_env(n, autoreset=True, horizon=horizon, normal_precision=normal,
                     track_history=True, philox_seed=4, **cfg) for _ in range(2))
    ag = learner(a, alpha=0.5, gamma=0.9, epsilon=epsilon)
    for T in (37, 64, 1):
        got = ag.learn(T, record=True)
        assert got["actions"].dtype == torch.int64
        assert tuple(got["actions"].shape) == (T, n, a._nd)
        want = b.rollout(T, actions=got["actions"])
        for k in ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(got[k], want[k]), (T, k)
    sa, sb = end_state(a), end_state(b)
    for t in sa:
        assert torch.equal(sa[t], sb[t]), t
    assert a._step_index == b._step_index == 102
    sta, stb = a.episode_stats(), b.episode_stats()
    for k in sta:
        assert np.array_equal(sta[k], stb[k]), k


# -- CUDA against the restatement ------------------------------------------------
@pytest.mark.parametrize("epsilon", [0.0, 0.1, 1.0])
@pytest.mark.parametrize("name", list(CASES))
def test_qlearn_matches_the_restatement(name, epsilon):
    n = 64
    env, ora = pair(name, n)
    ag = learner(env, alpha=0.3, gamma=0.95, epsilon=epsilon)
    assert ag.q.shape[1] == gqo.n_cells(ora.shape)
    assert ag.q.shape[2] == (8 if ora.nd == 2 else 9)
    q = np.zeros(tuple(ag.q.shape))
    acc = qo.new_accumulators(n)
    noisy = "reward_noise" in CASES[name][0]
    fast = CASES[name][1] == "fast"
    for T in (61, 14):  # from an even and from an odd step
        got = ag.learn(T, record=True)
        want = gqo.qlearn(ora, T, 0.3, 0.95, epsilon, q, acc)
        for k in ("obs", "terminated", "truncated", "actions"):
            assert np.array_equal(np_(got[k]), want[k]), (T, k)
        if noisy:
            tol = 1e-5 if fast else 1e-12
            np.testing.assert_allclose(np_(got["reward"]), want["reward"],
                                       rtol=tol, atol=tol)
        else:
            assert np.array_equal(np_(got["reward"]), want["reward"])
    if noisy:
        tol = 1e-5 if fast else 1e-9
        np.testing.assert_allclose(np_(ag.q), q, rtol=tol, atol=tol)
        np.testing.assert_allclose(np_(ag.ret_sum), acc["ret_sum"], rtol=tol, atol=tol)
    else:
        assert np.array_equal(np_(ag.q), q)
        assert np.array_equal(np_(ag.ep_return), acc["ep_return"])
        assert np.array_equal(np_(ag.ret_sum), acc["ret_sum"])
    assert np.array_equal(np_(ag.ret_count), acc["ret_count"])
    assert np.array_equal(np_(env._pos.t()), ora.pos)
    st = env.episode_stats()
    for k in ("episodes", "transitions", "noisy_transitions", "terminated"):
        assert st[k][0] == ora.stats[k], k


def test_no_outputs_and_overrides():
    env, ora = pair("scale_shift_term", 128)
    ag = learner(env, alpha=0.3, gamma=0.95, epsilon=0.2)
    q = np.zeros(tuple(ag.q.shape))
    assert ag.learn(50) is None
    gqo.qlearn(ora, 50, 0.3, 0.95, 0.2, q)
    assert np.array_equal(np_(ag.q), q)
    before = ag.q.clone()  # a greedy evaluation leaves q as it is
    out = ag.learn(20, record=True, epsilon=0.0, alpha=0.0)
    assert torch.equal(ag.q, before)
    want = gqo.qlearn(ora, 20, 0.0, 0.95, 0.0, q)
    assert np.array_equal(np_(out["actions"]), want["actions"])


# -- launch shapes ---------------------------------------------------------------
def test_one_launch_equals_two():
    cfg, normal, horizon = CASES["rnoise_zig"]
    envs = [make_env(512, autoreset=True, horizon=horizon, normal_precision=normal,
                     track_history=True, **cfg) for _ in range(2)]
    ags = [learner(e, epsilon=0.2) for e in envs]
    ags[0].learn(302)
    ags[1].learn(151)
    ags[1].learn(151)
    for t in ("q", "ep_return", "ret_sum", "ret_count"):
        assert torch.equal(getattr(ags[0], t), getattr(ags[1], t)), t
    sa, sb = end_state(envs[0]), end_state(envs[1])
    for t in sa:
        assert torch.equal(sa[t], sb[t]), t
    assert envs[0]._step_index == envs[1]._step_index == 302


GROUPS = [grid(), grid(grid_shape=(8, 8), target_point=[5, 5], transition_noise=0.25),
          grid(grid_shape=(3, 3), target_point=[1, 1], make_denser=False,
               reward_noise=0.5),
          grid(grid_shape=(6, 2), target_point=[4, 1], reward_every_n_steps=2)]
GSIZES = [64, 96, 32, 160]


def test_grouped_launch_equals_one_env_per_group():
    N, T = sum(GSIZES), 90
    het = make_env(N, autoreset=True, horizon=15, philox_seed=5,
                   config_groups=GROUPS, group_sizes=GSIZES)
    ag = learner(het, epsilon=0.3)
    assert tuple(ag.q.shape) == (N, 81, 8)
    out = ag.learn(T, record=True)
    begin = 0
    for cfg, n, sl in zip(GROUPS, GSIZES, het.group_slices):
        one = make_env(n, autoreset=True, horizon=15, philox_seed=5,
                       env_id_offset=begin, **cfg)
        ag1 = learner(one, epsilon=0.3)
        ref = ag1.learn(T, record=True)
        S = ag1.q.shape[1]
        assert torch.equal(ag.q[sl, :S], ag1.q)
        assert not ag.q[sl, S:].any()
        for k in ref:
            assert torch.equal(out[k][:, sl], ref[k]), k
        for t in ("ep_return", "ret_sum", "ret_count"):
            assert torch.equal(getattr(ag, t)[sl], getattr(ag1, t)), t
        begin += n
    ret = ag.episode_returns()
    assert ret["episodes"].shape == (4,) and (ret["episodes"] > 0).all()


def test_two_shards_equal_the_unsplit_job():
    T = 70
    full = make_env(sum(GSIZES), autoreset=True, horizon=15, philox_seed=9,
                    config_groups=GROUPS, group_sizes=GSIZES)
    agf = learner(full, epsilon=0.3)
    agf.learn(T)
    half = [n // 2 for n in GSIZES]
    for r in range(2):
        sh = make_env(sum(half), autoreset=True, horizon=15, philox_seed=9,
                      config_groups=GROUPS, group_sizes=half, shard=(r, 2))
        ag = learner(sh, epsilon=0.3)
        ag.learn(T)
        for sl_f, sl_s, n in zip(full.group_slices, sh.group_slices, half):
            part = slice(sl_f.start + r * n, sl_f.start + (r + 1) * n)
            assert torch.equal(agf.q[part], ag.q[sl_s])
            assert torch.equal(agf.ret_sum[part], ag.ret_sum[sl_s])


# -- it learns -------------------------------------------------------------------
def optimal_q(shape, target, gamma, iters=500):
    """Value iteration over the cells [0, shape_k] of a noise-free dense 2-D
    grid: every action row is a valid move (the no-op too), so the cell is
    clamped into the grid; reaching the target ends the episode."""
    cells = [(x, y) for x in range(shape[0] + 1) for y in range(shape[1] + 1)]
    rows = gqo.action_rows(2)
    S, A = len(cells), len(rows)
    nxt = np.zeros((S, A), dtype=np.int64)
    r = np.zeros((S, A))
    done = np.zeros((S, A), dtype=bool)
    tx, ty = target
    for s, (x, y) in enumerate(cells):
        for a, (dx, dy) in enumerate(rows):
            nx = min(max(x + dx, 0), shape[0] - 1)
            ny = min(max(y + dy, 0), shape[1] - 1)
            nxt[s, a] = gqo.cell_index([nx, ny], shape)
            r[s, a] = (abs(x - tx) + abs(y - ty)) - (abs(nx - tx) + abs(ny - ty))
            done[s, a] = (nx, ny) == (tx, ty)
    q = np.zeros((S, A))
    for _ in range(iters):
        q = r + gamma * np.where(done, 0.0, q.max(axis=1)[nxt])
    return q


def test_it_learns_the_optimal_greedy_policy():
    """After training, the greedy action of every cell an env visited often
    enough to learn it (20 times) is value-iteration optimal, and so is that
    of 99 % of all visited cells."""
    shape, target, gamma = (8, 8), (5, 5), 0.9
    n = 256
    env = make_env(n, autoreset=True, horizon=30, philox_seed=3,
                   **grid(grid_shape=shape, target_point=list(target)))
    ag = learner(env, alpha=0.3, gamma=gamma, epsilon=0.5)
    S = gqo.n_cells(shape)
    visits = torch.zeros(n * S, dtype=torch.int64, device=env.device)
    envs = torch.arange(n, device=env.device)
    for _ in range(100):
        out = ag.learn(2000, record=True)
        cell = out["obs"][..., 0] * (shape[1] + 1) + out["obs"][..., 1]  # [T, N]
        visits.index_add_(0, (envs * S + cell).reshape(-1),
                          torch.ones(cell.numel(), dtype=torch.int64, device=env.device))
    visits = np_(visits).reshape(n, S)
    qstar = optimal_q(shape, target, gamma)
    optimal = qstar >= qstar.max(axis=1, keepdims=True) - 1e-9  # [S, 5]
    greedy = np_(ag.q[:, :, :5].argmax(dim=2))                   # [N, S]
    ok = optimal[np.arange(S)[None, :], greedy]
    seen = visits > 0
    assert seen.sum(axis=1).min() >= S - 1  # (the target only by a reset draw)
    assert ok[visits >= 20].all(), np.argwhere((visits >= 20) & ~ok)[:10]
    assert ok[seen].mean() >= 0.99, ok[seen].mean()


# -- rejections ------------------------------------------------------------------
def test_python_rejections():
    from mdp_playground_b200 import GridQLearner, TabularQLearner
    disc = dict(seed=7, state_space_type="discrete", action_space_type="discrete",
                state_space_size=8, action_space_size=5, sequence_length=1, delay=0,
                reward_density=0.25, terminal_state_density=0.25)
    for cfg in (gu.case_config("cont_line_2d"), disc):
        with pytest.raises(ValueError, match="needs a grid env"):
            GridQLearner(make_env(8, **cfg))
    with pytest.raises(ValueError, match="train with GridQLearner"):
        TabularQLearner(make_env(8, **grid()))
    with pytest.raises(ValueError, match="noise='philox'"):
        GridQLearner(make_env(8, noise="replay", **grid()))
    with pytest.raises(ValueError, match="image_representations"):
        GridQLearner(make_env(8, **grid(image_representations=True)))
    with pytest.raises(ValueError, match="alpha"):
        GridQLearner(make_env(8, **grid()), alpha=1.5)
    env = make_env(8, track_history=True, **grid())
    ag = GridQLearner(env)
    with pytest.raises(ValueError, match="epsilon"):
        ag.learn(4, epsilon=-0.1)
    ag.learn(3)
    cells = env.get_augmented_state()["curr_state"].clone()
    bad = cells.clone()
    bad[5] = torch.tensor([6, 0])  # one beyond the one-past column
    env.set_augmented_state(bad)
    with pytest.raises(ValueError, match="outside"):
        ag.learn(3)
    bad[5] = torch.tensor([2, -1])
    env.set_augmented_state(bad)
    with pytest.raises(ValueError, match="outside"):
        ag.learn(3)
    env.reset(options={"init_state": np.tile([[0, 8]], (8, 1))})
    with pytest.raises(ValueError, match="outside"):
        ag.learn(3)
    env.reset(options={"init_state": np.tile([[5, 7]], (8, 1))})  # one past: fine
    ag.learn(3)


def test_c_abi_rejections_leave_the_learner_usable():
    from mdp_playground_b200 import _lib
    env = make_env(64, autoreset=True, philox_seed=2, **grid(transition_noise=0.25))
    twin = make_env(64, autoreset=True, philox_seed=2, **grid(transition_noise=0.25))
    ag, ag_twin = learner(env), learner(twin)
    lib = env._lib

    def call(io=None, qp=None, opts=None, env_=env):
        rc = lib.mdpp_grid_qlearn(
            env_._ctx, C.byref(env_._state), C.byref(io or _lib.GridIO()),
            C.byref(qp), C.byref(opts or env_._opts(8)), env_._stream())
        return rc, lib.mdpp_last_error(env_._ctx).decode()

    def params(**kw):
        qp = _lib.QlearnParams()
        qp.alpha, qp.gamma, qp.epsilon = 0.1, 0.9, 0.1
        qp.q = ag.q.data_ptr()
        qp.q_states, qp.q_actions = ag.q.shape[1], ag.q.shape[2]
        qp.ep_return, qp.ret_sum = ag.ep_return.data_ptr(), ag.ret_sum.data_ptr()
        qp.ret_count = ag.ret_count.data_ptr()
        for k, v in kw.items():
            setattr(qp, k, v)
        return qp

    acts = torch.zeros((8, 64, 2), dtype=torch.int64, device=env.device)
    io = _lib.GridIO()
    io.actions = acts.data_ptr()
    assert call(io=io, qp=params()) == (
        -1, "grid qlearn: io->actions must be NULL (the agent acts)")
    for mode in (_lib.MDPP_NOISE_OFF, _lib.MDPP_NOISE_REPLAY):
        o = env._opts(8)
        o.noise_mode = mode
        assert call(qp=params(), opts=o) == (-1, "grid qlearn: Philox noise only")
    for k in ("q", "ep_return", "ret_sum", "ret_count"):
        assert call(qp=params(**{k: None})) == (
            -1, "qlearn: q, ep_return, ret_sum or ret_count is NULL"), k
    for k, v in (("q_states", 47), ("q_actions", 4)):  # 6 x 8 cells, 5 actions
        assert call(qp=params(**{k: v})) == (
            -1, "qlearn: q_states / q_actions smaller than a group's S / A"), k
    for k, v in (("alpha", 1.5), ("gamma", -0.1), ("epsilon", float("nan")),
                 ("alpha", float("nan"))):
        assert call(qp=params(**{k: v})) == (
            -1, "qlearn: alpha, gamma and epsilon must lie in [0, 1]"), k
    assert call(qp=params(), opts=env._opts(0)) == (-1, "grid qlearn: T must be >= 1")
    huge = make_env(8, **grid(grid_shape=(65536, 65536), target_point=[1, 1]))
    assert call(qp=params(q_states=2**31 - 1), opts=huge._opts(8), env_=huge) == (
        -1, "grid qlearn: a group has more than 2^31 - 1 cells")
    # nothing ran: the learner goes on like its twin
    for a in (ag, ag_twin):
        a.learn(40)
    for t in ("q", "ep_return", "ret_sum", "ret_count"):
        assert torch.equal(getattr(ag, t), getattr(ag_twin, t)), t
    assert torch.equal(env._pos, twin._pos)


# -- Sweep -----------------------------------------------------------------------
def check_csv(sw, path, iterations, steps):
    lines = open(sw.write_csv(path)).read().splitlines()
    assert lines[0].startswith("# training_iteration, algorithm, ")
    rows = [ln.split(" ") for ln in lines[1:]]
    assert len(rows) == iterations * sw.n_cells
    assert [int(r[0]) for r in rows] == [i + 1 for i in range(iterations)
                                         for _ in range(sw.n_cells)]
    assert {r[1] for r in rows} == {"TabularQLearning"}
    ts = np.array([int(r[-3]) for r in rows]).reshape(iterations, sw.n_cells)
    assert (np.diff(ts, axis=0) > 0).all()
    assert (ts[0] == steps * sw.envs_per_cell).all()
    assert all(float(r[-1]) > 0 for r in rows)
    return rows


def test_sweep_train_on_a_grouped_grid_experiment(tmp_path):
    from mdp_playground_b200 import sweep
    sw = quiet(sweep.Sweep, os.path.join(HERE, "fixtures", "grid_noises_like.py"),
               envs_per_cell=16)
    assert len(sw.envs) == 1 and sw.env.n_groups == sw.n_cells
    sw.train_grid(3, 200, alpha=0.2, gamma=0.9, epsilon=0.2)
    rows = check_csv(sw, str(tmp_path / "g.csv"), 3, 200)
    assert all(np.isfinite(float(r[-2])) for r in rows)


IRR_EXPERIMENT = types.ModuleType("grid_irrelevant_like")
IRR_EXPERIMENT.var_env_configs = OrderedDict({
    "irrelevant_features": [False, True],
    "transition_noise": [0, 0.25]})
IRR_EXPERIMENT.env_config = {
    "env": "RLToy-v0", "horizon": 30,
    "env_config": {"seed": 0, "state_space_type": "grid", "grid_shape": (4, 4),
                   "target_point": [2, 2], "reward_function": "move_to_a_point",
                   "make_denser": True, "delay": 0, "sequence_length": 1}}


def test_sweep_train_one_learner_per_cell(tmp_path):
    from mdp_playground_b200 import VectorRLToyEnv, sweep
    sw = quiet(sweep.Sweep, IRR_EXPERIMENT, envs_per_cell=32)
    assert len(sw.envs) == sw.n_cells == 4 and not getattr(sw, "grouped", False)
    res = sw.train_grid(2, 100, alpha=0.2, gamma=0.9, epsilon=0.2, chunk=64)
    check_csv(sw, str(tmp_path / "c.csv"), 2, 100)
    # the per-cell results come in cell order: cell i is an env of its own
    for i, cfg in enumerate(sw.cell_configs):
        env = quiet(VectorRLToyEnv, 32, autoreset=True, horizon=30,
                    env_id_offset=i * 32, **cfg)
        ag = learner(env, alpha=0.2, gamma=0.9, epsilon=0.2)
        for it in range(2):
            ag.episode_returns(clear=True)
            for T in (64, 36):
                ag.learn(T)
            ret = ag.episode_returns()
            np.testing.assert_array_equal(res[it]["episode_reward_mean"][i],
                                          ret["episode_reward_mean"][0])
            assert res[it]["timesteps_total"][i] == env.episode_stats()["transitions"][0]
        assert torch.equal(sw.agents[i].q, ag.q)


def test_sweep_train_grid_rejects_the_other_kinds():
    from mdp_playground_b200 import sweep
    for fixture in ("ddpg_move_to_a_point_images_like.py", "dqn_seq_del_like.py"):
        sw = quiet(sweep.Sweep, os.path.join(HERE, "fixtures", fixture), envs_per_cell=4)
        with pytest.raises(NotImplementedError, match="grid-world experiments only"):
            sw.train_grid(1, 10)
