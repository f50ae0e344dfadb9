"""GPU tests of tabular Q-learning in the discrete rollout kernel
(mdpp_discrete_qlearn, mdp_playground_b200/qlearning.py, Sweep.train)."""
import ctypes as C
import os
import warnings

import numpy as np
import pytest
import torch

from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_oracle import VectorDiscreteOracle
from tests import golden_util as gu
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
    from mdp_playground_b200 import TabularQLearner
    return TabularQLearner(env, **k)


def base(**kw):
    c = dict(seed=7, state_space_type="discrete", action_space_type="discrete",
             state_space_size=8, action_space_size=5, sequence_length=1, delay=0,
             reward_density=0.25, terminal_state_density=0.25)
    c.update(kw)
    return c


# (config, normal_precision, oracle normal kwargs, autoreset horizon)
NORMALS = {"ziggurat": {}, "boxmuller": {"normal": "boxmuller"},
           "fast": {"fast_normal": True}}
CASES = {
    "plain": (base(), "ziggurat", 9),
    "delay2_seq3_pnoise": (base(delay=2, sequence_length=3, transition_noise=0.1,
                                reward_every_n_steps=True), "ziggurat", 12),
    "delay5": (base(delay=5, sequence_length=3), "ziggurat", 0),
    "delay17": (base(delay=17, transition_noise=0.2), "ziggurat", 25),
    "rnoise_zig": (base(delay=2, reward_noise=0.25), "ziggurat", 9),
    "rnoise_f64": (base(sequence_length=3, reward_noise=0.25), "boxmuller", 9),
    "rnoise_fast": (base(delay=1, reward_noise=0.25, transition_noise=0.1), "fast", 9),
    "scale_shift_term": (base(reward_scale=2.5, reward_shift=-0.5,
                              term_state_reward=1.5), "ziggurat", 9),
    "custom_mdp": (gu.case_config("custom_8x5"), "ziggurat", 9),
}


def pair(name, n):
    cfg, normal, horizon = CASES[name]
    env = make_env(n, autoreset=True, horizon=horizon, normal_precision=normal,
                   track_history=True, **cfg)
    ora = VectorDiscreteOracle(quiet(ScalarRLToyEnv, **cfg), n, autoreset=True,
                               horizon=horizon, seed=env.philox_seed,
                               **NORMALS[normal])
    ora.reset()  # mirrors the reset at the end of the env constructor
    assert np.array_equal(env._cur.cpu().numpy(), ora.cur)
    return env, ora


def np_(t):
    return t.cpu().numpy()


# -- epsilon = 1 is the random policy -----------------------------------------
@pytest.mark.parametrize("name", ["plain", "delay2_seq3_pnoise", "delay17", "rnoise_zig"])
def test_epsilon_one_equals_the_random_rollout(name):
    cfg, normal, horizon = CASES[name]
    n = 200
    a = make_env(n, autoreset=True, horizon=horizon, normal_precision=normal,
                 track_history=True, **cfg)
    b = make_env(n, autoreset=True, horizon=horizon, normal_precision=normal,
                 track_history=True, **cfg)
    ag = learner(a, alpha=0.5, gamma=0.9, epsilon=1.0)
    for T in (3, 107, 14):
        got = ag.learn(T, record=True)
        want = b.rollout(T)
        for k in ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(got[k], want[k]), (T, k)
    _, ora = pair(name, n)
    ora_acts = qo.qlearn(ora, 124, 0.5, 0.9, 1.0, np.zeros((n, 8, 5)))["actions"]
    assert np.array_equal(np_(got["actions"]), ora_acts[-14:])
    sa, sb = a.get_augmented_state(), b.get_augmented_state()
    assert torch.equal(sa["curr_state"], sb["curr_state"])
    assert torch.equal(sa["augmented_state"].nan_to_num(-1), sb["augmented_state"].nan_to_num(-1))
    for t in ("_key", "_t", "_episode", "_ring", "_history"):
        x, y = getattr(a, t), getattr(b, t)
        assert (x is None and y is None) or torch.equal(x, y), t
    sta, stb = a.episode_stats(), b.episode_stats()
    for k in sta:
        assert np.array_equal(sta[k], stb[k]), k


# -- CUDA against the oracle ---------------------------------------------------
@pytest.mark.parametrize("epsilon", [0.0, 0.1, 1.0])
@pytest.mark.parametrize("name", list(CASES))
def test_qlearn_matches_the_oracle(name, epsilon):
    n = 96
    env, ora = pair(name, n)
    ag = learner(env, alpha=0.3, gamma=0.95, epsilon=epsilon)
    q = np.zeros(tuple(ag.q.shape))
    acc = qo.new_accumulators(n)
    noisy = CASES[name][0].get("reward_noise")
    fast = CASES[name][1] == "fast"
    # 107 steps from step 0: full chunks and a tail; 14 more from step 107: a
    # peel, a full chunk, a half chunk and a tail
    for T in (107, 14):
        got = ag.learn(T, record=True)
        want = qo.qlearn(ora, T, 0.3, 0.95, epsilon, q, acc)
        for k in ("obs", "terminated", "truncated", "actions"):
            assert np.array_equal(np_(got[k]), want[k]), (T, k)
        if noisy:
            tol = 1e-5 if fast else 1e-12
            np.testing.assert_allclose(np_(got["reward"]), want["reward"],
                                       rtol=tol, atol=tol)
        else:
            assert np.array_equal(np_(got["reward"]), want["reward"])
    if noisy:
        np.testing.assert_allclose(np_(ag.q), q, rtol=1e-9, atol=1e-9 if not fast else 1e-5)
        np.testing.assert_array_equal(np_(ag.ret_count), acc["ret_count"])
    else:
        assert np.array_equal(np_(ag.q), q)
        assert np.array_equal(np_(ag.ep_return), acc["ep_return"])
        assert np.array_equal(np_(ag.ret_sum), acc["ret_sum"])
        assert np.array_equal(np_(ag.ret_count), acc["ret_count"])
    assert np.array_equal(np_(env._cur), ora.cur)


def test_no_outputs_and_overrides():
    env, ora = pair("delay2_seq3_pnoise", 128)
    ag = learner(env, alpha=0.3, gamma=0.95, epsilon=0.2)
    q = np.zeros(tuple(ag.q.shape))
    assert ag.learn(50) is None
    qo.qlearn(ora, 50, 0.3, 0.95, 0.2, q)
    assert np.array_equal(np_(ag.q), q)
    # greedy evaluation leaves q as it is
    before = ag.q.clone()
    out = ag.learn(20, record=True, epsilon=0.0, alpha=0.0)
    assert torch.equal(ag.q, before)
    want = qo.qlearn(ora, 20, 0.0, 0.95, 0.0, q)
    assert np.array_equal(np_(out["actions"]), want["actions"])


# -- invariances ---------------------------------------------------------------
def test_one_launch_equals_two():
    cfg, normal, horizon = CASES["rnoise_zig"]
    envs = [make_env(256, autoreset=True, horizon=horizon, **cfg) for _ in range(2)]
    ags = [learner(e, epsilon=0.2) for e in envs]
    ags[0].learn(301)
    ags[1].learn(118)
    ags[1].learn(183)
    for t in ("q", "ep_return", "ret_sum", "ret_count"):
        assert torch.equal(getattr(ags[0], t), getattr(ags[1], t)), t
    assert torch.equal(envs[0]._cur, envs[1]._cur)
    assert envs[0]._step_index == envs[1]._step_index == 301


GROUPS = [base(), base(state_space_size=6, action_space_size=3, delay=2),
          base(sequence_length=3, transition_noise=0.1),
          base(state_space_size=12, action_space_size=7, delay=17, seed=2)]
GSIZES = [64, 96, 32, 128]


def test_grouped_launch_equals_one_env_per_group():
    N, T = sum(GSIZES), 90
    het = make_env(N, autoreset=True, horizon=15, philox_seed=5,
                   config_groups=GROUPS, group_sizes=GSIZES)
    ag = learner(het, epsilon=0.3)
    S = max(t.n_states for t in het.group_tables)
    A = max(t.n_actions for t in het.group_tables)
    assert tuple(ag.q.shape) == (N, S, A)
    out = ag.learn(T, record=True)
    begin = 0
    for cfg, n, sl in zip(GROUPS, GSIZES, het.group_slices):
        one = make_env(n, autoreset=True, horizon=15, philox_seed=5,
                       env_id_offset=begin, **cfg)
        ag1 = learner(one, epsilon=0.3)
        ref = ag1.learn(T, record=True)
        S, A = ag1.q.shape[1:]
        assert torch.equal(ag.q[sl, :S, :A], ag1.q)
        assert not ag.q[sl, S:].any() and not ag.q[sl, :, A:].any()
        for k in ref:
            assert torch.equal(out[k][:, sl], ref[k]), k
        for t in ("ep_return", "ret_sum", "ret_count"):
            assert torch.equal(getattr(ag, t)[sl], getattr(ag1, t)), t
        begin += n
    # per-group returns
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


# -- it learns -----------------------------------------------------------------
def optimal_q(ora, gamma, iters=2000):
    """Value iteration over the env's own P, rewards and terminal states
    (sequence_length 1, no delay, no noise: the reward of (s, a) is that of
    reaching s' = P[s, a]); terminal states cut the target."""
    S, A = ora.S, ora.A
    nxt = ora.P
    r = np.array([[ora.seq.get((int(nxt[s, a]),), 0.0) for a in range(A)]
                  for s in range(S)])
    done = ora.term[nxt]
    r = r * ora.scale + ora.shift + np.where(done, ora.term_reward * ora.scale, 0.0)
    q = np.zeros((S, A))
    for _ in range(iters):
        q = r + gamma * np.where(done, 0.0, q.max(axis=1)[nxt])
    return q


def reachable(ora):
    init = np.diff(np.concatenate([[0.0], ora.init_cdf[:ora.S]])) > 0
    seen, todo = set(np.nonzero(init)[0].tolist()), list(np.nonzero(init)[0])
    while todo:
        s = int(todo.pop())
        if ora.term[s]:
            continue  # the episode ends there
        for s2 in ora.P[s]:
            if int(s2) not in seen:
                seen.add(int(s2))
                todo.append(int(s2))
    return sorted(seen)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_it_learns_the_optimal_greedy_policy(seed):
    cfg = base(seed=seed, action_space_size=4, reward_density=0.25,
               terminal_state_density=0.25)
    gamma = 0.9
    env = make_env(1024, autoreset=True, horizon=20, **cfg)
    ag = learner(env, alpha=0.1, gamma=gamma, epsilon=0.5)
    for _ in range(4):
        ag.learn(5000)
    ora = VectorDiscreteOracle(quiet(ScalarRLToyEnv, **cfg), 1)
    qstar = optimal_q(ora, gamma)
    states = [s for s in reachable(ora) if not ora.term[s]]
    srt = np.sort(qstar, axis=1)
    unique = [s for s in states if srt[s, -1] - srt[s, -2] > 1e-6]
    assert unique, "no state with a unique optimal action"
    best = qstar[unique].argmax(axis=1)
    greedy = np_(ag.q[:, unique, :ora.A].argmax(dim=2))
    ok = (greedy == best[None, :]).all(axis=1)
    assert ok.mean() >= 0.95, ok.mean()


# -- rejections ----------------------------------------------------------------
def test_python_rejections():
    from mdp_playground_b200 import TabularQLearner
    for case in ("cont_line_2d", "grid_dense_term"):
        with pytest.raises(ValueError, match="discrete env"):
            TabularQLearner(make_env(8, **gu.case_config(case)))
    with pytest.raises(ValueError, match="noise='philox'"):
        TabularQLearner(make_env(8, noise="replay", **base()))
    with pytest.raises(ValueError, match="irrelevant_features"):
        TabularQLearner(make_env(8, **gu.case_config("irr_8x5_det")))
    with pytest.raises(ValueError, match="image_representations"):
        TabularQLearner(make_env(8, **base(image_representations=True)))
    env = make_env(8, **base())
    with pytest.raises(ValueError, match="alpha"):
        TabularQLearner(env, alpha=1.5)
    with pytest.raises(ValueError, match="epsilon"):
        TabularQLearner(env).learn(4, epsilon=-0.1)


def test_c_abi_rejections():
    from mdp_playground_b200 import _lib
    env = make_env(64, autoreset=True, **base())
    ag = learner(env)
    lib = env._lib

    def call(st=None, io=None, qp=None, opts=None, env_=env):
        rc = lib.mdpp_discrete_qlearn(
            env_._ctx, C.byref(st or env_._state), C.byref(io or _lib.DiscreteIO()),
            C.byref(qp), C.byref(opts or env_._opts(8)), env_._stream())
        msg = lib.mdpp_last_error(env_._ctx).decode()
        return rc, msg

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

    assert call(qp=params())[0] == 0
    acts = torch.zeros((8, 64), dtype=torch.int32, device=env.device)
    io = _lib.DiscreteIO()
    io.actions = acts.data_ptr()
    assert call(io=io, qp=params()) == (
        -1, "qlearn: io->actions must be NULL (the agent acts)")
    o = env._opts(8)
    o.noise_mode = _lib.MDPP_NOISE_OFF
    assert call(qp=params(), opts=o) == (-1, "qlearn: Philox noise only")
    for k in ("q", "ep_return", "ret_sum", "ret_count"):
        assert call(qp=params(**{k: None})) == (
            -1, "qlearn: q, ep_return, ret_sum or ret_count is NULL"), k
    for k in ("q_states", "q_actions"):
        assert call(qp=params(**{k: 2})) == (
            -1, "qlearn: q_states / q_actions smaller than a group's S / A"), k
    for k, v in (("alpha", 1.5), ("gamma", -0.1), ("epsilon", float("nan"))):
        assert call(qp=params(**{k: v})) == (
            -1, "qlearn: alpha, gamma and epsilon must lie in [0, 1]"), k
    irr = make_env(64, **gu.case_config("irr_8x5_det"))
    assert call(qp=params(), env_=irr) == (
        -1, "qlearn: irrelevant features are not supported")


# -- Sweep ---------------------------------------------------------------------
FIXTURE = os.path.join(HERE, "fixtures", "dqn_seq_del_like.py")


def test_sweep_train_writes_learning_curves(tmp_path):
    from mdp_playground_b200 import sweep
    sw = quiet(sweep.Sweep, FIXTURE, envs_per_cell=64)
    res = sw.train(3, 200, alpha=0.2, gamma=0.9, epsilon=0.2)
    assert len(res) == 3
    lines = open(sw.write_csv(str(tmp_path / "q.csv"))).read().splitlines()
    assert lines[0].startswith("# training_iteration, algorithm, ")
    rows = [ln.split(" ") for ln in lines[1:]]
    assert len(rows) == 3 * sw.n_cells
    assert [int(r[0]) for r in rows] == [i for i in (1, 2, 3) for _ in range(sw.n_cells)]
    assert {r[1] for r in rows} == {"TabularQLearning"}
    ts = np.array([int(r[-3]) for r in rows]).reshape(3, sw.n_cells)
    assert (np.diff(ts, axis=0) > 0).all()
    assert (ts[0] == 200 * 64).all()
    assert all(np.isfinite(float(r[-2])) and float(r[-1]) > 0 for r in rows)
    with pytest.raises(NotImplementedError):
        quiet(sweep.Sweep, os.path.join(HERE, "fixtures", "grid_noises_like.py"),
              envs_per_cell=8).train(1, 10)


def test_sweep_without_train_writes_what_it_wrote_before(tmp_path):
    from mdp_playground_b200 import sweep
    rows = []
    for algo in ({}, {"algorithm": "RandomPolicy"}):
        sw = quiet(sweep.Sweep, FIXTURE, envs_per_cell=64, philox_seed=3)
        sw.run(100)
        rows.append(open(sw.write_csv(str(tmp_path / "r.csv"), **algo)).read())
    assert rows[0] == rows[1]
    lines = rows[0].splitlines()
    assert len(lines) == 1 + sw.n_cells
    assert all(ln.split(" ")[:2] == ["1", "RandomPolicy"] for ln in lines[1:])
