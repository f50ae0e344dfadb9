"""The Q-learning restatement (tests/qlearn_oracle.py) is pinned to the batched
oracle's rollout and to a plain per-transition update loop, and the ctypes
mirror of mdpp_qlearn_params matches the header.  No GPU needed."""
import ctypes as C
import warnings

import numpy as np
import pytest

from mdp_playground_b200 import _lib
from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_oracle import VectorDiscreteOracle, VectorGroupedOracle
from tests import qlearn_oracle as qo
from tests.test_image_group_abi import HEADER, header_fields


def cfg(**kw):
    c = dict(seed=3, state_space_type="discrete", action_space_type="discrete",
             state_space_size=8, action_space_size=5, sequence_length=1, delay=0,
             reward_density=0.25, terminal_state_density=0.25)
    c.update(kw)
    return c


def scalar(**kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ScalarRLToyEnv(**cfg(**kw))


def twins(n, **kw):
    """Two identical oracles, reset like the env constructor does."""
    out = []
    for _ in range(2):
        o = VectorDiscreteOracle(scalar(**kw), n, autoreset=True, horizon=9, seed=11)
        o.reset()
        out.append(o)
    return out


CONFIGS = [dict(), dict(sequence_length=3, delay=2, transition_noise=0.1,
                        reward_noise=0.25, reward_every_n_steps=True)]


@pytest.mark.parametrize("kw", CONFIGS)
def test_epsilon_one_is_the_random_policy(kw):
    a, b = twins(24, **kw)
    T = 37
    q = np.zeros((24, 8, 5))
    got = qo.qlearn(a, T, alpha=0.5, gamma=0.9, epsilon=1.0, q=q)
    want = b.rollout(T)
    for k in ("obs", "final_obs", "reward", "terminated", "truncated"):
        assert np.array_equal(got[k], want[k]), k
    assert a.stats == b.stats and a.step_index == b.step_index
    assert np.array_equal(a.cur, b.cur) and np.array_equal(a.t, b.t)


@pytest.mark.parametrize("kw", CONFIGS)
@pytest.mark.parametrize("epsilon", [0.0, 0.3, 1.0])
def test_q_equals_a_per_transition_loop(kw, epsilon):
    ora, _ = twins(16, **kw)
    alpha, gamma, T = 0.3, 0.95, 41
    q = np.zeros((16, 8, 5))
    start = ora.cur.copy()
    got = qo.qlearn(ora, T, alpha, gamma, epsilon, q)
    before = np.concatenate([start[None], got["obs"][:-1]])  # state at each step
    ref = np.zeros_like(q)
    ep, rsum, rcnt = np.zeros(16), np.zeros(16), np.zeros(16, dtype=np.int64)
    for t in range(T):
        for i in range(16):
            s, a = int(before[t, i]), int(got["actions"][t, i])
            r, nxt = float(got["reward"][t, i]), int(got["final_obs"][t, i])
            done = bool(got["terminated"][t, i])
            if epsilon == 0.0:  # greedy: the action is the argmax before the update
                assert a == int(np.argmax(ref[i, s]))
            target = r if done else r + gamma * float(np.max(ref[i, nxt]))
            ref[i, s, a] = ref[i, s, a] + alpha * (target - ref[i, s, a])
            ep[i] += r
            if done or got["truncated"][t, i]:
                rsum[i] += ep[i]
                rcnt[i] += 1
                ep[i] = 0.0
    assert np.array_equal(q, ref)
    assert np.array_equal(got["ep_return"], ep)
    assert np.array_equal(got["ret_sum"], rsum)
    assert np.array_equal(got["ret_count"], rcnt)


def test_grouped_qlearn_equals_one_oracle_per_group():
    envs = [scalar(), scalar(state_space_size=6, action_space_size=3, delay=1)]
    sizes = [8, 5]
    g = VectorGroupedOracle(envs, sizes, autoreset=True, horizon=7, seed=5)
    g.reset()
    q = np.zeros((13, 8, 5))
    got = qo.qlearn(g, 23, 0.2, 0.9, 0.2, q)
    begin = 0
    for e, n, base in zip(envs, sizes, (0, 8)):
        o = VectorDiscreteOracle(e, n, autoreset=True, horizon=7, seed=5,
                                 gids=base + np.arange(n))
        o.reset()
        qg = np.zeros((n, 8, 5))
        want = qo.qlearn(o, 23, 0.2, 0.9, 0.2, qg)
        sl = slice(begin, begin + n)
        assert np.array_equal(q[sl], qg)
        for k in ("obs", "reward", "actions"):
            assert np.array_equal(got[k][:, sl], want[k]), k
        begin += n
    # entries beyond group 1's S / A are never touched
    assert not q[8:, 6:, :].any() and not q[8:, :, 3:].any()


def test_qlearn_params_mirror_matches_the_header():
    fields = [f[0] for f in _lib.QlearnParams._fields_]
    assert fields == header_fields("mdpp_qlearn_params")
    assert fields == ["alpha", "gamma", "epsilon", "q", "q_states", "q_actions",
                      "ep_return", "ret_sum", "ret_count", "actions_taken"]
    assert C.sizeof(_lib.QlearnParams) == 3 * 8 + 8 + 2 * 4 + 4 * 8
    assert "mdpp_discrete_qlearn" in _lib.EXPORTED_SYMBOLS
    assert "mdpp_discrete_qlearn(" in open(HEADER).read()
