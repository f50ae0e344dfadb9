"""The grid Q-learning restatement (tests/grid_qlearn_oracle.py) is pinned to
the batched grid oracle's rollout and to a plain per-transition update loop;
its action and state indexing is checked on hand-made cases against the
package's, and the ctypes binding of mdpp_grid_qlearn against the header.
No GPU needed."""
import ctypes as C
import re
import warnings

import numpy as np
import pytest

from mdp_playground_b200 import _lib
from mdp_playground_b200.qlearning import grid_action_rows, grid_cells
from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_grid_oracle import VectorGridOracle, VectorGroupedGridOracle
from tests import grid_qlearn_oracle as gqo
from tests.test_image_group_abi import HEADER


def cfg(**kw):
    c = dict(seed=0, state_space_type="grid", grid_shape=(5, 7), delay=0,
             sequence_length=1, reward_function="move_to_a_point",
             target_point=[3, 4], make_denser=True)
    c.update(kw)
    return c


def scalar(**kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ScalarRLToyEnv(**cfg(**kw))


def oracle(n, horizon=9, **kw):
    o = VectorGridOracle(scalar(**kw), n, autoreset=True, horizon=horizon, seed=11)
    o.reset()
    return o


CONFIGS = [dict(), dict(transition_noise=0.25, make_denser=False),
           dict(irrelevant_features=True, grid_shape=(3, 4), target_point=[1, 2],
                transition_noise=1.0)]


@pytest.mark.parametrize("kw", CONFIGS)
@pytest.mark.parametrize("epsilon", [0.0, 0.3, 1.0])
def test_recorded_rows_replay_on_a_fresh_oracle(kw, epsilon):
    a, b = oracle(20, **kw), oracle(20, **kw)
    T = 45
    q = np.zeros((20, gqo.n_cells(a.shape), 2 * a.nd + 1))
    got = gqo.qlearn(a, T, 0.5, 0.9, epsilon, q)
    want = b.rollout(T, got["actions"])
    for k in ("obs", "final_obs", "reward", "terminated", "truncated"):
        assert np.array_equal(got[k], want[k]), k
    assert a.stats == b.stats and a.step_index == b.step_index == T
    for k in ("pos", "t", "episode", "reached"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k


@pytest.mark.parametrize("kw", CONFIGS)
@pytest.mark.parametrize("epsilon", [0.0, 0.3, 1.0])
def test_q_equals_a_per_transition_loop(kw, epsilon):
    ora = oracle(12, **kw)
    alpha, gamma, T = 0.3, 0.95, 41
    A = 2 * ora.nd + 1
    q = np.zeros((12, gqo.n_cells(ora.shape), 8 if ora.nd == 2 else 9))
    got = gqo.qlearn(ora, T, alpha, gamma, epsilon, q)
    ref = np.zeros_like(q)
    ep, rsum, rcnt = np.zeros(12), np.zeros(12), np.zeros(12, dtype=np.int64)
    for t in range(T):
        for i in range(12):
            s, a = int(got["state"][t, i]), int(got["action_index"][t, i])
            r = float(got["reward"][t, i])
            nxt = int(gqo.cell_index(got["final_obs"][t, i], ora.shape))
            done = bool(got["terminated"][t, i])
            if epsilon == 0.0:  # greedy: the action is the argmax before the update
                assert a == int(np.argmax(ref[i, s, :A]))
            target = r if done else r + gamma * float(np.max(ref[i, nxt, :A]))
            ref[i, s, a] = ref[i, s, a] + alpha * (target - ref[i, s, a])
            ep[i] += r
            if done or got["truncated"][t, i]:
                rsum[i] += ep[i]
                rcnt[i] += 1
                ep[i] = 0.0
    assert np.array_equal(q, ref)
    assert not q[:, :, A:].any()  # the padding entries are never touched
    assert np.array_equal(got["ep_return"], ep)
    assert np.array_equal(got["ret_sum"], rsum)
    assert np.array_equal(got["ret_count"], rcnt)
    if epsilon == 1.0:  # every action is drawn: all indices occur
        assert set(np.unique(got["action_index"]).tolist()) == set(range(A))


def test_grouped_qlearn_equals_one_oracle_per_group():
    envs = [scalar(), scalar(grid_shape=(4, 4), target_point=[1, 1],
                             transition_noise=0.5)]
    sizes = [7, 5]
    g = VectorGroupedGridOracle(envs, sizes, autoreset=True, horizon=6, seed=5)
    g.reset()
    q = np.zeros((12, 48, 8))
    got = gqo.qlearn(g, 23, 0.2, 0.9, 0.2, q)
    begin = 0
    for e, n in zip(envs, sizes):
        o = VectorGridOracle(e, n, autoreset=True, horizon=6, seed=5, env_id_offset=begin)
        o.reset()
        qg = np.zeros((n, 48, 8))
        want = gqo.qlearn(o, 23, 0.2, 0.9, 0.2, qg)
        sl = slice(begin, begin + n)
        assert np.array_equal(q[sl], qg)
        for k in ("obs", "reward", "actions"):
            assert np.array_equal(got[k][:, sl], want[k]), k
        begin += n
    assert not q[7:, 25:].any()  # beyond the 5 x 5 cells of group 1


def test_action_rows_and_cell_index_by_hand():
    two = [[0, 0], [-1, 0], [1, 0], [0, -1], [0, 1]]
    assert gqo.action_rows(2).tolist() == two
    assert grid_action_rows(2).tolist() == two
    four = gqo.action_rows(4)
    assert four.shape == (9, 4) and four[0].tolist() == [0, 0, 0, 0]
    assert four[7].tolist() == [0, 0, 0, -1] and four[6].tolist() == [0, 0, 1, 0]
    assert np.array_equal(four, grid_action_rows(4))
    # every row is a distinct GridActionSpace member (values in {-1, 0, 1},
    # at most one move)
    assert len({tuple(r) for r in four}) == 9 and (np.abs(four).sum(axis=1) <= 1).all()
    # 5 x 7: 6 x 8 cells, one past the grid included
    assert gqo.n_cells((5, 7)) == grid_cells((5, 7)) == 48
    assert gqo.cell_index([0, 0], (5, 7)) == 0
    assert gqo.cell_index([0, 7], (5, 7)) == 7      # one past in y
    assert gqo.cell_index([1, 0], (5, 7)) == 8
    assert gqo.cell_index([5, 7], (5, 7)) == 47     # one past in both
    assert gqo.n_cells((8, 8)) == 81
    # 4-D (irrelevant_features): 4 x 5 x 4 x 5 cells
    assert gqo.n_cells((3, 4, 3, 4)) == grid_cells((3, 4, 3, 4)) == 400
    assert gqo.cell_index([1, 2, 3, 4], (3, 4, 3, 4)) == ((1 * 5 + 2) * 4 + 3) * 5 + 4
    assert gqo.cell_index([3, 4, 3, 4], (3, 4, 3, 4)) == 399
    cells = np.array([[a, b] for a in range(6) for b in range(8)])
    assert gqo.cell_index(cells, (5, 7)).tolist() == list(range(48))


def test_grid_qlearn_binding_matches_the_header():
    assert "mdpp_grid_qlearn" in _lib.EXPORTED_SYMBOLS
    text = re.sub(r"\s+", " ", open(HEADER).read())
    decl = re.search(r"int mdpp_grid_qlearn\((.*?)\);", text)
    assert decl, "mdpp_grid_qlearn is not declared"
    params = [p.strip() for p in decl.group(1).split(",")]
    assert params == ["mdpp_ctx* ctx", "const mdpp_grid_state* st",
                      "const mdpp_grid_io* io", "const mdpp_qlearn_params* qp",
                      "const mdpp_step_opts* opts", "void* cuda_stream"]
    lib = _lib.load()
    P = C.c_void_p
    want = [P, C.POINTER(_lib.GridState), C.POINTER(_lib.GridIO),
            C.POINTER(_lib.QlearnParams), C.POINTER(_lib.StepOpts), P]
    assert list(lib.mdpp_grid_qlearn.argtypes) == want
    assert "STREAM_GRID_ACTION = %d," % gqo.STREAM_GRID_ACTION in open(
        HEADER.replace("include/mdpp_b200.h",
                       "mdp_playground_b200/csrc/philox.cuh")).read()
