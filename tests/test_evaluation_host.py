"""The evaluation restatement (tests/eval_oracle.py) is pinned to a plain
per-env loop, the ctypes mirror of mdpp_eval_params matches the header, the
noise-callable probe of the reference's evaluation configs reads sigma, and
Sweep's evaluation settings merge the reference-style eval_config of an
experiment file.  No GPU needed."""
import ctypes as C
import os
import re
import shutil
import subprocess
import warnings

import numpy as np
import pytest

from mdp_playground_b200 import _lib
from mdp_playground_b200.sweep import (env_grid, eval_cell_configs, eval_settings,
                                       load_experiment, noise_std)
from mdp_playground_b200.tables import build_discrete_tables
from mdp_playground_b200.config import parse_config
from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_continuous_oracle import VectorGroupedContinuousOracle
from oracle.vector_grid_oracle import VectorGroupedGridOracle
from oracle.vector_oracle import VectorDiscreteOracle, VectorGroupedOracle
from tests import eval_oracle as eo
from tests import grid_qlearn_oracle as go
from tests.test_image_group_abi import HEADER, header_fields

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "fixtures", "dqn_seq_del_eval_like.py")


def scalar(**c):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ScalarRLToyEnv(**c)


def dcfg(**kw):
    c = dict(seed=3, state_space_type="discrete", action_space_type="discrete",
             state_space_size=8, action_space_size=5, sequence_length=1, delay=0,
             reward_density=0.25, terminal_state_density=0.25)
    c.update(kw)
    return c


def check_pinned(got, E):
    ret_sum, count, len_sum = eo.first_episodes(got["reward"], got["ended"], E)
    assert np.array_equal(got["ret_sum"], ret_sum)
    assert np.array_equal(got["ret_count"], count)
    assert np.array_equal(got["len_sum"], len_sum)
    assert (count == E).all()


@pytest.mark.parametrize("kw", [dict(), dict(sequence_length=2, delay=1,
                                             transition_noise=0.1, reward_noise=0.25)])
def test_discrete_evaluation_is_a_per_env_loop(kw):
    H, E, n = 9, 3, 12
    o = VectorDiscreteOracle(scalar(**dcfg(**kw)), n, autoreset=True, horizon=H, seed=5)
    o.reset()
    q = np.random.default_rng(0).integers(0, 3, (n, 8, 5)).astype(np.float64)
    s0 = o.cur.copy()
    got = eo.evaluate(o, "discrete", q, E, H)
    check_pinned(got, E)
    # greedy from the reset states, lowest index on the seeded ties
    assert np.array_equal(got["actions"][0], np.argmax(q[np.arange(n), s0], axis=1))


def test_grouped_discrete_and_grid_and_continuous_evaluations_are_per_env_loops():
    H, E = 7, 2
    g = VectorGroupedOracle([scalar(**dcfg()), scalar(**dcfg(state_space_size=6,
                                                              action_space_size=4))],
                            [6, 4], autoreset=True, horizon=H, seed=9)
    g.reset()
    q = np.random.default_rng(1).normal(size=(10, 8, 5))
    check_pinned(eo.evaluate(g, "discrete", q, E, H), E)

    gcfg = [dict(seed=0, state_space_type="grid", grid_shape=(4, 4), target_point=[2, 2],
                 terminal_states=[[2, 2]], reward_function="move_to_a_point",
                 make_denser=True),
            dict(seed=1, state_space_type="grid", grid_shape=(3, 5), target_point=[1, 1],
                 terminal_states=[[1, 1]], reward_function="move_to_a_point",
                 make_denser=False)]
    gg = VectorGroupedGridOracle([scalar(**c) for c in gcfg], [4, 6], autoreset=True,
                                 horizon=H, seed=3)
    gg.reset()
    qg = np.random.default_rng(2).integers(0, 2, (10, go.n_cells((4, 4)) + 4, 8)) * 1.0
    check_pinned(eo.evaluate(gg, "grid", qg, E, H), E)

    _, cells = env_grid(load_experiment(os.path.join(HERE, "fixtures",
                                                     "ddpg_move_to_a_point_like.py")))
    cc = VectorGroupedContinuousOracle([scalar(**c) for c in cells[:2]], [4, 4],
                                       autoreset=True, horizon=H, seed=4)
    cc.reset()
    th = np.random.default_rng(3).normal(size=(2, 2, 3))
    check_pinned(eo.evaluate(cc, "continuous", th, E, H), E)


def test_first_episodes_counts_only_the_first_E():
    reward = np.array([[1.0], [2.0], [4.0], [8.0], [16.0]])
    ended = np.array([[False], [True], [True], [False], [True]])
    assert [x.tolist() for x in eo.first_episodes(reward, ended, 2)] == [[7.0], [2], [3]]
    assert [x.tolist() for x in eo.first_episodes(reward, ended, 5)] == [[31.0], [3], [5]]


def test_eval_params_binding_matches_the_header():
    assert [f[0] for f in _lib.EvalParams._fields_] == header_fields("mdpp_eval_params")
    for sym in ("mdpp_discrete_qeval", "mdpp_grid_qeval", "mdpp_continuous_ars_eval"):
        assert sym in _lib.EXPORTED_SYMBOLS
        assert re.search(r"\b%s\(" % sym, open(HEADER).read()), sym


@pytest.mark.skipif(shutil.which("cc") is None, reason="needs a C compiler")
def test_eval_params_offsets_match_the_header(tmp_path):
    names = [f[0] for f in _lib.EvalParams._fields_]
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mdpp_b200.h"\n'
                   "int main(void){"
                   + "".join('printf("%%zu\\n", offsetof(mdpp_eval_params, %s));' % n
                             for n in names)
                   + 'printf("%zu\\n", sizeof(mdpp_eval_params)); return 0;}\n')
    exe = tmp_path / "off"
    subprocess.check_call(["cc", "-I", os.path.dirname(HEADER), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [getattr(_lib.EvalParams, n).offset for n in names] + [C.sizeof(_lib.EvalParams)]
    assert got == want


def test_noise_probe_reads_sigma():
    assert noise_std("reward_noise", lambda a: a.normal(0, 0)) == 0.0
    assert noise_std("reward_noise", lambda a: a.normal(0, 0.5)) == 0.5
    assert noise_std("reward_noise", lambda a: a.normal(loc=0, scale=0.5)) == 0.5
    assert isinstance(noise_std("x", lambda a: a.normal(0, 0)), float)


@pytest.mark.parametrize("f", [
    lambda a: a.normal(1, 0.5),            # not centred
    lambda a: a.normal(0, 0.5) * 2,         # arithmetic on the draw
    lambda a: a.normal(0, 0.5) + a.normal(0, 0.5),
    lambda a: a.uniform(0, 1),
    lambda a: 0.0,                          # no draw
    lambda a: a.normal(0, a.normal(0, 1)),  # non-constant sigma
    lambda a: a.normal(0, -1.0),
    lambda a: a.normal(0, 0.5, size=3),
])
def test_noise_probe_rejects_other_callables(f):
    with pytest.raises(NotImplementedError, match="reward_noise"):
        noise_std("reward_noise", f)


def test_eval_settings_merge_the_reference_eval_config():
    mod = load_experiment(FIXTURE)
    st = eval_settings(mod, True, 100)
    assert st["interval"] == 1 and st["episodes"] == 10 and st["horizon"] == 100
    # agent keys dropped, noise callables resolved, the rest passed through
    assert st["env_config"] == {"dummy_eval": True, "transition_noise": 0,
                                "reward_noise": 0.0, "action_loss_weight": 0.0}
    over = eval_settings(mod, {"evaluation_interval": 3, "evaluation_num_episodes": 4,
                               "horizon": 20,
                               "env_config": {"reward_noise": lambda a: a.normal(0, 0.25)}},
                         100)
    assert (over["interval"], over["episodes"], over["horizon"]) == (3, 4, 20)
    assert over["env_config"]["reward_noise"] == 0.25
    assert over["env_config"]["transition_noise"] == 0
    with pytest.raises(ValueError):
        eval_settings(mod, {"evaluation_num_episodes": 0}, 100)
    with pytest.raises(ValueError):
        eval_settings(mod, {"episodes": 3}, 100)
    # a file without eval_config: every iteration, 10 episodes, the sweep's horizon
    plain = eval_settings(load_experiment(os.path.join(HERE, "fixtures",
                                                       "dqn_seq_del_like.py")), True, 50)
    assert (plain["interval"], plain["episodes"], plain["horizon"]) == (1, 10, 50)
    assert plain["env_config"] == {}


def test_eval_cells_keep_the_training_tables():
    mod = load_experiment(FIXTURE)
    keys, cells = env_grid(mod)
    ev = eval_cell_configs(cells, eval_settings(mod, True, 100)["env_config"])
    assert len(ev) == len(cells) == 32
    for c, e in zip(cells, ev):
        assert e["transition_noise"] == 0 and e["reward_noise"] == 0.0
        assert {k: v for k, v in e.items() if k not in ("transition_noise", "reward_noise",
                                                        "dummy_eval", "action_loss_weight")} \
            == {k: v for k, v in c.items() if k not in ("transition_noise", "reward_noise")}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            t, u = build_discrete_tables(parse_config(dict(c))), \
                build_discrete_tables(parse_config(dict(e)))
        for name in ("transition", "terminal_states", "init_cdf", "sequences",
                     "sequence_rewards"):
            assert np.array_equal(getattr(t, name), getattr(u, name)), name
