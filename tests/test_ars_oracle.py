"""The ARS restatement (tests/ars_oracle.py) agrees with a textbook
vectorised ARS update, learns on the batched continuous oracle, and the
ctypes binding of mdpp_ars_params matches the header.  No GPU needed."""
import ctypes as C
import os
import re
import shutil
import subprocess
import warnings

import numpy as np
import pytest

from mdp_playground_b200 import _lib
from mdp_playground_b200.sweep import env_grid, load_experiment
from oracle.scalar_env import ScalarRLToyEnv
from oracle.vector_continuous_oracle import VectorContinuousOracle
from tests import ars_oracle as ao
from tests.test_image_group_abi import HEADER, header_fields

FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fixtures",
                       "ddpg_move_to_a_point_like.py")


def textbook_update(theta, fitness, delta, b, step_size):
    """ARS V1-t step as usually written: argsort, np.std, a matrix product."""
    fp, fm = fitness[0::2], fitness[1::2]
    order = np.argsort(-np.maximum(fp, fm), kind="stable")[:b]
    sigma = np.std(np.concatenate([fp[order], fm[order]]))
    g = (fp[order] - fm[order]) @ delta[order].reshape(b, -1)
    return theta + (step_size / (b * sigma)) * g.reshape(theta.shape)


@pytest.mark.parametrize("n_pairs,b,ties", [(16, 16, False), (16, 5, False),
                                            (12, 4, True), (7, 1, True)])
def test_update_matches_textbook_ars(n_pairs, b, ties):
    rng = np.random.default_rng(n_pairs * 31 + b)
    D = 3
    theta = rng.normal(size=(D, D + 1))
    fitness = rng.normal(size=2 * n_pairs) * 5
    if ties:  # equal maxima across pairs: the lower p wins
        fitness[0::2][:4] = fitness.max() + 1.0
    delta = rng.normal(size=(n_pairs, D, D + 1))
    got, m, sigma, updated = ao.update(theta, fitness, delta, b, 0.05)
    assert updated
    np.testing.assert_allclose(got, textbook_update(theta, fitness, delta, b, 0.05),
                               rtol=1e-12, atol=1e-14)
    order = np.argsort(-np.maximum(fitness[0::2], fitness[1::2]), kind="stable")[:b]
    kept = np.concatenate([fitness[0::2][order], fitness[1::2][order]])
    assert m == pytest.approx(np.mean(kept), rel=1e-12)
    assert sigma == pytest.approx(np.std(kept), rel=1e-12)


def test_update_with_equal_fitness_leaves_theta():
    theta = np.arange(6.0).reshape(2, 3)
    got, m, sigma, updated = ao.update(theta, np.full(8, 0.25), np.ones((4, 2, 3)), 4, 0.1)
    assert not updated and sigma == 0.0 and m == 0.25
    assert np.array_equal(got, theta)


def test_perturbations_follow_the_philox_layout():
    d = ao.perturbations(7, [0, 2, 4], 3, 2)
    assert d.shape == (3, 2, 3)
    from oracle import philox as px
    w = px.philox4x32_10(2, 3, 0, ao.STREAM_ARS_DELTA + 1, 7)
    z = px.normal_pair_f64(w[0], w[1])
    assert d[1].reshape(-1)[4] == z[0] and d[1].reshape(-1)[5] == z[1]
    assert not np.array_equal(d[0], d[1])
    assert not np.array_equal(d, ao.perturbations(7, [0, 2, 4], 4, 2))


def test_policy_actions_round_each_operation_and_clip():
    w = np.array([[[0.5, -0.25, -0.7], [1.0, 1.0, 3.0]]])
    obs = np.array([[np.float32(1.5), np.float32(-2.0)]], dtype=np.float32)
    a = ao.policy_actions(w, obs, np.float32, 1.0)
    assert a.dtype == np.float32
    assert a[0, 0] == np.float32((0.5 * 1.5 + -0.25 * -2.0) + -0.7)
    assert a[0, 1] == np.float32(1.0)  # 1.5 - 2 + 3 = 2.5, clipped
    assert ao.policy_actions(w, obs, np.float32, np.inf)[0, 1] == np.float32(2.5)


def test_ars_learns_on_the_oracle():
    """8 pairs per order-1 cell of ddpg_move_to_a_point_like.py, 10
    iterations of 100 steps (horizon 100), step_size 0.02, noise_std 0.03,
    theta = 0.  Mean return of the episodes ending in each iteration,
    averaged over the 6 cells, as recorded when this test was written:
      -2.24, 0.77, 2.85, 5.48, 5.76, 6.67, 6.61, 6.69, 6.74, 6.87
    (an improvement of 9.1; tests/test_cuda_ars.py asks the device run for
    at least half of it)."""
    _, cells = env_grid(load_experiment(FIXTURE))
    cells = [c for c in cells if c["transition_dynamics_order"] == 1]
    n = 16
    oracles = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for i, c in enumerate(cells):
            o = VectorContinuousOracle(ScalarRLToyEnv(**c), n, autoreset=True,
                                       horizon=100, seed=5, env_id_offset=i * n)
            o.reset()
            oracles.append(o)
    _, curve = ao.run(oracles, [np.zeros((2, 3)) for _ in oracles], 10, 100,
                      0.02, 0.03, 5)
    means = [float(np.nanmean(row)) for row in curve]
    assert means[-1] - means[0] > 8.0, means


def test_ars_params_binding_matches_the_header():
    assert [f[0] for f in _lib.ArsParams._fields_] == header_fields("mdpp_ars_params")
    assert C.sizeof(_lib.ArsParams) == 112
    for sym in ("mdpp_continuous_ars", "mdpp_continuous_ars_update",
                "mdpp_continuous_ars_perturbations"):
        assert sym in _lib.EXPORTED_SYMBOLS
        assert re.search(r"\b%s\(" % sym, open(HEADER).read()), sym
    assert "STREAM_ARS_DELTA = 0x%x," % ao.STREAM_ARS_DELTA in open(
        HEADER.replace("include/mdpp_b200.h", "mdp_playground_b200/csrc/philox.cuh")).read()


@pytest.mark.skipif(shutil.which("cc") is None, reason="needs a C compiler")
def test_ars_params_offsets_match_the_header(tmp_path):
    names = [f[0] for f in _lib.ArsParams._fields_]
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mdpp_b200.h"\n'
                   "int main(void){"
                   + "".join('printf("%%zu\\n", offsetof(mdpp_ars_params, %s));' % n
                             for n in names)
                   + 'printf("%zu\\n", sizeof(mdpp_ars_params)); return 0;}\n')
    exe = tmp_path / "off"
    subprocess.check_call(["cc", "-I", os.path.dirname(HEADER), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [getattr(_lib.ArsParams, n).offset for n in names] + [C.sizeof(_lib.ArsParams)]
    assert got == want
