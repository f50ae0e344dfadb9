"""GPU tests of the state a VectorRLToyEnv carries from one call to the next:
the host step index (which picks the delay-ring, history and line-window
slots), the ring and history buffers, the Philox key and episode counters,
and the staging buffers of rollout_host().  Every other GPU test builds a
fresh env, resets it once and rolls forward; these tests reseed, reset
subsets, set states and move the step index between launches, and check the
result against a twin env or the batched oracle.  Observations, flags and
states are compared bit for bit, fp64 rewards to 1e-12."""
import numpy as np
import pytest
import torch

from oracle.vector_continuous_oracle import VectorContinuousOracle
from oracle.vector_grid_oracle import VectorGridOracle
from oracle.vector_oracle import VectorDiscreteOracle
from tests import golden_util as gu
from tests.test_cuda_discrete import _BENCH_CFG, make_env, scalar_oracle

pytestmark = pytest.mark.gpu

# noise-free discrete MDP: two twins given the same actions stay identical
_CLEAN = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
              state_space_size=8, action_space_size=8, reward_density=0.25,
              terminal_state_density=0.0, generate_random_mdp=True,
              sequence_length=3, reward_every_n_steps=2)
_OUTS = ("obs", "reward", "terminated", "truncated")


def _off_phase(after, moduli):
    """The first step index > `after` that is a multiple of none of `moduli`
    (a rewind to 0 there moves every slot these moduli index)."""
    s = after + 1
    while any(s % m == 0 for m in moduli if m > 1):
        s += 1
    return s


def _np(x):
    return x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def _assert_same(a, b, what):
    """Bit-exact, NaN == NaN."""
    a, b = _np(a), _np(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(a, b, equal_nan=a.dtype.kind == "f"), what


# ---------------------------------------------------------------------------
# 1. reseeding leaves the envs it does not reset where they were
# ---------------------------------------------------------------------------
def _roll(env, acts, fast):
    if not fast:
        return env.rollout(acts.shape[0], actions=acts)
    T, N = acts.shape[:2]
    dev = acts.device
    out = {"obs": torch.empty((T, N), dtype=torch.int64, device=dev),
           "reward": torch.empty((T, N), dtype=torch.float64, device=dev),
           "terminated": torch.empty((T, N), dtype=torch.bool, device=dev),
           "truncated": torch.empty((T, N), dtype=torch.bool, device=dev)}
    return env.rollout(T, actions=acts, out=out)   # the FAST signature


def _reseed_twins(A, B, moduli, acts, fast=False):
    """Roll both twins; reseed A off phase with seed(), then with a
    reset(seed, mask) sparing about 3/4 of the envs, and roll on.  The
    spared envs of A must match B in every output and, with history on, in
    the augmented state.  Returns how many nonzero rewards the spared envs
    were paid after the first reseed (the test has teeth only if some are)."""
    N = A.num_envs
    rng = np.random.default_rng(sum(moduli))
    spared = np.ones(N, dtype=bool)
    t, paid = 0, 0

    def compare(ra=None, rb=None):
        for k in (ra or {}):
            _assert_same(_np(ra[k])[:, spared], _np(rb[k])[:, spared], k)
        if A._history is not None:
            _assert_same(_np(A.get_augmented_state()["augmented_state"])[spared],
                         _np(B.get_augmented_state()["augmented_state"])[spared],
                         "augmented_state")
    for op in ("seed", "masked_reset", None):
        stop = _off_phase(t + 2, moduli) if op else acts.shape[0]
        while t < stop:     # launches of uneven length
            n = min(stop - t, 1 + (t % 5))
            ra, rb = _roll(A, acts[t:t + n], fast), _roll(B, acts[t:t + n], fast)
            compare(ra, rb)
            if A.philox_seed != B.philox_seed:
                paid += int((_np(ra["reward"])[:, spared] != 0).sum())
            t += n
        if op == "seed":
            A.seed(1234)
        elif op == "masked_reset":
            m = rng.random(N) < 0.25
            A.reset(seed=99, options={"mask": m})
            spared &= ~m
        compare()
    assert A._step_index == B._step_index == acts.shape[0]
    assert spared.sum() >= N // 2
    return paid


@pytest.mark.parametrize("delay,jit,fast", [
    (1, True, True), (1, False, False), (2, True, False), (2, False, True),
    (3, True, True), (3, False, False), (5, True, False), (5, False, True),
    (17, True, True), (17, False, False)])
def test_reseed_keeps_unreset_envs_in_phase_discrete(delay, jit, fast):
    """seed(s) and reset(seed=s, mask) at a step index off every ring phase
    (delay, history depth L + d + 1, L, reward_every_n_steps): the envs that
    were not reset go on exactly like a twin that was never reseeded --
    delayed rewards in order, same augmented state.  delay 17 takes the
    global-memory ring (deeper than the shared-memory one)."""
    N = 131
    A, B = [make_env(N, philox_seed=7, track_history=not fast, delay=delay,
                     **dict(_CLEAN)) for _ in range(2)]
    for e in (A, B):
        e.set_jit(jit)
    acts = torch.randint(0, 8, (60, N), dtype=torch.int32, device="cuda",
                         generator=torch.Generator("cuda").manual_seed(delay))
    assert _reseed_twins(A, B, (delay, 3 + delay + 1, 3, 2), acts, fast) > 20
    # (a ring deeper than 16 never fits shared memory: no specialised kernel)
    assert A.jit_last_used == (jit and delay <= 16), A.jit_log


@pytest.mark.parametrize("jit", [True, False])
def test_reseed_keeps_unreset_envs_in_phase_two_groups(jit):
    """One launch of two config groups with delays 2 and 3: the ring phase is
    step mod the group's own delay."""
    N = 130
    envs = [make_env(N, philox_seed=7, config_groups=[dict(delay=2), dict(delay=3)],
                     **dict(_CLEAN)) for _ in range(2)]
    for e in envs:
        e.set_jit(jit)
    acts = torch.randint(0, 8, (60, N), dtype=torch.int32, device="cuda",
                         generator=torch.Generator("cuda").manual_seed(23))
    assert _reseed_twins(*envs, (2, 3, 2), acts) > 20


_POINT = dict(seed=0, state_space_type="continuous", action_space_type="continuous",
              state_space_dim=2, action_space_dim=2, transition_dynamics_order=1,
              inertia=1.0, time_unit=1.0, target_point=[0.0, 0.0],
              state_space_max=5.0, action_space_max=1.0, delay=3,
              reward_function="move_to_a_point", make_denser=True)
_LINE = dict(seed=0, state_space_type="continuous", action_space_type="continuous",
             state_space_dim=2, action_space_dim=2, transition_dynamics_order=1,
             inertia=1.0, time_unit=1.0, delay=0, state_space_max=5.0,
             action_space_max=1.0, reward_function="move_along_a_line")


@pytest.mark.parametrize("cfg,moduli,jit", [
    (_POINT, (3,), True), (_POINT, (3,), False),
    (dict(_LINE, sequence_length=3), (3,), True),
    (dict(_LINE, sequence_length=5), (5,), False)])
def test_reseed_keeps_unreset_envs_in_phase_continuous(cfg, moduli, jit):
    """The continuous delay ring and the move_along_a_line window (slot =
    step mod L): a reseed off phase changes neither for the spared envs."""
    N = 97
    A, B = [make_env(N, philox_seed=7, **dict(cfg)) for _ in range(2)]
    for e in (A, B):
        e.set_jit(jit)
    acts = (torch.rand((60, N, 2), generator=torch.Generator("cuda").manual_seed(4),
                       device="cuda") * 2 - 1)
    spared = np.ones(N, dtype=bool)
    rng = np.random.default_rng(5)
    t = 0
    for op in ("seed", "masked_reset", None):
        stop = _off_phase(t + 2, moduli) if op else acts.shape[0]
        while t < stop:
            n = min(stop - t, 1 + (t % 4))
            a = acts[t:t + n].clone()   # (the kernels want 16-byte aligned rows)
            ra, rb = A.rollout(n, actions=a), B.rollout(n, actions=a)
            for k in ra:
                _assert_same(_np(ra[k])[:, spared], _np(rb[k])[:, spared], k)
            t += n
        if op == "seed":
            A.seed(1234)
        elif op == "masked_reset":
            m = rng.random(N) < 0.25
            A.reset(seed=99, options={"mask": m})
            spared &= ~m
    assert A._step_index == B._step_index == acts.shape[0]
    assert spared.sum() >= N // 2
    assert float(_np(ra["reward"])[:, spared].std()) > 0


# ---------------------------------------------------------------------------
# 2. reseeding with noise, against the oracle
# ---------------------------------------------------------------------------
def _bench_pair(N, seed=77, **kw):
    env = make_env(N, autoreset=True, horizon=9, philox_seed=seed,
                   track_history=True, **dict(_BENCH_CFG, **kw))
    ora = VectorDiscreteOracle(scalar_oracle(dict(_BENCH_CFG, **kw)), N,
                               autoreset=True, horizon=9, seed=seed)
    ora.reset()  # mirrors the reset at the end of the env constructor
    return env, ora


def _check_oracle(env, ora, got=None, want=None, ctx=""):
    if got is not None:
        for k in want:
            if k not in got:
                continue
            if k == "reward":
                np.testing.assert_allclose(_np(got[k]), want[k], rtol=1e-12,
                                           atol=1e-12, err_msg=ctx)
            else:
                assert np.array_equal(_np(got[k]), want[k]), (k, ctx)
    assert np.array_equal(_np(env._cur), ora.cur), ("cur", ctx)
    assert np.array_equal(_np(env._t), ora.t), ("t", ctx)
    assert np.array_equal(_np(env._episode), ora.episode), ("episode", ctx)
    if env._history is not None:
        aug = _np(env.get_augmented_state()["augmented_state"])
        assert np.array_equal(aug, ora.augmented_state(), equal_nan=True), \
            ("augmented_state", ctx)
    assert env._step_index == ora.step_index, ("step index", ctx)


@pytest.mark.parametrize("delay", [2, 3, 5])
def test_reseed_with_noise_matches_oracle(delay):
    """The bench configuration (P and R noise, fp64 ziggurat, autoreset) with
    seed(), masked reset(seed) and a full reset(seed) off phase: every env,
    reset or not, against VectorDiscreteOracle + reseed."""
    N = 97
    env, ora = _bench_pair(N, delay=delay)
    rng = np.random.default_rng(delay)
    moduli = (delay, 3 + delay + 1, 3)
    for op in ("seed", "masked_reset", "reset", "masked_reset", None):
        stop = _off_phase(env._step_index + 3, moduli)
        while env._step_index < stop:
            n = min(stop - env._step_index, 4)
            a = rng.integers(0, 8, size=(n, N))
            got = env.rollout(n, actions=torch.as_tensor(a, dtype=torch.int32,
                                                           device="cuda"))
            _check_oracle(env, ora, got, ora.rollout(n, actions=a), op)
        s = int(rng.integers(1 << 40))
        if op == "seed":
            env.seed(s)
            ora.reseed(s)
        elif op == "masked_reset":
            m = rng.random(N) < 0.3
            obs, _ = env.reset(seed=s, options={"mask": m})
            ora.reseed(s, mask=m)
            assert np.array_equal(_np(obs), ora.reset(mask=m))
        elif op == "reset":
            obs, _ = env.reset(seed=s)
            ora.reseed(s, rewind=True)
            assert np.array_equal(_np(obs), ora.reset())
            assert env._step_index == 0
        _check_oracle(env, ora, ctx=f"after {op}")


# ---------------------------------------------------------------------------
# 3. random API programs against the oracle
# ---------------------------------------------------------------------------
# (seeds of the programs; a failure prints the seed and the program so far)
PROGRAM_SEEDS = list(range(24))
_PROGRAM_T = (1, 3, 7, 8, 9, 37)


def _run_program(seed, n_ops=40):
    rng = np.random.default_rng(seed)
    N = 97   # ragged against the 64-thread CTA
    env = make_env(N, autoreset=True, horizon=11, philox_seed=seed,
                   track_history=True, step_buffers=2 if seed % 2 == 0 else 0,
                   **dict(_BENCH_CFG, delay=3))
    env.set_jit(seed % 3 == 0)
    ora = VectorDiscreteOracle(scalar_oracle(dict(_BENCH_CFG, delay=3)), N,
                               autoreset=True, horizon=11, seed=seed)
    ora.reset()
    gstep = None
    done = []
    ops = ["step", "rollout", "rollout", "reset_mask", "reset_init",
           "reset_seed_mask", "reset_seed", "seed", "aug_round_trip",
           "aug_bare", "graph", "graph"]
    for i in range(n_ops):
        op = ops[int(rng.integers(len(ops)))]
        mask = rng.random(N) < 0.3
        s = int(rng.integers(1 << 62))
        got = want = None
        if op == "step" or op == "graph":
            a = rng.integers(0, 8, size=N)
            at = torch.as_tensor(a, dtype=torch.int32, device="cuda")
            if op == "graph":
                if gstep is None:
                    gstep = env.make_graphed_step()
                r = gstep(at)
            else:
                r = env.step(at)
            want = {k: v[0] for k, v in ora.rollout(1, actions=a[None]).items()}
            got = dict(zip(_OUTS, r[:4]))
            if "final_obs" in r[4]:
                got["final_obs"] = r[4]["final_obs"]
        elif op == "rollout":
            T = _PROGRAM_T[int(rng.integers(len(_PROGRAM_T)))]
            a = rng.integers(0, 8, size=(T, N))
            op = f"rollout({T})"
            got = env.rollout(T, actions=torch.as_tensor(a, device="cuda"))
            want = ora.rollout(T, actions=a)
        elif op == "reset_mask":
            got, want = {"obs": env.reset(options={"mask": mask})[0]}, \
                {"obs": ora.reset(mask=mask)}
        elif op == "reset_init":
            init = rng.integers(0, 8, size=N)
            got = {"obs": env.reset(options={"mask": mask, "init_state": init})[0]}
            want = {"obs": ora.reset(mask=mask, init_state=init)}
        elif op == "reset_seed_mask":
            got = {"obs": env.reset(seed=s, options={"mask": mask})[0]}
            ora.reseed(s, mask=mask)
            want = {"obs": ora.reset(mask=mask)}
            gstep = None
        elif op == "reset_seed":
            got = {"obs": env.reset(seed=s)[0]}
            ora.reseed(s, rewind=True)
            want = {"obs": ora.reset()}
            gstep = None
        elif op == "seed":
            env.seed(s)
            ora.reseed(s)
            gstep = None
        elif op == "aug_round_trip":
            env.set_augmented_state(env.get_augmented_state())
        elif op == "aug_bare":
            st = rng.integers(0, 8, size=N)
            env.set_augmented_state(torch.as_tensor(st, device="cuda"))
            ora.set_state(st)
        done.append(op)
        try:
            _check_oracle(env, ora, got, want, op)
        except AssertionError as e:
            raise AssertionError(f"program seed {seed}, ops {done}: {e}") from e
    return done


@pytest.mark.parametrize("seed", PROGRAM_SEEDS)
def test_random_api_program_matches_oracle(seed):
    """~40 random calls of step (rotating buffers or not), rollout(T),
    reset (mask / init_state / seed), seed(), set_augmented_state and a
    graphed step (re-captured after a reseed), each checked against the
    oracle: N = 97, delay 3, sequence_length 3, both noises, history on."""
    _run_program(seed)


# ---------------------------------------------------------------------------
# 4. the step index past 2^32 (Philox counter words split across two words)
# ---------------------------------------------------------------------------
_BIG_STEPS = [2**32 - 5, 2**33 + 3]


@pytest.mark.parametrize("jit", [True, False])
@pytest.mark.parametrize("step0", _BIG_STEPS)
def test_step_index_beyond_32_bits_discrete(step0, jit):
    """fp64 ziggurat (its rejected draws retry with counter = step), P and R
    noise and autoreset across the 2^32 boundary: against the oracle."""
    N = 512
    env, ora = _bench_pair(N, seed=3)
    env.set_jit(jit)
    env._step_index = ora.step_index = step0
    _check_oracle(env, ora, {"obs": env.reset()[0]}, {"obs": ora.reset()})
    a = np.random.default_rng(1).integers(0, 8, size=(20, N))
    got = env.rollout(20, actions=torch.as_tensor(a, device="cuda"))
    _check_oracle(env, ora, got, ora.rollout(20, actions=a))
    assert env.jit_last_used == jit, env.jit_log


@pytest.mark.parametrize("step0", _BIG_STEPS)
def test_step_index_beyond_32_bits_continuous(step0):
    """Ziggurat transition and reward noise, delay ring, autoreset."""
    name = "cont_noise_delay"
    N = 256
    env = make_env(N, autoreset=True, horizon=7, philox_seed=3,
                   normal_precision="ziggurat", **gu.case_config(name))
    ora = VectorContinuousOracle(scalar_oracle(gu.case_config(name)), N,
                                 autoreset=True, horizon=7, seed=3,
                                 normal="ziggurat")
    ora.reset()
    env._step_index = ora.step_index = step0
    env.reset()
    ora.reset()
    a = np.random.default_rng(2).uniform(-1, 1, size=(20, N, ora.D)).astype(np.float32)
    got = env.rollout(20, actions=torch.as_tensor(a, device="cuda"))
    want = ora.rollout(20, a)
    for k in ("obs", "final_obs"):
        np.testing.assert_allclose(_np(got[k]), want[k], rtol=1e-5, atol=1e-6)
    for k in ("terminated", "truncated"):
        assert np.array_equal(_np(got[k]), want[k]), k
    np.testing.assert_allclose(_np(got["reward"]), want["reward"], rtol=1e-4,
                               atol=1e-5)
    assert want["truncated"].any()


@pytest.mark.parametrize("step0", _BIG_STEPS)
def test_step_index_beyond_32_bits_grid(step0):
    """Transition noise (substitute actions), ziggurat reward noise,
    autoreset."""
    name = "grid_sparse_noise"
    N = 256
    env = make_env(N, autoreset=True, horizon=7, philox_seed=3,
                   normal_precision="ziggurat", **gu.case_config(name))
    ora = VectorGridOracle(scalar_oracle(gu.case_config(name)), N,
                           autoreset=True, horizon=7, seed=3, normal="ziggurat")
    ora.reset()
    env._step_index = ora.step_index = step0
    assert np.array_equal(_np(env.reset()[0]), ora.reset())
    a = np.zeros((20, N, 2), dtype=np.int64)
    r = np.random.default_rng(3)
    a[np.arange(20)[:, None], np.arange(N)[None], r.integers(0, 2, (20, N))] = \
        r.integers(-1, 2, (20, N))
    got = env.rollout(20, actions=torch.as_tensor(a, device="cuda"))
    want = ora.rollout(20, a)
    for k in ("obs", "final_obs", "terminated", "truncated"):
        assert np.array_equal(_np(got[k]), want[k]), k
    np.testing.assert_allclose(_np(got["reward"]), want["reward"], rtol=1e-12,
                               atol=1e-12)


# ---------------------------------------------------------------------------
# 5. rollout_host == rollout
# ---------------------------------------------------------------------------
def _host_out(like, keys, pinned, obs_dtype=None):
    out = {}
    for k in keys:
        v = like[k]
        dt = obs_dtype if (obs_dtype is not None and k in ("obs", "final_obs")) \
            else v.dtype
        out[k] = torch.empty(tuple(v.shape), dtype=dt)
        if pinned:
            out[k] = out[k].pin_memory()
    return out


def _host_actions(kind, T, N, rng):
    if kind == "continuous":
        return torch.as_tensor(rng.uniform(-1, 1, size=(T, N, 2)).astype(np.float32))
    if kind == "grid":
        a = np.zeros((T, N, 2), dtype=np.int64)
        a[..., 0] = rng.integers(-1, 2, (T, N))
        return torch.as_tensor(a)
    if kind == "irr":
        return torch.as_tensor(rng.integers(0, 8, (T, N, 2)), dtype=torch.int32)
    return torch.as_tensor(rng.integers(0, 8, (T, N)), dtype=torch.int32)


_HOST_CFGS = {
    "discrete": lambda: dict(_BENCH_CFG),
    "irr": lambda: gu.case_config("irr_8x8_noise"),
    "continuous": lambda: dict(gu.case_config("cont_noise_delay"),
                               state_space_dim=2, action_space_dim=2,
                               relevant_indices=[0, 1], irrelevant_features=False),
    "grid": lambda: gu.case_config("grid_sparse_noise"),
}


@pytest.mark.parametrize("kind,pinned", [("discrete", True), ("irr", False),
                                         ("continuous", True), ("grid", False)])
def test_rollout_host_equals_rollout(kind, pinned):
    """Host buffers through the three-stream pipeline == rollout() of a twin
    env on device buffers, for T in {1, 49, 50, 51, 237} against chunk_steps
    in {1, 7, 50, 300} (one call after the other on the same env, so the
    step index must carry over), then a device rollout() right after."""
    N = 67
    mk = lambda: make_env(N, autoreset=True, horizon=9, philox_seed=5,  # noqa: E731
                          **_HOST_CFGS[kind]())
    H, D = mk(), mk()
    rng = np.random.default_rng(11)
    keys = ("obs", "reward", "terminated", "truncated")
    for T in (1, 49, 50, 51, 237):
        for chunk in (1, 7, 50, 300):
            a = _host_actions(kind, T, N, rng)
            want = D.rollout(T, actions=a.cuda(), want_final_obs=False)
            got = H.rollout_host(T, a.pin_memory() if pinned else a,
                                 _host_out(want, keys, pinned), chunk_steps=chunk)
            torch.cuda.current_stream().synchronize()
            for k in keys:
                _assert_same(got[k], want[k], (k, T, chunk))
            assert H._step_index == D._step_index
    a = _host_actions(kind, 5, N, rng).cuda()
    ra, rb = H.rollout(5, actions=a), D.rollout(5, actions=a)
    for k in ra:
        _assert_same(ra[k], rb[k], k)


def test_rollout_host_follows_changes_of_its_buffers():
    """Consecutive rollout_host calls on one env that change chunk_steps,
    then the observation dtype, then add final_obs: each equals rollout()."""
    N, T = 67, 23
    H = make_env(N, autoreset=True, horizon=9, philox_seed=5, **dict(_BENCH_CFG))
    D = make_env(N, autoreset=True, horizon=9, philox_seed=5, **dict(_BENCH_CFG))
    rng = np.random.default_rng(2)
    for chunk, obs_dt, keys in [
            (10, torch.int64, ("obs", "reward", "terminated", "truncated")),
            (4, torch.int64, ("obs", "reward", "terminated", "truncated")),
            (4, torch.uint8, ("obs", "reward", "terminated", "truncated")),
            (4, torch.uint8, ("obs", "final_obs", "reward", "terminated",
                              "truncated")),
            (6, torch.int32, ("obs", "final_obs", "reward"))]:
        a = _host_actions("discrete", T, N, rng)
        want = D.rollout(T, actions=a.cuda())
        out = _host_out(want, keys, True, obs_dtype=obs_dt)
        got = H.rollout_host(T, a.pin_memory(), out, chunk_steps=chunk)
        torch.cuda.current_stream().synchronize()
        for k in keys:
            assert got[k].dtype == out[k].dtype
            _assert_same(got[k].to(want[k].dtype), want[k], (k, chunk, obs_dt))
        # the device staging mirrors the caller's buffers
        assert {k: v.dtype for k, v in H._stage["outs"][0].items()} == \
            {k: v.dtype for k, v in out.items()}


# ---------------------------------------------------------------------------
# 6. input checks
# ---------------------------------------------------------------------------
def _two_group_env(**kw):
    """Group 0 has the SMALLER state space (4 states), group 1 has 8."""
    base = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
                reward_density=0.25, terminal_state_density=0.25,
                generate_random_mdp=True, sequence_length=1, delay=0, **kw)
    return make_env(10, config_groups=[dict(state_space_size=4, action_space_size=4),
                                       dict(state_space_size=8, action_space_size=8)],
                    group_sizes=[5, 5], **base)


def test_init_state_is_checked_against_its_own_group():
    """reset(init_state) on a two-group launch: a state of 4..7 in the
    4-state group is rejected although the other group has 8 states.  The
    rejection comes before any launch; only valid states are stepped."""
    env = _two_group_env()
    for bad in (4, 7):
        init = np.zeros(10, dtype=np.int64)
        init[2] = bad
        with pytest.raises(ValueError, match="out of range"):
            env.reset(options={"init_state": init})
    init = np.zeros(10, dtype=np.int64)
    init[8] = 8
    with pytest.raises(ValueError, match="out of range"):
        env.reset(options={"init_state": init})
    init = np.array([3] * 5 + [7] * 5)
    obs, _ = env.reset(options={"init_state": init})
    assert np.array_equal(_np(obs), init)
    out = env.rollout(3, actions=torch.zeros((3, 10), dtype=torch.int32,
                                             device="cuda"))
    assert int(out["final_obs"][:, :5].max()) < 4
    with pytest.raises(RuntimeError, match="track_history"):
        env.set_augmented_state(torch.full((10,), 3))  # no history per group


def test_irrelevant_state_is_checked_against_its_own_group():
    """The irrelevant column: group 0's irrelevant sub-MDP has 4 states,
    group 1's has 8."""
    base = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
                reward_density=0.25, terminal_state_density=0.25,
                generate_random_mdp=True, sequence_length=1, delay=0,
                irrelevant_features=True)
    env = make_env(10, config_groups=[
        dict(state_space_size=[8, 4], action_space_size=[8, 4]),
        dict(state_space_size=[8, 8], action_space_size=[8, 8])],
        group_sizes=[5, 5], **base)
    init = np.zeros((10, 2), dtype=np.int64)
    init[1, 1] = 5
    with pytest.raises(ValueError, match="out of range"):
        env.reset(options={"init_state": init})
    init[1, 1] = 3
    init[7, 1] = 7
    obs, _ = env.reset(options={"init_state": init})
    assert np.array_equal(_np(obs), init)


def test_set_augmented_state_is_checked_per_entry_and_column():
    """Single group, history on: an out-of-range entry of a bare state or of
    the augmented_state window, or an out-of-range irrelevant state, is
    rejected and leaves the env untouched."""
    env = make_env(16, track_history=True, **gu.case_config("irr_8x5_det"))
    before = {k: v.clone() for k, v in
              (("cur", env._cur), ("irr", env._cur_irr), ("t", env._t))}
    bad = torch.zeros((16, 2), dtype=torch.int64)
    bad[4, 1] = 5                      # the irrelevant sub-MDP has 5 states
    with pytest.raises(ValueError, match="out of range"):
        env.set_augmented_state(bad)
    bad = torch.zeros((16, 2), dtype=torch.int64)
    bad[4, 0] = 8
    with pytest.raises(ValueError, match="out of range"):
        env.set_augmented_state(bad)
    aug = env.get_augmented_state()
    aug["augmented_state"] = aug["augmented_state"].clone()
    aug["augmented_state"][3, 0] = 9   # an older window entry
    with pytest.raises(ValueError, match="out of range"):
        env.set_augmented_state(aug)
    assert torch.equal(env._cur, before["cur"])
    assert torch.equal(env._cur_irr, before["irr"])
    assert torch.equal(env._t, before["t"])
    ok = torch.zeros((16, 2), dtype=torch.int64)
    ok[:, 0], ok[:, 1] = 7, 4
    env.set_augmented_state(ok)
    assert torch.equal(env._cur_irr, ok[:, 1].to(torch.int32).cuda())


def test_set_obs_dtype_refuses_image_envs():
    """The renderer reads int64 states: an image env must not get its state
    buffer in another dtype.  Checked host side, before any launch."""
    env = make_env(8, **gu.case_config("c4_img_all"))
    for dt in (torch.uint8, torch.int32):
        with pytest.raises(ValueError, match="image"):
            env.set_obs_dtype(dt)
        assert env._obs_torch_dtype() == torch.int64
    plain = make_env(8, **dict(_BENCH_CFG))
    plain.set_obs_dtype(torch.uint8)
    assert plain.rollout(2)["obs"].dtype == torch.uint8
