"""GPU tests of the five config-group sets of the C library (discrete,
continuous and grid steps; discrete and continuous images) through their
setters: a set must tile the env range, a rejected set leaves the previous one
in place, a second set replaces the first, and a launch must cover the set's
envs.  The group arrays are the ones the envs hand to the library."""
import warnings

import numpy as np
import pytest
import torch

from tests import golden_util as gu

pytestmark = pytest.mark.gpu

EINVAL = -1  # MDPP_EINVAL


def make_env(*a, **k):
    from mdp_playground_b200 import VectorRLToyEnv
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return VectorRLToyEnv(*a, **k)


def _continuous_base():
    return dict(seed=0, state_space_type="continuous", action_space_type="continuous",
                state_space_dim=4, action_space_dim=4, relevant_indices=[0, 1],
                irrelevant_features=True, transition_dynamics_order=2, inertia=1.0,
                target_point=[0.0, 0.0], state_space_max=4.0, make_denser=True)


def _grid_base():
    return dict(seed=0, state_space_type="grid", delay=0, sequence_length=1,
                reward_function="move_to_a_point", grid_shape=(8, 8), target_point=[5, 5],
                make_denser=True)


def _discrete_image_base():
    return dict(seed=3, state_space_type="discrete", action_space_type="discrete",
                reward_density=0.25, terminal_state_density=0.25,
                generate_random_mdp=True, completely_connected=True,
                image_representations=True)


def _step_launch(actions):
    """A rollout of 12 steps with `actions(T, N)` (None: the device's random
    policy), and the env state and statistics it leaves."""
    def launch(env):
        T = 12
        acts = actions(T, env.num_envs)
        out = env.rollout(T, actions=acts) if acts is not None else env.rollout(T)
        return dict(out, **{f"state{i}": t for i, t in enumerate(env._state_tensors())},
                    stats=env._stats.sum(dim=0))
    return launch


def _continuous_actions(T, N):
    g = torch.Generator("cuda").manual_seed(6)
    return torch.rand((T, N, 4), device="cuda", generator=g) * 2.2 - 1.1


def _grid_actions(T, N):
    g = torch.Generator("cuda").manual_seed(6)
    acts = torch.zeros((T, N, 2), dtype=torch.int64, device="cuda")
    dim = torch.randint(0, 2, (T, N, 1), device="cuda", generator=g)
    return acts.scatter_(2, dim, torch.randint(-1, 2, (T, N, 1), device="cuda", generator=g))


def _render_discrete(env):
    g = torch.Generator("cuda").manual_seed(1)
    st = torch.randint(0, 8, (env.num_envs,), dtype=torch.int64, device="cuda", generator=g)
    return dict(pixels=env.render_observation(st), params=env.last_image_params)


def _render_continuous(env):
    rng = np.random.default_rng(2)
    st = torch.as_tensor(rng.uniform(-4, 4, size=(env.num_envs, 4)), dtype=torch.float32,
                         device="cuda")
    return dict(pixels=env.render_observation(st))


# kind -> (setter, base config, groups A, groups B, launch)
KINDS = {
    "discrete": (
        "mdpp_set_discrete_groups", {},
        [gu.case_config(n) for n in ("c1_seq1", "c2_every1")],
        [gu.case_config(n) for n in ("big50", "custom_8x5", "diam3_seq4")],
        _step_launch(lambda T, N: None)),
    "continuous": (
        "mdpp_set_continuous_groups", _continuous_base(),
        [dict(time_unit=0.1, action_space_max=1.0, delay=0, target_radius=0.5),
         dict(time_unit=0.5, action_space_max=0.25, delay=2, target_radius=0.5,
              transition_noise=0.05, transition_dynamics_order=1)],
        [dict(time_unit=1.0, action_space_max=0.5, delay=1, target_radius=1.0,
              reward_noise=0.2),
         dict(time_unit=0.25, action_space_max=1.0, delay=4, target_radius=0.25,
              transition_noise=0.1, reward_noise=0.1, transition_dynamics_order=3),
         dict(time_unit=0.05, action_space_max=0.1, delay=0, target_radius=0.5)],
        _step_launch(_continuous_actions)),
    "grid": (
        "mdpp_set_grid_groups", _grid_base(),
        [dict(make_denser=True, reward_scale=3.0, terminal_states=[[5, 5]]),
         dict(make_denser=False, transition_noise=0.3, reward_noise=1.0)],
        [dict(grid_shape=(5, 9), target_point=[1, 7], transition_noise=0.2,
              reward_every_n_steps=2),
         dict(grid_shape=(3, 4), target_point=[0, 0], reward_noise=0.5),
         dict(grid_shape=(12, 6), target_point=[11, 2], transition_noise=1.0)],
        _step_launch(_grid_actions)),
    "image_discrete": (
        "mdpp_set_image_discrete_groups", _discrete_image_base(),
        [dict(action_space_size=8, image_transforms="none"),
         dict(action_space_size=12, image_transforms="shift", image_sh_quant=2)],
        [dict(action_space_size=16, image_transforms="scale",
              image_scale_range=(0.5, 1.5)),
         dict(action_space_size=8, image_transforms="rotate", image_ro_quant=15),
         dict(action_space_size=12, image_transforms="flip")],
        _render_discrete),
    "image_continuous": (
        "mdpp_set_image_continuous_groups", dict(gu.case_config("cont_img")),
        [dict(target_point=[3.0, -3.0], state_space_max=5.0,
              terminal_states=[[1.0, 1.0], [-2.0, 0.5]]),
         dict(target_point=[-1.0, 2.0], state_space_max=4.0,
              terminal_states=[[0.0, -2.0]], term_state_edge=1.0)],
        [dict(target_point=[0.5, 0.5], state_space_max=8.0, terminal_states=[]),
         dict(target_point=[-1.0, 2.0], state_space_max=4.0, terminal_states=[]),
         dict(target_point=[3.0, -3.0], state_space_max=5.0,
              terminal_states=[[1.0, 1.0]])],
        _render_continuous),
}
STEP_KINDS = ["discrete", "continuous", "grid"]
SIZES_A, SIZES_B = [64, 37], [40, 1, 60]


@pytest.fixture
def sets(monkeypatch):
    """Records the group array each env's context is given by each setter:
    sets[(setter, ctx)] = (groups, n_groups)."""
    from mdp_playground_b200 import _lib
    lib = _lib.load()
    seen = {}
    for kind in KINDS.values():
        fn = getattr(lib, kind[0])

        def record(ctx, groups, n, fn=fn, name=kind[0]):
            seen[(name, ctx.value)] = (groups, n)
            return fn(ctx, groups, n)
        monkeypatch.setattr(lib, kind[0], record)
    return seen


def _env(kind, which, N=None):
    _, base, ga, gb, _ = KINDS[kind]
    groups, sizes = (ga, SIZES_A) if which == "A" else (gb, SIZES_B)
    if N is not None:  # the same groups over another env count
        sizes = [N - sum(sizes[1:])] + sizes[1:]
    return make_env(sum(sizes), autoreset=True, horizon=9, philox_seed=5,
                    config_groups=[dict(g) for g in groups], group_sizes=sizes,
                    **dict(base))


def _groups_of(sets, kind, env):
    """A copy of the group array `env`'s context was given."""
    groups, n = sets[(KINDS[kind][0], env._ctx.value)]
    return type(groups).from_buffer_copy(groups), n


def _set(env, kind, groups, n):
    from mdp_playground_b200 import _lib
    lib = _lib.load()
    return getattr(lib, KINDS[kind][0])(env._ctx, groups, n), \
        lib.mdpp_last_error(env._ctx).decode()


def _assert_same(got, want):
    assert got.keys() == want.keys()
    for k in want:
        assert torch.equal(got[k], want[k]), k


def _tiling_defects(groups):
    """(name, the array with that defect in group 1)."""
    out = []
    for name, field, delta in (("gap", "env_begin", 1), ("overlap", "env_begin", -1),
                               ("negative", "env_count", None)):
        g = type(groups).from_buffer_copy(groups)
        setattr(g[1], field, -1 if delta is None else getattr(g[1], field) + delta)
        out.append((name, g))
    return out


@pytest.mark.parametrize("kind", list(KINDS))
def test_tiling_errors_name_the_setter_and_the_group(kind, sets):
    env = _env(kind, "A")
    groups, n = _groups_of(sets, kind, env)
    for name, bad in _tiling_defects(groups):
        rc, msg = _set(env, kind, bad, n)
        assert rc == EINVAL, name
        assert KINDS[kind][0] in msg and "group 1" in msg and "tile" in msg, (name, msg)


@pytest.mark.parametrize("kind", list(KINDS))
def test_a_set_without_envs_is_rejected_when_set(kind, sets):
    env = _env(kind, "A")
    groups, n = _groups_of(sets, kind, env)
    for g in groups:
        g.env_begin = g.env_count = 0
    rc, msg = _set(env, kind, groups, n)
    assert rc == EINVAL and KINDS[kind][0] in msg, msg


@pytest.mark.parametrize("kind", list(KINDS))
def test_a_rejected_set_leaves_the_previous_one(kind, sets):
    fresh, env = _env(kind, "A"), _env(kind, "A")
    groups, n = _groups_of(sets, kind, env)
    rejected = [bad for _, bad in _tiling_defects(groups)]
    empty = type(groups).from_buffer_copy(groups)
    for g in empty:
        g.env_begin = g.env_count = 0
    for bad in rejected + [empty]:
        assert _set(env, kind, bad, n)[0] == EINVAL
    launch = KINDS[kind][4]
    _assert_same(launch(env), launch(fresh))


@pytest.mark.parametrize("kind", list(KINDS))
def test_a_second_set_replaces_the_first(kind, sets):
    a = _env(kind, "A")
    fresh, env = _env(kind, "B"), _env(kind, "B")
    ga, na = _groups_of(sets, kind, a)
    gb, nb = _groups_of(sets, kind, env)
    assert na != nb
    assert _set(env, kind, ga, na)[0] == 0
    assert _set(env, kind, gb, nb)[0] == 0
    launch = KINDS[kind][4]
    _assert_same(launch(env), launch(fresh))


@pytest.mark.parametrize("kind", STEP_KINDS)
def test_a_launch_must_cover_the_sets_envs(kind, sets):
    from mdp_playground_b200._lib import MdppError
    env, other = _env(kind, "A"), _env(kind, "A", N=sum(SIZES_A) + 64)
    groups, n = _groups_of(sets, kind, other)
    assert _set(env, kind, groups, n)[0] == 0
    with pytest.raises(MdppError, match=f"error {EINVAL}: .*n_envs"):
        KINDS[kind][4](env)
    with pytest.raises(MdppError, match=f"error {EINVAL}: .*n_envs"):
        env.reset()
