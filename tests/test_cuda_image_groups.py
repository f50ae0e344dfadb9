"""GPU tests of image observations in heterogeneous launches: every config
group renders with its own image settings.  A grouped env equals one env per
group pixel for pixel (discrete, continuous, grid), the images equal the
scalar oracle's Pillow rendering, shards reassemble to the unsplit job, the
renderer tables are shared between groups that render alike, and the C ABI
rejects inconsistent group sets."""
import ctypes as C
import os
import warnings

import numpy as np
import pytest
import torch

from tests import golden_util as gu

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def make_env(*a, **k):
    from mdp_playground_b200 import VectorRLToyEnv
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return VectorRLToyEnv(*a, **k)


def scalar_oracle(cfg):
    from oracle.scalar_env import ScalarRLToyEnv
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ScalarRLToyEnv(**cfg)


def cuda_actions(shape, high, seed, dtype=torch.int32):
    g = torch.Generator("cuda").manual_seed(seed)
    return torch.randint(0, high, shape, dtype=dtype, device="cuda", generator=g)


# ---------------------------------------------------------------------------
# discrete
# ---------------------------------------------------------------------------
DISCRETE_SIZES = [1, 37, 64, 5, 100, 50]


def discrete_groups(irr):
    """Six groups: transforms none / shift / scale / rotate / flip / all four
    with their own quantisations and scale ranges; 8, 12 and 16 states (S =
    action_space_size x diameter), the largest not in group 0."""
    rows = [("none", 8, None, None, None),
            ("shift", 12, 2, None, None),
            ("scale", 16, None, None, (0.5, 1.5)),
            ("rotate", 8, None, 15, None),
            ("flip", 12, None, None, None),
            ("shift,scale,rotate,flip", 16, 4, 30, (0.75, 1.25))]
    out = []
    for tr, S, shq, roq, sr in rows:
        c = dict(action_space_size=[S, 8] if irr else S, image_transforms=tr)
        if shq is not None:
            c["image_sh_quant"] = shq
        if roq is not None:
            c["image_ro_quant"] = roq
        if sr is not None:
            c["image_scale_range"] = sr
        out.append(c)
    return out


def discrete_base(irr):
    return dict(seed=3, state_space_type="discrete", action_space_type="discrete",
                irrelevant_features=irr, reward_density=0.25,
                terminal_state_density=0.25, generate_random_mdp=True,
                completely_connected=True, image_representations=True)


def params_rows(prm, n_sub, sl, T=None):
    """The rows of last_image_params ([M, 5], M = [T x] N x n_sub) of the
    envs in slice `sl`."""
    if T is None:
        return prm[sl.start * n_sub:sl.stop * n_sub]
    return prm.reshape(T, -1, 5)[:, sl.start * n_sub:sl.stop * n_sub]


@pytest.mark.parametrize("irr", [False, True])
def test_discrete_grouped_images_equal_one_env_per_group(irr):
    base, groups = discrete_base(irr), discrete_groups(irr)
    N, n_sub = sum(DISCRETE_SIZES), 2 if irr else 1
    kw = dict(autoreset=True, horizon=4, philox_seed=17)
    het = make_env(N, config_groups=groups, group_sizes=DISCRETE_SIZES, **kw, **base)
    assert het.n_groups == 6
    ones = [make_env(n, env_id_offset=sl.start, **kw, **{**base, **g})
            for g, n, sl in zip(groups, DISCRETE_SIZES, het.group_slices)]
    het_prm0 = het.last_image_params.clone()
    row = (N, 2) if irr else (N,)
    for one, sl in zip(ones, het.group_slices):  # the constructor's reset
        assert torch.equal(het.curr_obs[sl], one.curr_obs)
        assert torch.equal(params_rows(het_prm0, n_sub, sl), one.last_image_params)
    # step(): the pre-marshalled step + renderer pair
    acts = cuda_actions((5,) + row, 8, 1)
    for t in range(5):
        o, r, term, _, info = het.step(acts[t])
        prm = het.last_image_params
        for one, sl in zip(ones, het.group_slices):
            o1, r1, term1, _, _ = one.step(acts[t][sl].clone())
            assert torch.equal(o[sl], o1), (t, sl)
            assert torch.equal(r[sl], r1) and torch.equal(term[sl], term1)
            assert torch.equal(params_rows(prm, n_sub, sl), one.last_image_params)
    # rollout(7) and one render of the [T, N] block
    T = 7
    acts = cuda_actions((T,) + row, 8, 2)
    out = het.rollout(T, actions=acts)
    imgs = het.render_observation(out["obs"], step_index=het._step_index - T + 1)
    prm = het.last_image_params
    assert imgs.shape == (T, N, 100 * n_sub, 100, 1)
    for one, sl in zip(ones, het.group_slices):
        o1 = one.rollout(T, actions=acts[:, sl].clone())
        assert torch.equal(out["obs"][:, sl], o1["obs"])
        i1 = one.render_observation(o1["obs"], step_index=one._step_index - T + 1)
        assert torch.equal(imgs[:, sl], i1), sl
        assert torch.equal(params_rows(prm, n_sub, sl, T),
                           one.last_image_params.reshape(T, -1, 5))
    # the CUDA-graph step
    fh = het.make_graphed_step()
    fo = [one.make_graphed_step() for one in ones]
    acts = cuda_actions((3,) + row, 8, 3)
    for t in range(3):
        o = fh(acts[t])[0]
        prm = het.last_image_params
        for f, one, sl in zip(fo, ones, het.group_slices):
            o1 = f(acts[t][sl].clone())[0]
            assert torch.equal(o[sl], o1), (t, sl)
            assert torch.equal(params_rows(prm, n_sub, sl), one.last_image_params)


def test_discrete_grouped_images_equal_pillow():
    """For sampled envs of every group: the scalar oracle's image for the
    transform parameters the GPU reports equals the GPU image."""
    base, groups = discrete_base(False), discrete_groups(False)
    N = sum(DISCRETE_SIZES)
    het = make_env(N, autoreset=True, horizon=4, philox_seed=5,
                   config_groups=groups, group_sizes=DISCRETE_SIZES, **base)
    acts = cuda_actions((2, N), 8, 4)
    for t in range(2):
        o, _, _, _, info = het.step(acts[t])
    imgs = o.cpu().numpy()
    st = info["state"].cpu().numpy()
    prm = het.last_image_params.cpu().numpy()
    keys = ("R", "shift_w", "shift_h", "rotation", "flip")
    for g, sl in zip(groups, het.group_slices):
        ref = scalar_oracle({**base, **g})
        for i in list(range(sl.start, sl.stop, 7)) + [sl.stop - 1]:
            p = dict(zip(keys, (int(v) for v in prm[i])))
            if p["rotation"] < 0:
                p["rotation"] = None
            ref.image_params = lambda state, p=p: p
            assert np.array_equal(imgs[i, :, :, 0], ref._image_discrete(int(st[i]))), \
                (g["image_transforms"], i, p)


def test_discrete_grouped_images_two_shards_equal_the_unsplit_job():
    base, groups = discrete_base(False), discrete_groups(False)
    half = [8, 16, 24, 8, 40, 32]
    full = [2 * h for h in half]
    kw = dict(autoreset=True, horizon=5, philox_seed=9, config_groups=groups, **base)
    whole = make_env(sum(full), group_sizes=full, **kw)
    r0 = make_env(sum(half), group_sizes=half, shard=(0, 2), **kw)
    r1 = make_env(sum(half), group_sizes=half, shard=(1, 2), **kw)

    def check(ow, o0, o1):
        for sw, s0 in zip(whole.group_slices, r0.group_slices):
            assert torch.equal(ow[sw], torch.cat([o0[s0], o1[s0]]))
    check(whole.curr_obs, r0.curr_obs, r1.curr_obs)
    acts = cuda_actions((3, sum(full)), 8, 6)
    for t in range(3):
        a0 = torch.cat([acts[t][sw][:h] for sw, h in zip(whole.group_slices, half)])
        a1 = torch.cat([acts[t][sw][h:] for sw, h in zip(whole.group_slices, half)])
        check(whole.step(acts[t])[0], r0.step(a0)[0], r1.step(a1)[0])


def test_image_tables_are_built_once_per_distinct_image_configuration():
    """200 groups with 2 distinct image configurations: 2 table sets, sized
    for the largest state count that uses each; the images are those of the
    per-group envs."""
    base = discrete_base(False)
    groups = [dict(action_space_size=8 + 4 * (g % 3),
                   image_transforms="shift" if g % 2 else "rotate",
                   image_sh_quant=2, image_ro_quant=5) for g in range(200)]
    env = make_env(400, autoreset=True, horizon=6, philox_seed=2,
                   config_groups=groups, group_sizes=[2] * 200, **base)
    sets = env.image_table_sets
    assert len(sets) == 2
    assert sorted(tb.n_states for tb, _ in sets.values()) == [16, 16]
    o = env.step(cuda_actions((400,), 8, 8))[0]
    for g in (0, 1, 2, 3, 197, 199):
        sl = env.group_slices[g]
        one = make_env(2, autoreset=True, horizon=6, philox_seed=2,
                       env_id_offset=sl.start, **{**base, **groups[g]})
        assert torch.equal(o[sl], one.step(cuda_actions((400,), 8, 8)[sl])[0])


@pytest.mark.parametrize("key,value", [("image_width", 64), ("image_height", 80),
                                       ("image_representations", False)])
def test_groups_that_disagree_on_the_image_shape_are_rejected(key, value):
    base = discrete_base(False)
    groups = [dict(action_space_size=8), dict(action_space_size=8, **{key: value})]
    with pytest.raises(ValueError, match="group 1"):
        make_env(4, config_groups=groups, **base)
    cont = dict(gu.case_config("cont_img"))
    with pytest.raises(ValueError, match="group 1"):
        make_env(4, config_groups=[{}, {key: value}], **cont)
    grid = dict(gu.case_config("grid_img"))
    with pytest.raises(ValueError, match="group 1"):
        make_env(4, config_groups=[{}, {key: value}], **grid)


# ---------------------------------------------------------------------------
# continuous and grid
# ---------------------------------------------------------------------------
def continuous_groups(D, f64):
    extra = dict(state_space_dim=D, action_space_dim=D, relevant_indices=[0, 1],
                 irrelevant_features=D == 4)
    if f64:
        extra["dtype_s"] = np.float64
    return extra, [
        dict(target_point=[3.0, -3.0], state_space_max=5.0,
             terminal_states=[[1.0, 1.0], [-2.0, 0.5]]),
        dict(target_point=[-1.0, 2.0], state_space_max=4.0,
             terminal_states=[[0.0, -2.0]], term_state_edge=1.0),
        dict(target_point=[0.5, 0.5], state_space_max=8.0, terminal_states=[]),
    ]


def _compare_grouped_box_envs(base, groups, sizes, acts_fn, states_fn, oracle_image):
    N = sum(sizes)
    kw = dict(autoreset=True, horizon=4, philox_seed=21)
    het = make_env(N, config_groups=groups, group_sizes=sizes, **kw, **base)
    assert het.n_groups == len(groups)
    ones = [make_env(n, env_id_offset=sl.start, **kw, **{**base, **g})
            for g, n, sl in zip(groups, sizes, het.group_slices)]
    for one, sl in zip(ones, het.group_slices):
        assert torch.equal(het.curr_obs[sl], one.curr_obs)
    acts = acts_fn(4, N)
    for t in range(4):
        o = het.step(acts[t])[0]
        for one, sl in zip(ones, het.group_slices):
            # (a copy: the kernels want 16-byte aligned action rows)
            assert torch.equal(o[sl], one.step(acts[t][sl].clone())[0]), (t, sl)
    # random states of every group's box, every few against Pillow
    st = states_fn(N)
    imgs = het.render_observation(st).cpu().numpy()
    st_h = st.cpu().numpy()
    for g, one, sl in zip(groups, ones, het.group_slices):
        assert np.array_equal(imgs[sl], one.render_observation(st[sl]).cpu().numpy())
        ref = scalar_oracle({**base, **g})
        for i in range(sl.start, sl.stop, 5):
            assert np.array_equal(imgs[i], oracle_image(ref, st_h[i])), (g, i)


@pytest.mark.parametrize("D", [2, 4])
@pytest.mark.parametrize("f64", [False, True])
def test_continuous_grouped_images_equal_one_env_per_group_and_pillow(D, f64):
    base = dict(gu.case_config("cont_img"))
    extra, groups = continuous_groups(D, f64)
    base.update(extra)
    real = torch.float64 if f64 else torch.float32
    sizes = [37, 1, 90]

    def acts_fn(T, N):
        g = torch.Generator("cuda").manual_seed(D)
        return (torch.rand((T, N, D), generator=g, device="cuda", dtype=real) * 2 - 1)

    def states_fn(N):
        rng = np.random.default_rng(D)
        # (inside every group's box: state_space_max >= 4)
        return torch.as_tensor(rng.uniform(-4, 4, size=(N, D)), dtype=real,
                               device="cuda")
    _compare_grouped_box_envs(base, groups, sizes, acts_fn, states_fn,
                              lambda ref, s: ref._image_continuous(s))


def test_grid_grouped_images_equal_one_env_per_group_and_pillow():
    base = dict(gu.case_config("grid_img"))
    groups = [dict(grid_shape=(8, 8), target_point=[5, 5],
                   terminal_states=[[5, 5], [2, 3], [2, 4]]),
              dict(grid_shape=(5, 7), target_point=[1, 4], terminal_states=[[0, 0]]),
              dict(grid_shape=(10, 6), target_point=[7, 2], terminal_states=[])]
    sizes = [64, 37, 1]

    def acts_fn(T, N):
        g = torch.Generator("cuda").manual_seed(0)
        acts = torch.zeros((T, N, 2), dtype=torch.int64, device="cuda")
        dim = torch.randint(0, 2, (T, N, 1), device="cuda", generator=g)
        return acts.scatter_(2, dim, torch.randint(-1, 2, (T, N, 1), device="cuda",
                                                   generator=g))

    def states_fn(N):
        rng = np.random.default_rng(1)
        return torch.as_tensor(rng.integers(0, 5, size=(N, 2)), device="cuda")
    _compare_grouped_box_envs(base, groups, sizes, acts_fn, states_fn,
                              lambda ref, s: ref._image_grid(s))


# ---------------------------------------------------------------------------
# sweeps
# ---------------------------------------------------------------------------
def _sweep(name, **kw):
    from mdp_playground_b200 import sweep
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return sweep.Sweep(os.path.join(HERE, "fixtures", name), **kw)


@pytest.mark.parametrize("name", ["ddpg_move_to_a_point_images_like.py",
                                  "grid_images_like.py"])
def test_continuous_and_grid_image_sweeps_run_grouped(name):
    sw = _sweep(name, envs_per_cell=16)
    assert sw.grouped and len(sw.envs) == 1 and sw.env.n_groups == sw.n_cells == 4
    res = sw.run(20, chunk=10)
    assert np.all(res["transitions"] == 16 * 20)


def test_discrete_image_transform_sweep_equals_per_cell_envs():
    epc = 8
    sw = _sweep("dqn_image_transforms_like.py", envs_per_cell=epc, philox_seed=4)
    assert sw.env.n_groups == sw.n_cells == 6
    N = sw.env.num_envs
    acts = cuda_actions((N,), 8, 5)
    o = sw.env.step(acts)[0]
    for i, cfg in enumerate(sw.cell_configs):
        one = make_env(epc, autoreset=True, horizon=100, philox_seed=4,
                       env_id_offset=i * epc, **cfg)
        sl = slice(i * epc, (i + 1) * epc)
        assert torch.equal(o[sl], one.step(acts[sl])[0]), cfg["image_transforms"]


# ---------------------------------------------------------------------------
# C ABI checks
# ---------------------------------------------------------------------------
@pytest.fixture
def ctx():
    from mdp_playground_b200 import _lib
    lib = _lib.load()
    c = C.c_void_p()
    assert lib.mdpp_create(torch.cuda.current_device(), C.byref(c)) == 0
    yield lib, c
    lib.mdpp_destroy(c)


def _discrete_groups(counts, buf, over=None):
    from mdp_playground_b200 import _lib
    groups = (_lib.ImageDiscreteGroup * len(counts))()
    begin = 0
    for g, n in zip(groups, counts):
        t = g.tb
        t.width = t.height = 100
        t.n_states, t.r_min, t.n_radii, t.n_xvar, t.n_yvar = 8, 20, 1, 1, 1
        t.sh_quant = t.ro_quant = t.n_sub_images = 1
        p = buf.data_ptr()
        t.mask_bits = t.mask_index = t.xvar = t.yvar = t.rot_coeff = p
        t.r_thresholds = p
        g.env_begin, g.env_count, g.global_id_base = begin, n, begin
        begin += n
    for (gi, field), v in (over or {}).items():
        obj = groups[gi] if field in ("env_begin", "env_count") else groups[gi].tb
        setattr(obj, field, v)
    return groups


EINVAL = -1  # MDPP_EINVAL


def _error(lib, c):
    return lib.mdpp_last_error(c).decode()


def test_c_abi_rejects_inconsistent_discrete_image_groups(ctx):
    from mdp_playground_b200 import _lib
    lib, c = ctx
    buf = torch.zeros(64, dtype=torch.int64, device="cuda")
    set_ = lib.mdpp_set_image_discrete_groups
    bad = _discrete_groups([10, 5], buf, {(1, "env_begin"): 12})
    assert set_(c, bad, 2) == EINVAL and "tile" in _error(lib, c)
    bad = _discrete_groups([10, 5], buf, {(1, "height"): 64})
    assert set_(c, bad, 2) == EINVAL and "height" in _error(lib, c)
    bad = _discrete_groups([10, 5], buf, {(1, "n_sub_images"): 2})
    assert set_(c, bad, 2) == EINVAL and "n_sub_images" in _error(lib, c)
    bad = _discrete_groups([10, 5], buf, {(0, "xvar"): None})
    assert set_(c, bad, 2) == EINVAL and "table pointer" in _error(lib, c)
    # a render call before any successful set
    opts = _lib.StepOpts()
    states = torch.zeros(15, dtype=torch.int64, device="cuda")
    out = torch.zeros((15, 100, 100), dtype=torch.uint8, device="cuda")
    render = lib.mdpp_render_discrete_groups
    assert render(c, states.data_ptr(), None, None, out.data_ptr(), 15, 15, 3,
                  C.byref(opts), None) == EINVAL
    good = _discrete_groups([10, 5], buf)
    assert set_(c, good, 2) == 0
    assert render(c, states.data_ptr(), None, None, out.data_ptr(), 16, 16, 3,
                  C.byref(opts), None) == EINVAL
    assert "n_envs" in _error(lib, c)
    # a second set replaces the first
    assert set_(c, _discrete_groups([3, 4, 9], buf), 3) == 0


def test_c_abi_rejects_inconsistent_continuous_image_groups(ctx):
    from mdp_playground_b200 import _lib
    lib, c = ctx
    env = make_env(4, **gu.case_config("cont_img"))
    cfg = env._img_cfg

    def groups(counts, over=None):
        gs = (_lib.ImageContinuousGroup * len(counts))()
        begin = 0
        for g, n in zip(gs, counts):
            g.cfg = cfg
            g.env_begin, g.env_count = begin, n
            begin += n
        for (gi, field), v in (over or {}).items():
            setattr(gs[gi] if field.startswith("env_") else gs[gi].cfg, field, v)
        return gs
    set_ = lib.mdpp_set_image_continuous_groups
    assert set_(c, groups([4, 4], {(1, "env_count"): -1}), 2) == EINVAL
    assert "tile" in _error(lib, c)
    assert set_(c, groups([4, 4], {(1, "width"): 50}), 2) == EINVAL
    assert "width" in _error(lib, c)
    assert set_(c, groups([4, 4], {(1, "dim"): 2}), 2) == EINVAL
    assert "dim" in _error(lib, c)
    assert set_(c, groups([4, 4], {(1, "is_f64"): 1}), 2) == EINVAL
    assert "is_f64" in _error(lib, c)
    assert set_(c, groups([4, 4]), 2) == 0
    st = torch.zeros((9, 4), dtype=torch.float32, device="cuda")
    out = torch.zeros((9, 200, 100, 3), dtype=torch.uint8, device="cuda")
    assert lib.mdpp_render_continuous_groups(
        c, st.data_ptr(), out.data_ptr(), 9, 9, None) == EINVAL
    assert "n_envs" in _error(lib, c)
    assert lib.mdpp_render_continuous_groups(
        c, st.data_ptr(), out.data_ptr(), 9, 8, None) == 0
    torch.cuda.synchronize()
    one = env.render_observation(st[:1])
    assert torch.equal(out[:8], one.expand(8, -1, -1, -1))
