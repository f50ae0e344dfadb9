"""VectorRLToyEnv: N independent RLToyEnv instances stepped by sm_100a kernels.

Drop-in for the reference's `RLToyEnv` on the step path (constructor keys,
`reset` / `step` return tuples, `get_augmented_state`; rl_toy_env.py:216,
:2217, :1992, :2127), batched over a leading env axis.  All state lives in
PyTorch-owned device tensors; every operation is a call into libmdpp_b200.so
(include/mdpp_b200.h) on the current CUDA stream.  There is no CPU path.

`VectorRLToyEnv(...)` builds the subclass of the config's state-space kind:
discrete_env.DiscreteEnv, continuous_env.ContinuousEnv or grid_env.GridEnv.
This module holds what does not depend on the kind: the constructor's common
part, the reset / rollout skeletons, step() and its pre-marshalled fast path,
the CUDA-graph step and the host-buffer rollout.

Noise modes (SURVEY.md 8b):
  "philox"  (default) native counter-based noise, stream = (seed, env, step)
  "replay"  the caller passes the draws (bit-exact replays of reference runs)
  "numpy"   the host draws from the reference's own PCG64 streams and feeds
            them through the replay inputs: lane 0 reproduces the reference
            env with the same seed bit for bit (small N; parity / debugging)
  "off" is implied when the config has no noise.
"""
import copy
import ctypes as C
import inspect

import numpy as np
import torch

from . import _lib
from ._lib import _ptr
from .config import np_random, parse_config, state_space_kind


# raw handle of the current stream of a device (the public accessor builds a
# Stream object per call: ~2 us, a third of a 65 536-env step)
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None) or (
    lambda idx: torch.cuda.current_stream(idx).cuda_stream)


class VectorRLToyEnv:
    metadata = {"render_modes": []}

    # Per-kind values the subclasses set (as class attributes here, or in
    # _init_kind): the "fp64" normal generator, the state tensors of the
    # kind's state struct, the IO struct, whether rollout(actions=None) runs
    # the kernels' random policy, whether step() renders images on its fast
    # path, and the reset options that replay mode requires.
    _FP64_NORMAL = _lib.MDPP_NORMAL_F64
    _STATE_TENSORS = ()
    _IO = None
    _random_policy = False
    _renders_in_step = False
    _REPLAY_RESET = "options['init_state']"
    _reward_dtype = torch.float64

    def __new__(cls, *args, **kwargs):
        """VectorRLToyEnv(...) constructs the class of the config's kind."""
        if cls is not VectorRLToyEnv:
            return super().__new__(cls)
        a = inspect.signature(cls.__init__).bind(None, *args, **kwargs).arguments
        config, groups = a.get("config", {}), a.get("config_groups")
        kinds = {state_space_kind({**config, **c}) for c in groups} if groups \
            else {state_space_kind(config)}
        if len(kinds) != 1:
            raise NotImplementedError(
                "config_groups: one state_space_type per launch")
        from .continuous_env import ContinuousEnv
        from .discrete_env import DiscreteEnv
        from .grid_env import GridEnv
        return super().__new__({"discrete": DiscreteEnv, "continuous": ContinuousEnv,
                                "grid": GridEnv}[kinds.pop()])

    def __init__(self, num_envs, device=None, noise="philox", autoreset=False,
                 horizon=0, env_id_offset=0, philox_seed=None,
                 normal_precision="fp64", track_history=None,
                 config_groups=None, group_sizes=None, shard=(0, 1),
                 step_buffers=2, strict=True, **config):
        """config_groups: optional list of config dicts (a heterogeneous
        sweep: each entry is merged over **config); envs are laid out
        group-major, `group_sizes` per group (default: as equal as possible).
        shard=(rank, world): this object holds rank's share of a job that
        runs the same groups on `world` GPUs (global Philox ids follow).
        step_buffers: step() writes into this many rotating, pre-allocated
        output sets (the tensors it returns stay valid until `step_buffers`
        further step() calls; 0 = allocate fresh tensors on every call).
        A 65 536-env step is a ~5 us kernel: allocating and marshalling five
        tensors per call would cost several times that."""
        # strict=False reproduces what the reference does with actions of a
        # dtype its action space does not contain (rl_toy_env.py:1640,
        # :1671-1679, :1730-1733) instead of raising: continuous envs freeze
        # the state for that step, grid envs apply a no-op
        self.strict = bool(strict)
        self._step_buffers = int(step_buffers)
        self._step_sets = None
        self._step_flip = 0
        if not torch.cuda.is_available():
            raise RuntimeError(
                "VectorRLToyEnv needs a CUDA device: the step path is CUDA "
                "only, there is no CPU fallback")
        self._lib = _lib.load()
        self.num_envs = N = int(num_envs)
        assert self.num_envs > 0
        self.device = torch.device(
            "cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        dev = self.device
        assert noise in ("philox", "replay", "numpy")
        self.noise = noise
        self.autoreset = bool(autoreset)
        self.horizon = int(horizon)
        self.env_id_offset = int(env_id_offset)
        # noise normals of the Philox mode (reward noise; the continuous
        # transition noise): "ziggurat" = numpy's 256-layer ziggurat in fp64 on
        # Philox words -- the algorithm behind the reference's np_random.normal
        # calls --, "boxmuller" = fp64 Box-Muller, "fast" = fp32 Box-Muller on
        # the SFU; "fp64" (default) = the faster of the two fp64 generators
        # for the kernel: ziggurat for discrete envs (staged a window ahead in
        # shared memory), Box-Muller for continuous / grid envs
        assert normal_precision in ("fp64", "ziggurat", "boxmuller", "fast")
        self.normal_precision = normal_precision
        # the state history behind get_augmented_state() costs one extra
        # store per step; on by default for gym-style (non-autoreset) use
        self.track_history = (not self.autoreset) if track_history is None \
            else bool(track_history)
        self._shard = (int(shard[0]), int(shard[1]))
        if config_groups:
            cfgs = [dict(copy.deepcopy(config), **copy.deepcopy(c))
                    for c in config_groups]
            self._group_specs = [parse_config(c) for c in cfgs]
            G = len(cfgs)
            if group_sizes is None:
                from .sharding import even_group_sizes
                group_sizes = even_group_sizes(self.num_envs, G)
            assert len(group_sizes) == G and sum(group_sizes) == self.num_envs
            self._group_sizes = [int(x) for x in group_sizes]
        else:
            self._group_specs = [parse_config(config)]
            self._group_sizes = [self.num_envs]
        specs = self._group_specs
        self.spec = specs[0]
        self.n_groups = len(specs)
        self.normal_mode = {
            "fast": _lib.MDPP_NORMAL_FAST, "boxmuller": _lib.MDPP_NORMAL_F64,
            "ziggurat": _lib.MDPP_NORMAL_ZIGGURAT,
            "fp64": self._FP64_NORMAL}[normal_precision]
        self.config = self.spec.config
        self.seed_dict = self.spec.seed_dict
        if philox_seed is None:
            philox_seed = self.seed_dict["env"]
            if philox_seed is None:
                philox_seed = int(np.random.SeedSequence().entropy & (2**63 - 1))
        self.philox_seed = int(philox_seed) & (2**64 - 1)
        self._step_index = 0
        self._seed_epoch = 0
        self._noise_mode = {"philox": _lib.MDPP_NOISE_PHILOX,
                            "replay": _lib.MDPP_NOISE_REPLAY,
                            "numpy": _lib.MDPP_NOISE_REPLAY}[noise]
        # CUDA-graph capture (make_graphed_step) switches these on
        self._use_dev_counter = False
        self._overlap_render = False
        self._ctx = C.c_void_p()
        _lib.check(self._lib, None,
                   self._lib.mdpp_create(self.device.index, C.byref(self._ctx)))
        self.has_pnoise = any(bool(s_.transition_noise) for s_ in specs)
        self.has_rnoise = any(s_.has_reward_noise for s_ in specs)
        self._t = torch.zeros(N, dtype=torch.int32, device=dev)
        self._episode = torch.zeros(N, dtype=torch.int32, device=dev)
        self._stats = torch.zeros((_lib.STATS_SLOTS, self.n_groups,
                                   _lib.MDPP_N_STATS),
                                  dtype=torch.float64, device=dev)
        self._history = None
        if self.noise == "numpy":
            self._rng_E = [None] * N  # seeded by the first reset
        self._check_image_groups()
        self._init_kind()
        self._fast_step = (self.noise == "philox" and self._step_buffers > 0
                           and (self._renders_in_step
                                or not self.spec.image_representations))
        if self.spec.image_representations:
            self._init_images()
        # rl_toy_env.py:831-833: the constructor ends with reset(seed=env seed)
        self.curr_obs, _ = self.reset(seed=self.seed_dict["env"],
                                      options={"_ctor": True})

    # ------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.mdpp_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_jit(self, enabled):
        """Enable/disable the NVRTC-specialised rollout kernel (on by default;
        the ahead-of-time kernels are used when off or unavailable)."""
        self._lib.mdpp_set_jit(self._ctx, int(bool(enabled)))

    @property
    def jit_last_used(self):
        return bool(self._lib.mdpp_jit_last_used(self._ctx))

    @property
    def jit_log(self):
        return self._lib.mdpp_jit_log(self._ctx).decode()

    def _check(self, rc):
        _lib.check(self._lib, self._ctx, rc)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------
    # construction helpers of the kinds
    # ------------------------------------------------------------------
    def _group_layout(self):
        """(env_begin, env_count, global_id_base) of every config group.  Envs
        are laid out group-major: group g owns the contiguous range
        group_slices[g].  Global Philox ids: all ranks' envs of a group are
        contiguous (sharding.group_id_bases)."""
        from .sharding import group_id_bases, local_slices
        self.group_slices = local_slices(self._group_sizes)
        return [(s.start, s.stop - s.start, base) for s, base in zip(
            self.group_slices, group_id_bases(self._group_sizes, *self._shard))]

    def _group_array(self, group_cls):
        """A ctypes array of `group_cls`, one per config group, with env_begin,
        env_count and (where the struct has it) global_id_base filled in from
        _group_layout()."""
        groups = (group_cls * self.n_groups)()
        has_base = any(f[0] == "global_id_base" for f in group_cls._fields_)
        for g, (begin, count, id_base) in zip(groups, self._group_layout()):
            g.env_begin, g.env_count = begin, count
            if has_base:
                g.global_id_base = id_base
        return groups

    def _set_configs(self, cfgs, group_cls, set_groups, set_config):
        """Hand the config structs of a continuous or grid env (one per
        group) to the library.  A single configuration keeps its own entry
        point and kernels; config groups run as one GROUPS launch."""
        if len(cfgs) == 1:
            if self._shard[1] > 1:
                # a single configuration is one group: rank r owns the global
                # Philox ids [offset + r N, offset + (r + 1) N)
                self.env_id_offset += self._shard[0] * self.num_envs
            self._check(set_config(self._ctx, C.byref(cfgs[0])))
            return
        groups = self._group_array(group_cls)
        for g, cfg in zip(groups, cfgs):
            g.cfg = cfg
        self._check(set_groups(self._ctx, groups, len(cfgs)))

    def _check_image_groups(self):
        """Config groups share one observation tensor: they must agree on
        whether observations are images and on the image size."""
        sp = self.spec
        for gi, s_ in enumerate(self._group_specs):
            if s_.image_representations != sp.image_representations or (
                    sp.image_representations
                    and (s_.image_width, s_.image_height)
                    != (sp.image_width, sp.image_height)):
                raise ValueError(
                    "config_groups must agree on image_representations, "
                    f"image_width and image_height (group {gi} differs from "
                    "group 0)")

    def _set_image_groups(self, cfgs):
        """Hand the image configs of a continuous or grid env (one per
        group) to the library: a single one is passed to each render call,
        config groups are set once for the grouped renderer."""
        self._img_cfg = cfgs[0]
        if len(cfgs) == 1:
            return
        groups = self._group_array(_lib.ImageContinuousGroup)
        for g, cfg in zip(groups, cfgs):
            g.cfg = cfg
        self._check(self._lib.mdpp_set_image_continuous_groups(
            self._ctx, groups, len(cfgs)))

    def _new_state(self, cls):
        """The kind's state struct, with the fields every kind has set."""
        st = cls()
        st.n_envs = self.num_envs
        st.t_episode, st.episode = _ptr(self._t), _ptr(self._episode)
        st.stats, st.stats_slots = _ptr(self._stats), _lib.STATS_SLOTS
        return st

    def _box_image_cfg(self, sp, dim, lo, hi, rects, target, is_f64):
        """ImageContinuousConfig of the renderer of the feature box [lo, hi]
        of parsed config `sp` (image_continuous.py): black `rects` given as
        (low, high) corners, the green target disc at `target` and the agent
        discs of circle_radius=5 (rl_toy_env.py:774).  Dimensions 0 and 1 are
        the relevant ones (ImageContinuous' default; the env does not pass its
        own); with dim 4, 2 and 3 are drawn in a second sub-image."""
        from .image_tables import disc_stamp
        W, H = sp.image_width, sp.image_height

        def to_pixel(vec):  # image_continuous.py:248-277
            frac = (np.asarray(vec) - lo) / (hi - lo)
            return (frac * (W, H)).astype(int)
        c = _lib.ImageContinuousConfig()
        c.width, c.height, c.dim, c.n_sub_images = W, H, dim, dim // 2
        c.is_f64 = int(is_f64)
        for k in range(2):
            c.rel_index[k], c.irr_index[k] = k, (2 + k if dim == 4 else 0)
            c.feat_low[k], c.feat_high[k] = float(lo[k]), float(hi[k])
        c.n_rects = len(rects)
        for b, (r0, r1) in enumerate(rects):
            p0, p1 = to_pixel(r0), to_pixel(r1)
            c.rect[b][0], c.rect[b][1] = int(p0[0]), int(p0[1])
            c.rect[b][2], c.rect[b][3] = int(p1[0]), int(p1[1])
        c.has_target = 1
        tp = to_pixel(target)
        c.target_pixel[0], c.target_pixel[1] = int(tp[0]), int(tp[1])
        spans = disc_stamp(5)
        c.stamp_rows, c.stamp_radius = len(spans), 5
        for r, (x0, wdt) in enumerate(spans):
            c.stamp[r][0], c.stamp[r][1] = int(x0), int(wdt)
        self.obs_shape = (W * c.n_sub_images, H, 3)
        return c

    # ------------------------------------------------------------------
    # seeding
    # ------------------------------------------------------------------
    def _reseed(self, seed, mask=None, rewind=False):
        """reset(seed=s) / seed(s) in Philox mode: re-key the streams and zero
        the episode counters of the envs in `mask` (all when None).

        `rewind` (an unmasked reset(seed=s)) also sets the global step back to
        0, so that the same seed gives the same trajectory -- the gym
        reset(seed) contract the reference meets by re-seeding `_np_random`.
        Every env's delay ring and state history are dead at that point.  A
        masked reset(seed) or a bare seed(s) keeps the step index: the envs
        it does not reset still find their ring, history and line-window slots
        from it (slot = step mod depth).  It re-keys every env, so it does not
        promise a reproducible trajectory.  CUDA graphs captured before keep
        the old key baked into their kernel parameters: they refuse to replay
        (make_graphed_step)."""
        self.philox_seed = int(seed) & (2**64 - 1)
        if rewind:
            self._step_index = 0
        if mask is None:
            self._episode.zero_()
        else:
            self._episode.masked_fill_(mask.to(torch.bool), 0)
        self._seed_epoch += 1

    def _numpy_lanes(self, seed, first=0):
        """noise='numpy': PCG64 streams of lanes first..N-1, lane i like the
        reference seeded with seed + i (fresh entropy when seed is None)."""
        return [np_random(None if seed is None else seed + i)[0]
                for i in range(first, self.num_envs)]

    def seed(self, seed=None):
        """RLToyEnv.seed (:2379): re-keys the environment's noise stream."""
        if self.noise == "numpy":
            self._rng_E = self._numpy_lanes(seed)
        elif seed is not None:
            self._reseed(seed)
        return seed

    def _opts(self, T, noise_mode=None):
        o = _lib.StepOpts()
        o.n_steps = T
        o.noise_mode = self._noise_mode if noise_mode is None else noise_mode
        o.autoreset = int(self.autoreset)
        o.horizon = self.horizon
        o.normal_mode = self.normal_mode
        o.seed = self.philox_seed
        o.step_index = self._step_index
        o.env_id_offset = self.env_id_offset
        if self._use_dev_counter:
            # CUDA-graph mode: the step index lives in a device scalar that
            # the graph itself advances BEFORE the kernels run (see
            # make_graphed_step): index = counter - 1 (mod 2^64)
            o.step_index = 2**64 - 1
            o.step_index_dev = self._step_ctr.data_ptr()
        return o

    # ------------------------------------------------------------------
    def reset(self, seed=None, options=None):
        """(obs, info) like RLToyEnv.reset (:2217).  options: {"mask": bool[N],
        "init_state": [N(, ...)] states, "reset_u": float64[N] (discrete,
        replay mode)}; with irrelevant_features discrete init_state / reset_u
        / obs are [N, 2] rows (relevant, irrelevant)."""
        options = options or {}
        ctor = bool(options.get("_ctor"))
        N, dev = self.num_envs, self.device
        mask = options.get("mask")
        if mask is not None:
            mask = torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
        init = options.get("init_state")
        if init is not None:
            init = self._init_states(init)
        draws = None
        if self.noise == "numpy" and init is None:
            if seed is not None or self._rng_E[0] is None:
                self._rng_E = self._numpy_lanes(seed)
            draws = self._numpy_reset_draws(
                None if mask is None else mask.cpu().numpy())
        elif seed is not None and self.noise == "philox" and not ctor:
            # re-keying the counter-based streams is the analogue of re-seeding
            self._reseed(seed, mask, rewind=mask is None)
        mode, inputs = self._reset_inputs(init, draws, options)
        if self.noise == "replay" and not ctor and all(t is None for t in inputs):
            raise ValueError(f"replay mode: pass {self._REPLAY_RESET} to reset()")
        obs = torch.empty((N,) + self._row, dtype=self._state_dtype, device=dev)
        opts = self._opts(1, mode)
        self._check(self._reset_fn(
            self._ctx, C.byref(self._state), _ptr(mask),
            *[_ptr(t) for t in inputs], _ptr(obs), C.byref(opts), self._stream()))
        self.curr_obs = self._observe(obs, options.get("image_params"),
                                      reset=True, ctor=ctor)
        return self.curr_obs, {}

    def _init_states(self, init):
        """Caller-supplied (or host-drawn) reset states as the kernel reads
        them."""
        return torch.as_tensor(init, device=self.device).to(
            self._state_dtype).reshape((self.num_envs,) + self._row).contiguous()

    def _reset_inputs(self, init, draws, options):
        """(noise mode, the reset entry point's inputs after the mask)."""
        if draws is not None:
            init = self._init_states(draws)
        return _lib.MDPP_NOISE_PHILOX, (init,)

    def _observe(self, state, image_params=None, reset=False, ctor=False):
        """Underlying state -> observation (identity, dtype_o cast, or the
        image renderer when image_representations is on)."""
        if self.spec.image_representations:
            return self.render_observation(state, image_params=image_params,
                                           reset=reset, allow_philox=ctor)
        return self._cast_obs(state)

    def _cast_obs(self, obs):
        return obs

    def _obs_torch_dtype(self):
        """dtype the kernels write observations in."""
        return self._state_dtype

    def render_observation(self, state, image_params=None, reset=False,
                           step_index=None, allow_philox=False):
        """State tensor -> uint8 image observations on the GPU:
        [..., N, D] -> [..., N, k*W, H, 3] (continuous and grid envs)."""
        st = self._render_states(state)
        out = torch.empty(tuple(st.shape[:-1]) + self.obs_shape,
                          dtype=torch.uint8, device=self.device)
        n_images = st.numel() // self._row[0]
        if self.n_groups > 1:  # each image with its config group's settings
            self._check(self._lib.mdpp_render_continuous_groups(
                self._ctx, _ptr(st), _ptr(out), n_images, self.num_envs,
                self._stream()))
        else:
            self._check(self._lib.mdpp_render_continuous(
                self._ctx, C.byref(self._img_cfg), _ptr(st), _ptr(out),
                n_images, self._stream()))
        return out

    # ------------------------------------------------------------------
    # stepping
    # ------------------------------------------------------------------
    def step(self, actions, replay=None):
        """(obs, reward, terminated, truncated, info) like RLToyEnv.step
        (:1992).  `replay`: dict with "transition_u", "reward_noise",
        "reset_u" float64[N] arrays (noise='replay').  info["state"] is the
        underlying state, info["final_obs"] (autoreset only) the state before
        the same-step reset."""
        if replay is None and self._fast_step and not self._use_dev_counter:
            return self._step_fast(actions)
        actions = torch.as_tensor(actions).reshape((1, self.num_envs) + self._row)
        out = self.rollout(1, actions=actions, replay=None if replay is None else
                           {k: torch.as_tensor(v)[None] for k, v in replay.items()})
        state = out["obs"][0]
        obs = self._observe(
            state, None if replay is None else replay.get("image_params"))
        self.curr_obs = obs
        return (obs, out["reward"][0], out["terminated"][0],
                out["truncated"][0],
                {"final_obs": out["final_obs"][0], "state": state})

    def _alloc_out(self, T, obs_dtype, final_obs):
        """Output buffers of a T-step launch."""
        N, dev = self.num_envs, self.device
        row = (T, N) + self._row
        out = {"obs": torch.empty(row, dtype=obs_dtype, device=dev),
               "reward": torch.empty((T, N), dtype=self._reward_dtype, device=dev),
               "terminated": torch.empty((T, N), dtype=torch.bool, device=dev),
               "truncated": torch.empty((T, N), dtype=torch.bool, device=dev)}
        if final_obs:
            out["final_obs"] = torch.empty(row, dtype=obs_dtype, device=dev)
        return out

    def _io(self, actions, out):
        """The kind's IO struct pointing at `actions` and the buffers of `out`."""
        io = self._IO()
        io.actions = _ptr(actions)
        io.obs, io.reward = _ptr(out.get("obs")), _ptr(out.get("reward"))
        io.final_obs = _ptr(out.get("final_obs"))
        io.terminated = _ptr(out.get("terminated"))
        io.truncated = _ptr(out.get("truncated"))
        return io

    def _replay_io(self, io, replay, T):
        """Point the IO struct's replay fields at the draws in `replay`
        (self._replay_fields: name, IO field, dtype, per-env shape).  Returns
        the tensors, which must outlive the launch."""
        keep = []
        for name, field, dtype, shape in self._replay_fields:
            if replay.get(name) is not None:
                t = self._replay_tensor(replay, name, dtype,
                                        (T, self.num_envs) + shape)
                keep.append(t)
                setattr(io, field, _ptr(t))
        return keep

    def _replay_tensor(self, replay, name, dtype, shape):
        return torch.as_tensor(replay[name], device=self.device).to(
            dtype).reshape(shape).contiguous()

    # -- step() without per-call allocation / marshalling -------------------
    def _step_render(self, state):
        """(observation, pre-marshalled renderer launch or None) of a step()
        output set whose state buffer is `state`."""
        return state, None

    def _build_step_sets(self):
        """`step_buffers` output sets, each with its I/O struct marshalled once
        and the tuple step() returns built once."""
        odt = self._obs_torch_dtype()
        self._step_arow = (1, self.num_envs) + self._row
        self._step_numel = int(np.prod(self._step_arow))
        self._dev_index = self.device.index
        sets = []
        for _ in range(self._step_buffers):
            out = self._alloc_out(1, odt, self.autoreset)
            io = self._io(None, out)
            state = out["obs"][0]
            obs, render = self._step_render(state)
            info = {"state": state}
            if self.autoreset:
                info["final_obs"] = out["final_obs"][0]
            ret = (obs, out["reward"][0], out["terminated"][0], out["truncated"][0], info)
            sets.append((io, C.byref(io), ret, out, render))
        self._step_sets = sets
        self._step_opts = self._opts(1)
        self._step_opts_ref = C.byref(self._step_opts)
        self._step_state_ref = C.byref(self._state)
        # dtype_o values the kernels do not write (e.g. int16): cast per call
        self._step_cast = sets[0][4] is None and \
            self._cast_obs(sets[0][3]["obs"][0]).dtype != odt

    def _step_fast(self, actions):
        sets = self._step_sets
        if sets is None:
            self._build_step_sets()
            sets = self._step_sets
        if not (torch.is_tensor(actions) and actions.dtype == self._adt
                and actions.is_cuda and actions.is_contiguous()):
            actions = self._coerce_actions(torch.as_tensor(actions, device=self.device))
        if actions.numel() != self._step_numel:
            raise AssertionError((tuple(actions.shape), self._step_arow))
        flip = self._step_flip
        io, io_ref, ret, _, render = sets[flip]
        self._step_flip = flip + 1 if flip + 1 < len(sets) else 0
        io.actions = actions.data_ptr()
        o = self._step_opts
        o.step_index = self._step_index
        o.seed = self.philox_seed
        rc = self._rollout_fn(self._ctx, self._step_state_ref, io_ref,
                              self._step_opts_ref, _raw_stream(self._dev_index))
        if rc:
            self._check(rc)
        self._step_index += 1
        if render is not None:
            fn, ropts, args, prm = render
            ropts.step_index = self._step_index  # the observation AFTER the step
            ropts.seed = self.philox_seed
            rc = fn(self._ctx, *args, _raw_stream(self._dev_index))
            if rc:
                self._check(rc)
            self.last_image_params = prm
        if self._step_cast:
            ret = (self._cast_obs(ret[4]["state"]),) + ret[1:]
        self.curr_obs = ret[0]
        return ret

    def rollout(self, n_steps, actions=None, replay=None, out=None,
                want_final_obs=True):
        """T fused steps in ONE kernel launch.  actions: [T, N(, ...)] tensor,
        or None for the uniform random policy drawn on device (discrete envs).
        Returns dict of time-major [T, N(, ...)] tensors: obs, final_obs,
        reward, terminated, truncated."""
        return self._launch_rollout(int(n_steps), actions, replay, out,
                                    want_final_obs)[2]

    def _launch_rollout(self, T, actions, replay, out, want_final_obs):
        """rollout(); returns (IO struct, actions as launched, outputs)."""
        row = (T, self.num_envs) + self._row
        if actions is not None:
            actions = self._coerce_actions(torch.as_tensor(actions, device=self.device))
            assert actions.shape == row, (actions.shape, row)
        elif not self._random_policy:
            raise ValueError(f"rollout needs an actions tensor of shape {row}")
        if out is None:
            out = self._alloc_out(T, self._obs_torch_dtype(), want_final_obs)
        io = self._io(actions, out)
        if self.noise == "numpy":
            replay = self._draw_numpy(T, actions)
        # (holds the replay tensors until the launch is enqueued)
        keep = None if self.noise == "philox" else self._replay_io(io, replay or {}, T)
        opts = self._opts(T)
        self._check(self._rollout_fn(
            self._ctx, C.byref(self._state), C.byref(io), C.byref(opts),
            self._stream()))
        self._step_index += T
        return io, actions, out

    # ------------------------------------------------------------------
    # CUDA-graph step: the gym-style path without per-step launch overhead
    # ------------------------------------------------------------------
    def _state_tensors(self):
        return [t for t in (getattr(self, n) for n in self._STATE_TENSORS)
                if t is not None]

    def make_graphed_step(self):
        """Capture one step() -- the step kernel, the renderer when images
        are on, and the advance of the Philox step counter -- into a CUDA
        graph.  Returns `fn(actions) -> (obs, reward, terminated, truncated,
        info)` with the same meaning as step(); the returned tensors are
        static buffers that the next call overwrites.  `fn.actions` is the
        graph's own input buffer: filling it in place and passing it to `fn`
        avoids the device copy of the actions.  Philox noise only."""
        assert self.noise == "philox", "graphed step needs noise='philox'"
        dev = self.device
        a_shape = (1, self.num_envs) + self._row
        static_a = torch.zeros(a_shape, dtype=self._adt, device=dev)
        # (discrete observations: int64 states, cast by _observe)
        out = self._alloc_out(1, self._state_dtype, final_obs=False)
        self._step_ctr = torch.zeros(1, dtype=torch.int64, device=dev)

        def body():
            # counter first, so that the step kernel and the renderer are
            # neighbours in the stream: the renderer is then launched as a
            # programmatic dependent of the step and zero-fills the images
            # while the step runs (MDPP_LAUNCH_OVERLAP_PREVIOUS)
            self._step_ctr += 1
            self.rollout(1, actions=static_a, out=out)
            self._step_index -= 1  # the device counter is the clock here
            self._overlap_render = True
            try:
                return self._observe(out["obs"][0])
            finally:
                self._overlap_render = False

        snapshot = [t.clone() for t in self._state_tensors()]
        host_index = self._step_index
        self._step_ctr.fill_(host_index)
        self._use_dev_counter = True
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):  # warm-up: JIT compile, allocator
                    body()
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                obs = body()
        finally:
            self._use_dev_counter = False
        for t, saved in zip(self._state_tensors(), snapshot):
            t.copy_(saved)  # warm-up and capture must not advance the envs
        self._step_index = host_index
        self._step_ctr.fill_(host_index)
        mirror = [host_index]
        epoch = self._seed_epoch

        def step_fn(actions):
            if epoch != self._seed_epoch:
                raise RuntimeError(
                    "the environment was re-seeded after this graphed step was "
                    "captured (its Philox key is baked into the graph): call "
                    "make_graphed_step() again")
            if mirror[0] != self._step_index:  # eager calls happened in between
                self._step_ctr.fill_(self._step_index)
            if not (torch.is_tensor(actions)
                    and actions.data_ptr() == static_a.data_ptr()):
                # (callers that fill `step_fn.actions` in place skip this copy)
                static_a.copy_(torch.as_tensor(actions).reshape(a_shape),
                               non_blocking=True)
            graph.replay()
            self._step_index += 1
            mirror[0] = self._step_index
            self.curr_obs = obs
            return (obs, out["reward"][0], out["terminated"][0],
                    out["truncated"][0], {"state": out["obs"][0]})

        step_fn.graph = graph
        step_fn.actions = static_a[0]  # the graph's input buffer, [N(, ...)]
        return step_fn

    def rollout_host(self, n_steps, actions_host, out_host, chunk_steps=100):
        """rollout() for HOST buffers: `actions_host` [T, N(, D)] and the
        tensors of `out_host` (obs / reward / terminated / truncated, [T, N...])
        are pinned CPU tensors.  The T steps are cut into chunks whose
        host->device copy, kernel and device->host copy run on three streams
        with double-buffered device staging, so PCIe (both directions) and the
        GPU overlap.  Results are complete once the current stream is
        synchronised."""
        T, N = int(n_steps), self.num_envs
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        if not hasattr(self, "_h2d_stream"):
            self._h2d_stream = torch.cuda.Stream(dev)
            self._d2h_stream = torch.cuda.Stream(dev)
            self._stage = {}
        chunk = max(1, min(int(chunk_steps), T))
        # the staging mirrors one chunk of the caller's buffers: any change of
        # their names, dtypes or trailing shapes needs new staging
        key = (chunk, tuple(actions_host.shape[1:]), actions_host.dtype) + tuple(
            (k, v.dtype, tuple(v.shape[1:])) for k, v in sorted(out_host.items()))
        if self._stage.get("key") != key:
            acts = [torch.empty((chunk,) + tuple(actions_host.shape[1:]),
                                dtype=actions_host.dtype, device=dev)
                    for _ in range(2)]
            outs = [{k: torch.empty((chunk,) + tuple(v.shape[1:]), dtype=v.dtype,
                                    device=dev) for k, v in out_host.items()}
                    for _ in range(2)]
            self._stage = {"key": key, "acts": acts, "outs": outs}
        acts, outs = self._stage["acts"], self._stage["outs"]
        ev_in, ev_comp, ev_out = {}, {}, {}
        self._h2d_stream.wait_stream(cur)
        self._d2h_stream.wait_stream(cur)
        n_chunks = (T + chunk - 1) // chunk
        for c in range(n_chunks):
            t0, t1 = c * chunk, min(T, (c + 1) * chunk)
            n, b = t1 - t0, c % 2
            with torch.cuda.stream(self._h2d_stream):
                if c >= 2:  # staging buffer b is free once chunk c-2 has run
                    self._h2d_stream.wait_event(ev_comp[c - 2])
                acts[b][:n].copy_(actions_host[t0:t1], non_blocking=True)
                ev_in[c] = torch.cuda.Event()
                ev_in[c].record(self._h2d_stream)
            cur.wait_event(ev_in[c])
            if c >= 2:  # output staging b is free once chunk c-2 is on the host
                cur.wait_event(ev_out[c - 2])
            self.rollout(n, actions=acts[b][:n],
                         out={k: v[:n] for k, v in outs[b].items()})
            ev_comp[c] = torch.cuda.Event()
            ev_comp[c].record(cur)
            with torch.cuda.stream(self._d2h_stream):
                self._d2h_stream.wait_event(ev_comp[c])
                for k, v in out_host.items():
                    v[t0:t1].copy_(outs[b][k][:n], non_blocking=True)
                ev_out[c] = torch.cuda.Event()
                ev_out[c].record(self._d2h_stream)
        cur.wait_stream(self._d2h_stream)
        return out_host

    def episode_stats(self, reduce=False):
        """Per-group counters of rl_toy_env.py:2360-2369 summed over envs and
        episodes; `reduce=True` all-reduces over torch.distributed ranks."""
        from . import sharding
        total = self._stats.sum(dim=0)  # the kernels spread atomics over slots
        stats = sharding.reduce_stats(total) if reduce else total
        return sharding.summarize_stats(stats)
