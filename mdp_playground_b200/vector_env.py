"""VectorRLToyEnv: N independent RLToyEnv instances stepped by sm_100a kernels.

Drop-in for the reference's `RLToyEnv` on the step path (constructor keys,
`reset` / `step` return tuples, `get_augmented_state`; rl_toy_env.py:216,
:2217, :1992, :2127), batched over a leading env axis.  All state lives in
PyTorch-owned device tensors; every operation is a call into libmdpp_b200.so
(include/mdpp_b200.h) on the current CUDA stream.  There is no CPU path.

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

import numpy as np
import torch

from . import _lib
from .config import np_random, parse_config
from .spaces import BoxSpace, DiscreteSpace
from .tables import build_discrete_tables


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# raw handle of the current stream of a device (the public accessor builds a
# Stream object per call: ~2 us, a third of a 65 536-env step)
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None) or (
    lambda idx: torch.cuda.current_stream(idx).cuda_stream)


class VectorRLToyEnv:
    metadata = {"render_modes": []}

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
        self.num_envs = int(num_envs)
        assert self.num_envs > 0
        self.device = torch.device(
            "cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
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
            kinds = {s_.kind for s_ in self._group_specs}
            if len(kinds) != 1:
                raise NotImplementedError(
                    "config_groups: one state_space_type per launch")
            G = len(cfgs)
            if group_sizes is None:
                from .sharding import even_group_sizes
                group_sizes = even_group_sizes(self.num_envs, G)
            assert len(group_sizes) == G and sum(group_sizes) == self.num_envs
            self._group_sizes = [int(x) for x in group_sizes]
            self.spec = self._group_specs[0]
        else:
            self.spec = parse_config(config)
            self._group_specs = [self.spec]
            self._group_sizes = [self.num_envs]
        self.normal_mode = {
            "fast": _lib.MDPP_NORMAL_FAST, "boxmuller": _lib.MDPP_NORMAL_F64,
            "ziggurat": _lib.MDPP_NORMAL_ZIGGURAT,
            "fp64": _lib.MDPP_NORMAL_ZIGGURAT if self.spec.kind == "discrete"
            else _lib.MDPP_NORMAL_F64}[normal_precision]
        self.config = self.spec.config
        self.seed_dict = self.spec.seed_dict
        if philox_seed is None:
            philox_seed = self.seed_dict["env"]
            if philox_seed is None:
                philox_seed = int(np.random.SeedSequence().entropy & (2**63 - 1))
        self.philox_seed = int(philox_seed) & (2**64 - 1)
        self._step_index = 0
        self._ctx = C.c_void_p()
        _lib.check(self._lib, None,
                   self._lib.mdpp_create(self.device.index, C.byref(self._ctx)))
        if self.spec.kind != "discrete" and self._shard[1] > 1:
            # the discrete path derives global Philox ids from `shard` per group
            # (sharding.group_id_bases), and so do continuous / grid
            # config_groups (which undo this); a single configuration is one
            # group: rank r owns the ids [offset + r N, offset + (r + 1) N)
            self.env_id_offset += self._shard[0] * self.num_envs
        self._seed_epoch = 0
        if self.spec.kind == "discrete":
            self._init_discrete()
        elif self.spec.kind == "grid":
            self._init_grid()
        else:
            self._init_continuous()
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

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------
    # discrete backend
    # ------------------------------------------------------------------
    def _init_discrete(self):
        """One configuration group per entry of self._group_specs (a single
        one for the plain drop-in use).  Envs are laid out group-major: group
        g owns the contiguous range group_slices[g]."""
        sp = self.spec
        N, dev = self.num_envs, self.device
        specs = self._group_specs
        G = len(specs)
        sizes = self._group_sizes
        self.group_tables = [build_discrete_tables(s_) for s_ in specs]
        self.tables = tb = self.group_tables[0]
        self.transition_matrix = tb.transition
        self.rewardable_sequences = tb.rewardable_sequences
        self.reward_matrix = tb.reward_matrix
        self.observation_space = DiscreteSpace(
            tb.n_states, seed=self.seed_dict.get("relevant_state_space"))
        self.action_space = DiscreteSpace(
            tb.n_actions, seed=self.seed_dict.get("relevant_action_space"))
        # irrelevant_features: a second sub-MDP; states, actions and
        # observations become rows (relevant, irrelevant) -- the reference's
        # tuples (rl_toy_env.py:2085-2088)
        self._irr = bool(sp.irrelevant_features)
        assert all(bool(s_.irrelevant_features) == self._irr for s_ in specs), \
            "config_groups must agree on irrelevant_features"
        if self._irr:
            self.transition_matrix_irrelevant = tb.transition_irr
            self.observation_spaces = [
                self.observation_space,
                DiscreteSpace(tb.n_states_irr,
                              seed=self.seed_dict.get("irrelevant_state_space"))]
            self.action_spaces = [
                self.action_space,
                DiscreteSpace(tb.n_actions_irr,
                              seed=self.seed_dict.get("irrelevant_action_space"))]
        self.has_pnoise = any(bool(s_.transition_noise) for s_ in specs)
        self.has_rnoise = any(s_.has_reward_noise for s_ in specs)
        from .sharding import group_id_bases
        rank, world = self._shard
        id_bases = group_id_bases(sizes, rank, world)
        groups = (_lib.DiscreteGroup * G)()
        self._host_keep = []
        begin = 0
        self.group_slices = []
        for gi, (s_, t_) in enumerate(zip(specs, self.group_tables)):
            g = groups[gi]
            g.n_states, g.n_actions = t_.n_states, t_.n_actions
            g.sequence_length, g.delay = s_.sequence_length, s_.delay
            g.reward_every_n_steps = s_.reward_every_n_steps
            g.custom_reward = int(s_.use_custom_mdp)
            g.n_sequences = int(t_.sequences.shape[0])
            g.has_transition_noise = int(bool(s_.transition_noise))
            g.has_reward_noise = int(s_.has_reward_noise)
            g.transition_noise = s_.transition_noise
            g.reward_noise_std = s_.reward_noise_std
            g.reward_scale, g.reward_shift = s_.reward_scale, s_.reward_shift
            g.term_state_reward = s_.term_state_reward
            keep = [t_.transition, t_.terminal_mask, t_.init_cdf, t_.noise_cdf,
                    t_.sequences, t_.sequence_rewards, t_.reward_matrix]
            self._host_keep.append(keep)
            hp = [None if a is None else a.ctypes.data_as(C.c_void_p)
                  for a in keep]
            (g.transition, g.terminal, g.init_cdf, g.noise_cdf, g.sequences,
             g.sequence_rewards, g.reward_matrix) = hp
            if t_.n_states_irr:
                g.n_states_irr, g.n_actions_irr = t_.n_states_irr, t_.n_actions_irr
                keep_irr = [t_.transition_irr, t_.init_cdf_irr, t_.noise_cdf_irr]
                keep.extend(keep_irr)
                (g.transition_irr, g.init_cdf_irr, g.noise_cdf_irr) = [
                    None if a is None else a.ctypes.data_as(C.c_void_p)
                    for a in keep_irr]
            g.env_begin, g.env_count = begin, sizes[gi]
            # global Philox ids: all ranks' envs of group g are contiguous
            g.global_id_base = id_bases[gi]
            self.group_slices.append(slice(begin, begin + sizes[gi]))
            begin += sizes[gi]
        assert begin == N
        self._check(self._lib.mdpp_set_discrete_groups(self._ctx, groups, G))
        self.n_groups = G
        max_delay = max(s_.delay for s_ in specs)

        self._cur = torch.zeros(N, dtype=torch.int32, device=dev)
        self._cur_irr = torch.zeros(N, dtype=torch.int32, device=dev) \
            if self._irr else None
        self._key = torch.zeros(N, dtype=torch.int64, device=dev)
        self._t = torch.zeros(N, dtype=torch.int32, device=dev)
        self._episode = torch.zeros(N, dtype=torch.int32, device=dev)
        self._ring = torch.zeros((max_delay, N), dtype=torch.float64,
                                 device=dev) if max_delay > 0 else None
        self._hist_depth = sp.sequence_length + sp.delay + 1
        if G > 1:
            self.track_history = False  # augmented_state differs per group
        self._history = torch.zeros((self._hist_depth, N), dtype=torch.int32,
                                    device=dev) if self.track_history else None
        self._stats = torch.zeros((_lib.STATS_SLOTS, self.n_groups,
                                   _lib.MDPP_N_STATS),
                                  dtype=torch.float64, device=dev)
        st = _lib.DiscreteState()
        st.n_envs = N
        st.cur_state, st.seq_key = _ptr(self._cur), _ptr(self._key)
        st.t_episode, st.episode = _ptr(self._t), _ptr(self._episode)
        st.ring = _ptr(self._ring)
        st.ring_depth = max_delay
        st.history_depth = self._hist_depth
        st.history = _ptr(self._history)
        st.stats = _ptr(self._stats)
        st.stats_slots = _lib.STATS_SLOTS
        st.cur_state_irr = _ptr(self._cur_irr)
        self._state = st
        if self.noise == "numpy":
            assert G == 1, "noise='numpy' is a single-configuration mode"
            self._init_numpy_streams()

    def _init_numpy_streams(self):
        """Per-lane PCG64 streams; lane 0 = the reference's own (appendix C):
        S continues after the P-table draws, E is re-seeded at the first reset."""
        sd = self.seed_dict
        from .tables import _next_set_probabilities, sub_space_rngs

        def lanes(key, rng0):
            s = sd.get(key)
            return [rng0] + [np_random(None if s is None else s + i)[0]
                             for i in range(1, self.num_envs)]
        rng0, rng1 = sub_space_rngs(self.spec)
        self._rng_S = lanes("relevant_state_space", rng0)
        if self._irr:
            self._rng_S1 = lanes("irrelevant_state_space", rng1)
        if not self.spec.use_custom_mdp:
            # replay lane 0's consumption during P generation
            S, A = self.tables.n_states, self.tables.n_actions
            rng = self._rng_S[0]
            for s in range(S):
                if self.spec.maximally_connected:
                    p = None if self.spec.diameter == 1 else \
                        _next_set_probabilities(s, S, A)
                    rng.choice(S, size=A, p=p, replace=False)
                else:
                    p = _next_set_probabilities(s, S, A)
                    for _ in range(A):
                        rng.choice(S, size=1, p=p)
            if self._irr:
                S1, A1 = self.tables.n_states_irr, self.tables.n_actions_irr
                rng = self._rng_S1[0]
                for s in range(S1):
                    p = _next_set_probabilities(s, S1, A1)
                    if self.spec.maximally_connected:
                        rng.choice(S1, size=A1, p=p, replace=False)
                    else:
                        for _ in range(A1):
                            rng.choice(S1, size=1, p=p)
        self._rng_E = [None] * self.num_envs

    def _opts(self, T, noise_mode=None):
        o = _lib.StepOpts()
        o.n_steps = T
        if noise_mode is None:
            noise_mode = {"philox": _lib.MDPP_NOISE_PHILOX,
                          "replay": _lib.MDPP_NOISE_REPLAY,
                          "numpy": _lib.MDPP_NOISE_REPLAY}[self.noise]
            if not (self.has_pnoise or self.has_rnoise) and self.noise == "philox":
                pass  # philox still drives resets
        o.noise_mode = noise_mode
        o.autoreset = int(self.autoreset)
        o.horizon = self.horizon
        o.normal_mode = self.normal_mode
        o.seed = self.philox_seed
        o.step_index = self._step_index
        o.env_id_offset = self.env_id_offset
        if getattr(self, "_use_dev_counter", False):
            # CUDA-graph mode: the step index lives in a device scalar that
            # the graph itself advances BEFORE the kernels run (see
            # make_graphed_step): index = counter - 1 (mod 2^64)
            o.step_index = 2**64 - 1
            o.step_index_dev = self._step_ctr.data_ptr()
        return o

    # ------------------------------------------------------------------
    def reset(self, seed=None, options=None):
        """(obs, info) like RLToyEnv.reset (:2217).  options: {"mask": bool[N],
        "init_state": int[N], "reset_u": float64[N] (replay mode)}; with
        irrelevant_features init_state / reset_u / obs are [N, 2] rows
        (relevant, irrelevant)."""
        options = options or {}
        if self.spec.kind == "continuous":
            return self._reset_continuous(seed, options)
        if self.spec.kind == "grid":
            return self._reset_grid(seed, options)
        N, dev = self.num_envs, self.device
        mask = options.get("mask")
        if mask is not None:
            mask = torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
        init = options.get("init_state")
        if init is not None:
            init = torch.as_tensor(init, device=dev).to(torch.int32).contiguous()
            self._check_state_range(init)
        reset_u = options.get("reset_u")
        if self.noise == "numpy" and init is None:
            if seed is not None:
                for i in range(N):
                    self._rng_E[i], _ = np_random(seed + i)
            elif self._rng_E[0] is None:
                for i in range(N):
                    self._rng_E[i], _ = np_random(None)
            m = None if mask is None else mask.cpu().numpy()
            reset_u = np.zeros((N, 2) if self._irr else N)
            for i in range(N):
                if m is None or m[i]:  # one E draw per sub-space (:2255-2264)
                    reset_u[i] = [self._rng_E[i].random() for _ in range(2)] \
                        if self._irr else self._rng_E[i].random()
        elif (seed is not None and self.noise == "philox"
              and not options.get("_ctor")):
            # re-keying the counter-based streams is the analogue of re-seeding
            self._reseed(seed, mask, rewind=mask is None)
        if reset_u is not None:
            reset_u = torch.as_tensor(reset_u, dtype=torch.float64,
                                      device=dev).contiguous()
        row = (N, 2) if self._irr else (N,)
        if init is not None:
            assert tuple(init.shape) == row, (tuple(init.shape), row)
        if reset_u is not None:
            assert tuple(reset_u.shape) == row, (tuple(reset_u.shape), row)
        obs = torch.empty(row, dtype=torch.int64, device=dev)
        mode = _lib.MDPP_NOISE_REPLAY if reset_u is not None \
            else _lib.MDPP_NOISE_PHILOX
        if (init is None and reset_u is None and self.noise == "replay"
                and not options.get("_ctor")):
            raise ValueError("replay mode: pass options['reset_u'] or "
                             "options['init_state'] to reset()")
        opts = self._opts(1, mode)
        self._check(self._lib.mdpp_discrete_reset(
            self._ctx, C.byref(self._state), _ptr(mask), _ptr(init),
            _ptr(reset_u), _ptr(obs), C.byref(opts), self._stream()))
        self.curr_obs = self._observe(obs, options.get("image_params"), reset=True,
                                      ctor=bool(options.get("_ctor")))
        return self.curr_obs, {}

    def _check_state_range(self, states):
        """Caller-supplied discrete states index the tables on the device:
        reject anything outside [0, S) (rows (relevant, irrelevant) with
        irrelevant_features) instead of reading out of bounds.  Each env is
        checked against the state count of its own config group."""
        st = states.reshape(self.num_envs, -1)
        for k in range(2 if self._irr else 1):
            self._check_column(st[:, k:k + 1], irr=k == 1,
                               what=f"state in column {k}")

    def _check_column(self, states, irr, what):
        """Raise unless every entry of row i of `states` [N, k] lies in
        [0, S) of env i's config group (S of the irrelevant sub-MDP when
        `irr`): the kernels index that group's tables with it."""
        n = torch.tensor([t.n_states_irr if irr else t.n_states
                          for t in self.group_tables], device=states.device)
        hi = torch.repeat_interleave(
            n, torch.tensor(self._group_sizes, device=states.device))[:, None]
        bad = ((states < 0) | (states >= hi)).any(dim=1)
        if bool(bad.any()):
            i = int(bad.nonzero()[0, 0])
            raise ValueError(f"{what} out of range [0, {int(hi[i, 0])}) at env "
                             f"{i} (its config group's state count)")

    def _observe(self, state, image_params=None, reset=False, ctor=False):
        """Underlying state -> observation (identity, dtype_o cast, or the
        image renderer when image_representations is on)."""
        if self.spec.image_representations:
            return self.render_observation(state, image_params=image_params,
                                           reset=reset, allow_philox=ctor)
        if self.spec.kind in ("continuous", "grid"):
            return state
        return self._cast_obs(state)

    # ------------------------------------------------------------------
    # image observations
    # ------------------------------------------------------------------
    def _init_images(self):
        from . import image_tables as it
        sp, dev = self.spec, self.device
        W, H = sp.image_width, sp.image_height
        self._img_keep = []

        def up(a, dtype):
            t = torch.as_tensor(np.ascontiguousarray(a)).to(dtype).to(dev).contiguous()
            self._img_keep.append(t)
            return _ptr(t)
        if sp.kind == "discrete":
            tb = it.build_discrete_image_tables(
                max(self.tables.n_states, self.tables.n_states_irr), W, H,
                sp.image_transforms,
                sp.image_sh_quant, sp.image_ro_quant, sp.image_scale_range)
            self.image_tables = tb
            c = _lib.ImageDiscreteTables()
            c.width, c.height, c.n_states = W, H, tb.n_states
            c.r_min, c.n_radii = tb.r_min, tb.n_radii
            c.n_xvar, c.n_yvar = tb.n_xvar, tb.n_yvar
            c.has_scale, c.has_shift = int(tb.has_scale), int(tb.has_shift)
            c.has_rotate, c.has_flip = int(tb.has_rotate), int(tb.has_flip)
            c.sh_quant, c.ro_quant = tb.sh_quant, tb.ro_quant
            c.mask_bits = up(tb.mask_bits.view(np.int64), torch.int64)
            c.mask_index = up(tb.mask_index, torch.int32)
            c.xvar, c.yvar = up(tb.xvar, torch.uint8), up(tb.yvar, torch.uint8)
            c.rot_coeff = up(tb.rot_coeff, torch.int32)
            c.r_thresholds = up(tb.r_thresholds if len(tb.r_thresholds)
                                else np.zeros(1), torch.float64)
            # irrelevant_features: one polygon image per sub-state, stacked
            # along x (image_multi_discrete.py:272-288)
            self._n_sub = 2 if self._irr else 1
            c.n_sub_images = self._n_sub
            self._img_cfg = c
            self.obs_shape = (W * self._n_sub, H, 1)
            if self.noise == "numpy":
                s = self.seed_dict.get("image_representations")
                self._rng_I = [np_random(None if s is None else s + i)[0]
                               for i in range(self.num_envs)]
        elif sp.kind == "grid":
            # ImageContinuous with grid_shape (image_continuous.py:139-207):
            # white grid lines, black terminal cells, green target and blue
            # agent discs at the cell centres (+0.5), per sub-grid
            nd, gs = self._nd, sp.grid_shape
            if W > 256 or H > 256:
                raise NotImplementedError("grid images: width, height <= 256")
            hi = np.array(gs[:2], dtype=np.int64)

            def to_pixel(vec):  # image_continuous.py:248-277 over Box(0, shape)
                frac = (np.asarray(vec) - 0) / (hi - 0)
                return (frac * (W, H)).astype(int)
            c = _lib.ImageContinuousConfig()
            c.width, c.height, c.dim = W, H, nd
            c.n_sub_images = nd // 2
            for k in range(2):
                c.rel_index[k], c.irr_index[k] = k, (2 + k if nd == 4 else 0)
                c.feat_low[k], c.feat_high[k] = 0.0, float(hi[k])
            c.is_f64 = 1
            cells = sp.terminal_cells or []
            if len(cells) > _lib.MDPP_MAX_TERM_BOXES:
                raise NotImplementedError("at most 8 terminal cells in images")
            c.n_rects = len(cells)
            for b, cell in enumerate(cells):
                lo_ = np.array(cell, dtype=np.float64).astype(np.int64)
                p0, p1 = to_pixel(lo_), to_pixel(lo_ + 1.0)
                c.rect[b][0], c.rect[b][1] = int(p0[0]), int(p0[1])
                c.rect[b][2], c.rect[b][3] = int(p1[0]), int(p1[1])
            c.has_target = 1
            tp = to_pixel(np.array(sp.target_point, dtype=float) + 0.5)
            c.target_pixel[0], c.target_pixel[1] = int(tp[0]), int(tp[1])
            spans = it.disc_stamp(5)
            c.stamp_rows, c.stamp_radius = len(spans), 5
            for r, (x0, wdt) in enumerate(spans):
                c.stamp[r][0], c.stamp[r][1] = int(x0), int(wdt)
            for sub in range(nd // 2):
                off = 2 * sub
                for i in range(1, gs[off] + 1):      # vertical lines (:141-151)
                    x = i * W // gs[off] - 1
                    if 0 <= x < W:
                        c.vline[sub][x >> 6] |= 1 << (x & 63)
                for j in range(1, gs[off + 1]):      # horizontal (:153-160; the
                    y = j * H // gs[off]             # divisor is the FIRST extent)
                    if 0 <= y < H:
                        c.hline[sub][y >> 6] |= 1 << (y & 63)
            self._img_cfg = c
            self.obs_shape = (W * c.n_sub_images, H, 3)
        else:
            D = sp.state_space_dim
            assert np.isfinite(sp.state_space_max), \
                "image observations need a bounded state space"
            rel = [0, 1]  # ImageContinuous default; the env does not pass its own
            irr = sorted(set(range(D)) - set(rel))
            if D < 2 or len(irr) not in (0, 2):
                raise NotImplementedError(
                    "continuous image observations: 2 relevant (+ 0 or 2 "
                    "irrelevant) dimensions")
            dt = self._np_real
            lo = np.full((D,), -sp.state_space_max).astype(dt)[rel]
            hi = np.full((D,), sp.state_space_max).astype(dt)[rel]

            def to_pixel(vec):  # image_continuous.py:248-277
                frac = (np.asarray(vec) - lo) / (hi - lo)
                return (frac * (W, H)).astype(int)
            c = _lib.ImageContinuousConfig()
            c.width, c.height, c.dim = W, H, D
            c.n_sub_images = 2 if irr else 1
            for k in range(2):
                c.rel_index[k] = rel[k]
                c.irr_index[k] = irr[k] if irr else 0
                c.feat_low[k], c.feat_high[k] = float(lo[k]), float(hi[k])
            c.is_f64 = int(self._real == torch.float64)
            c.n_rects = len(self._term_lows)
            for b, (tl_, th_) in enumerate(zip(self._term_lows, self._term_highs)):
                p0, p1 = to_pixel(tl_), to_pixel(th_)
                c.rect[b][0], c.rect[b][1] = int(p0[0]), int(p0[1])
                c.rect[b][2], c.rect[b][3] = int(p1[0]), int(p1[1])
            c.has_target = 1
            tp = to_pixel(np.asarray(sp.target_point, dtype=dt))
            c.target_pixel[0], c.target_pixel[1] = int(tp[0]), int(tp[1])
            spans = it.disc_stamp(5)  # circle_radius=5 (rl_toy_env.py:774)
            c.stamp_rows, c.stamp_radius = len(spans), 5
            for r, (x0, wdt) in enumerate(spans):
                c.stamp[r][0], c.stamp[r][1] = int(x0), int(wdt)
            self._img_cfg = c
            self.obs_shape = (W * c.n_sub_images, H, 3)

    def _numpy_image_params(self, states_host):
        """The reference's I-stream draws (image_multi_discrete.py:149-181,
        :251, :258-259), one image per lane, lane 0 = the reference."""
        tb, sp = self.image_tables, self.spec
        W, H = tb.width, tb.height
        n_sub = self._n_sub
        out = np.zeros((self.num_envs * n_sub, 5), dtype=np.int32)
        for i in range(self.num_envs * n_sub):
            rng = self._rng_I[i // n_sub]  # sub-images drawn in order
            R, sw, sh, rot, flip = 20, int(W / 2), int(H / 2), -1, 0
            if tb.has_scale:
                lo, hi = sp.image_scale_range
                mx, mn = np.log(hi * 20), np.log(lo * 20)
                R = int(np.exp(mn + rng.random() * (mx - mn)))
            if tb.has_shift:
                mw, mh = W / 2 - R, H / 2 - R
                aw = rng.integers(-mw + 1, mw).item()
                ah = rng.integers(-mh + 1, mh).item()
                sw += (aw // tb.sh_quant) * tb.sh_quant
                sh += (ah // tb.sh_quant) * tb.sh_quant
            if tb.has_rotate:
                rot = (rng.integers(360).item() // tb.ro_quant) * tb.ro_quant
            if tb.has_flip:
                if rng.integers(2).item() == 0:
                    flip = 1 if rng.integers(2).item() == 0 else 2
            out[i] = (R, sw, sh, rot, flip)
        return out

    def render_observation(self, state, image_params=None, reset=False,
                           step_index=None, allow_philox=False):
        """State tensor -> uint8 image observations on the GPU.
        discrete: int64 [..., N] -> [..., N, W, H, 1]; continuous:
        real [..., N, D] -> [..., N, k*W, H, 3]."""
        sp, dev = self.spec, self.device
        N = self.num_envs
        if step_index is None:
            step_index = self._step_index
        opts = self._opts(1)
        if not getattr(self, "_use_dev_counter", False):
            opts.step_index = step_index
        else:  # observation after the step: index + 1 = the device counter
            opts.step_index = 0
        if sp.kind == "discrete":
            st = state.to(torch.int64).contiguous()
            M = st.numel()  # images = sub-images when irrelevant_features
            lead = tuple(st.shape[:-1]) if self._irr else tuple(st.shape)
            if self.noise == "numpy" and image_params is None:
                assert M == N * self._n_sub, \
                    "noise='numpy' renders one step at a time"
                image_params = self._numpy_image_params(None)
            if image_params is not None:
                image_params = torch.as_tensor(image_params, device=dev).to(
                    torch.int32).reshape(M, 5).contiguous()
            elif self.noise == "replay" and not allow_philox and (
                    self.image_tables.has_scale or self.image_tables.has_shift
                    or self.image_tables.has_rotate or self.image_tables.has_flip):
                raise ValueError("replay mode: pass image_params [N, 5]")
            out = torch.empty(lead + self.obs_shape, dtype=torch.uint8, device=dev)
            self.last_image_params = torch.empty((M, 5), dtype=torch.int32,
                                                 device=dev)
            if getattr(self, "_overlap_render", False) and st.data_ptr() == state.data_ptr():
                # (no cast / copy kernel sits between the step and this launch)
                opts.flags = _lib.MDPP_LAUNCH_OVERLAP_PREVIOUS
            self._check(self._lib.mdpp_render_discrete(
                self._ctx, C.byref(self._img_cfg), _ptr(st), _ptr(image_params),
                _ptr(self.last_image_params), _ptr(out), M, N,
                6 if reset else 3, C.byref(opts), self._stream()))
            return out
        if sp.kind == "grid":  # cell centres, float64 like the reference
            st = (state.to(torch.float64) + 0.5).contiguous()
            M = st.numel() // self._nd
        else:
            st = state.to(self._real).contiguous()
            M = st.numel() // sp.state_space_dim
        lead = tuple(st.shape[:-1])
        out = torch.empty(lead + self.obs_shape, dtype=torch.uint8, device=dev)
        self._check(self._lib.mdpp_render_continuous(
            self._ctx, C.byref(self._img_cfg), _ptr(st), _ptr(out), M,
            self._stream()))
        return out

    _OBS_CODES = {torch.int64: _lib.MDPP_OBS_I64, torch.int32: _lib.MDPP_OBS_I32,
                  torch.uint8: _lib.MDPP_OBS_U8}

    def _obs_torch_dtype(self):
        """dtype the discrete kernels write observations in: the config's
        dtype_o (rl_toy_env.py:571, :611-614) when it is int64 / int32 / uint8
        (written in-kernel), else int64 followed by a cast."""
        forced = getattr(self, "_obs_dtype_override", None)
        if forced is not None:
            return forced
        if self.spec.image_representations:
            return torch.int64  # states feed the renderer, not the caller
        dt = getattr(torch, np.dtype(self.spec.dtype_o).name, None)
        if dt == torch.uint8 and self.tables.n_states > 256:
            dt = None
        return dt if dt in self._OBS_CODES else torch.int64

    def set_obs_dtype(self, dtype):
        """Override dtype_o for the observations rollout() / step() write
        (torch.int64 / int32 / uint8): 8 -> 1 byte per env-step of output for
        the toy state spaces.  Not for image envs: their observations are
        the images, and the renderer reads the int64 states."""
        if self.spec.image_representations:
            raise ValueError("set_obs_dtype: image observations are uint8 "
                             "images already; the states stay int64")
        assert dtype in self._OBS_CODES
        if dtype == torch.uint8:
            assert max(self.tables.n_states, self.tables.n_states_irr or 0) <= 256
        self._obs_dtype_override = dtype
        self._io_cache = None
        self._step_sets = None

    def _cast_obs(self, obs):
        target = getattr(self, "_obs_dtype_override", None) or getattr(
            torch, np.dtype(self.spec.dtype_o).name)
        return obs if obs.dtype == target else obs.to(target)

    def step(self, actions, replay=None):
        """(obs, reward, terminated, truncated, info) like RLToyEnv.step
        (:1992).  `replay`: dict with "transition_u", "reward_noise",
        "reset_u" float64[N] arrays (noise='replay').  info["state"] is the
        underlying state, info["final_obs"] (autoreset only) the state before
        the same-step reset."""
        if (replay is None and self.noise == "philox" and self._step_buffers > 0
                and (not self.spec.image_representations
                     or self.spec.kind == "discrete")
                and not getattr(self, "_use_dev_counter", False)):
            return self._step_fast(actions)
        N = self.num_envs
        actions = torch.as_tensor(actions)
        if self.spec.kind == "continuous":
            actions = actions.reshape(1, N, self.spec.state_space_dim)
        elif self.spec.kind == "grid":
            actions = actions.reshape(1, N, len(self.spec.grid_shape))
        elif self._irr:
            actions = actions.reshape(1, N, 2)
        else:
            actions = actions.reshape(1, N)
        out = self.rollout(1, actions=actions,
                           replay=None if replay is None else
                           {k: torch.as_tensor(v).reshape((1,) + tuple(
                               torch.as_tensor(v).shape))
                            for k, v in replay.items()})
        state = out["obs"][0]
        obs = self._observe(
            state, None if replay is None else replay.get("image_params"))
        self.curr_obs = obs
        return (obs, out["reward"][0], out["terminated"][0],
                out["truncated"][0],
                {"final_obs": out["final_obs"][0], "state": state})

    # -- step() without per-call allocation / marshalling -------------------
    def _build_step_sets(self):
        """`step_buffers` output sets, each with its I/O struct marshalled once
        and the tuple step() returns built once."""
        N, dev, kind = self.num_envs, self.device, self.spec.kind
        if kind == "continuous":
            row, odt, rdt = (1, N, self.spec.state_space_dim), self._real, self._real
            io_cls, self._step_fn = _lib.ContinuousIO, self._lib.mdpp_continuous_rollout
            self._step_adt = self._real
        elif kind == "grid":
            row, odt, rdt = (1, N, self._nd), torch.int64, torch.float64
            io_cls, self._step_fn = _lib.GridIO, self._lib.mdpp_grid_rollout
            self._step_adt = torch.int64
        else:
            row = (1, N, 2) if self._irr else (1, N)
            odt, rdt = self._obs_torch_dtype(), torch.float64
            io_cls, self._step_fn = _lib.DiscreteIO, self._lib.mdpp_discrete_rollout
            self._step_adt = torch.int32
        self._step_arow = row
        self._step_numel = int(np.prod(row))
        self._dev_index = self.device.index
        sets = []
        for _ in range(self._step_buffers):
            out = {"obs": torch.empty(row, dtype=odt, device=dev),
                   "reward": torch.empty((1, N), dtype=rdt, device=dev),
                   "terminated": torch.empty((1, N), dtype=torch.bool, device=dev),
                   "truncated": torch.empty((1, N), dtype=torch.bool, device=dev)}
            if self.autoreset:
                out["final_obs"] = torch.empty(row, dtype=odt, device=dev)
            io = io_cls()
            io.obs, io.reward = _ptr(out["obs"]), _ptr(out["reward"])
            io.final_obs = _ptr(out.get("final_obs"))
            io.terminated, io.truncated = _ptr(out["terminated"]), _ptr(out["truncated"])
            if kind == "discrete":
                io.obs_dtype = self._OBS_CODES[odt]
            state = out["obs"][0]
            obs = state  # (replaced per call when dtype_o needs a cast)
            render = None
            if kind == "discrete" and self.spec.image_representations:
                # the renderer runs as a programmatic dependent of the step
                # kernel (its zero fill overlaps it), marshalled once as well
                M = state.numel()
                img = torch.empty(tuple(state.shape[:1]) + self.obs_shape,
                                  dtype=torch.uint8, device=dev)
                prm = torch.empty((M, 5), dtype=torch.int32, device=dev)
                ropts = self._opts(1)
                ropts.flags = _lib.MDPP_LAUNCH_OVERLAP_PREVIOUS
                render = (ropts, C.byref(ropts), _ptr(state), _ptr(prm), _ptr(img),
                          M, prm)
                obs = img
            info = {"state": state}
            if self.autoreset:
                info["final_obs"] = out["final_obs"][0]
            ret = (obs, out["reward"][0], out["terminated"][0], out["truncated"][0], info)
            sets.append((io, C.byref(io), ret, out, render))
        self._step_sets = sets
        self._step_opts = self._opts(1)
        if kind == "continuous" and not (self.has_pnoise or self.has_rnoise) \
                and not self.autoreset:
            self._step_opts.noise_mode = _lib.MDPP_NOISE_OFF
        self._step_opts_ref = C.byref(self._step_opts)
        if self.spec.image_representations and kind == "discrete":
            self._img_cfg_ref = C.byref(self._img_cfg)
        self._step_state_ref = C.byref(self._state)
        # dtype_o values the kernels do not write (e.g. int16): cast per call
        self._step_cast = kind == "discrete" and \
            not self.spec.image_representations and \
            self._cast_obs(sets[0][3]["obs"][0]).dtype != odt

    def _step_fast(self, actions):
        sets = self._step_sets
        if sets is None:
            self._build_step_sets()
            sets = self._step_sets
        if not (torch.is_tensor(actions) and actions.dtype == self._step_adt
                and actions.is_cuda and actions.is_contiguous()):
            actions = torch.as_tensor(actions, device=self.device)
            if self.spec.kind == "continuous":
                actions = self._continuous_actions(actions)
            elif self.spec.kind == "grid":
                actions = self._grid_actions(actions)
            else:
                actions = actions.to(self._step_adt).contiguous()
        if actions.numel() != self._step_numel:
            raise AssertionError((tuple(actions.shape), self._step_arow))
        flip = self._step_flip
        io, io_ref, ret, _, render = sets[flip]
        self._step_flip = flip + 1 if flip + 1 < len(sets) else 0
        io.actions = actions.data_ptr()
        o = self._step_opts
        o.step_index = self._step_index
        o.seed = self.philox_seed
        rc = self._step_fn(self._ctx, self._step_state_ref, io_ref, self._step_opts_ref,
                           _raw_stream(self._dev_index))
        if rc:
            self._check(rc)
        self._step_index += 1
        if render is not None:
            ropts, ropts_ref, st_p, prm_p, img_p, M, prm = render
            ropts.step_index = self._step_index  # the observation AFTER the step
            ropts.seed = self.philox_seed
            rc = self._lib.mdpp_render_discrete(
                self._ctx, self._img_cfg_ref, st_p, None, prm_p, img_p, M,
                self.num_envs, 3, ropts_ref, _raw_stream(self._dev_index))
            if rc:
                self._check(rc)
            self.last_image_params = prm
        if self._step_cast:
            ret = (self._cast_obs(ret[4]["state"]),) + ret[1:]
        self.curr_obs = ret[0]
        return ret

    def rollout(self, n_steps, actions=None, replay=None, out=None,
                want_final_obs=True):
        """T fused steps in ONE kernel launch.  actions: int[T, N] tensor or
        None (uniform random policy drawn on device).  Returns dict of
        time-major [T, N] tensors: obs, final_obs, reward, terminated,
        truncated."""
        if self.spec.kind == "continuous":
            return self._rollout_continuous(n_steps, actions, replay, out,
                                            want_final_obs)
        if self.spec.kind == "grid":
            return self._rollout_grid(n_steps, actions, replay, out,
                                      want_final_obs)
        T, N, dev = int(n_steps), self.num_envs, self.device
        # step()-granularity callers repeat the same launch (same action and
        # output buffers): reuse the marshalled I/O struct -- the Python side is
        # what bounds a T = 1 call (a 5 us kernel)
        fast_key = None
        if (out is not None and self.noise == "philox" and torch.is_tensor(actions)
                and actions.dtype == torch.int32 and actions.is_cuda
                and actions.is_contiguous()):
            fast_key = (T, actions.data_ptr(), tuple(actions.shape)) + tuple(
                (k, v.data_ptr(), v.dtype) for k, v in out.items())
            hit = getattr(self, "_io_cache", None)
            if hit is not None and hit[0] == fast_key:
                opts = self._opts(T)
                self._check(self._lib.mdpp_discrete_rollout(
                    self._ctx, C.byref(self._state), C.byref(hit[1]),
                    C.byref(opts), self._stream()))
                self._step_index += T
                return out
        row = (T, N, 2) if self._irr else (T, N)  # (relevant, irrelevant) rows
        if actions is not None:
            actions = torch.as_tensor(actions, device=dev)
            if actions.dtype != torch.int32:
                actions = actions.to(torch.int32)
            actions = actions.contiguous()
            assert actions.shape == row, (actions.shape, row)
        io = _lib.DiscreteIO()
        if out is None:
            odt = self._obs_torch_dtype()
            out = {
                "obs": torch.empty(row, dtype=odt, device=dev),
                "reward": torch.empty((T, N), dtype=torch.float64, device=dev),
                "terminated": torch.empty((T, N), dtype=torch.bool, device=dev),
                "truncated": torch.empty((T, N), dtype=torch.bool, device=dev),
            }
            if want_final_obs:
                out["final_obs"] = torch.empty(row, dtype=odt, device=dev)
        io.actions = _ptr(actions)
        # the kernels write observations in the dtype of the caller's buffer
        odt = out["obs"].dtype if out.get("obs") is not None else torch.int64
        if odt not in self._OBS_CODES or (
                out.get("final_obs") is not None and out["final_obs"].dtype != odt):
            raise TypeError("obs / final_obs buffers must both be int64, int32 or uint8")
        io.obs_dtype = self._OBS_CODES[odt]
        io.obs, io.reward = _ptr(out.get("obs")), _ptr(out.get("reward"))
        io.final_obs = _ptr(out.get("final_obs"))
        io.terminated = _ptr(out.get("terminated"))
        io.truncated = _ptr(out.get("truncated"))
        keep = []
        if self.noise == "numpy":
            replay = self._draw_numpy(T)
        if self.noise in ("replay", "numpy"):
            replay = replay or {}
            for name, field in (("transition_u", "replay_transition_u"),
                                ("reward_noise", "replay_reward_noise"),
                                ("reset_u", "replay_reset_u")):
                if name in replay and replay[name] is not None:
                    t = torch.as_tensor(replay[name], dtype=torch.float64,
                                        device=dev).reshape(T, N)
                    if self._irr and name != "reward_noise":
                        # the irrelevant sub-space's draw rides in the same row
                        t1 = replay.get("irr_" + name)
                        t1 = torch.zeros_like(t) if t1 is None else torch.as_tensor(
                            t1, dtype=torch.float64, device=dev).reshape(T, N)
                        t = torch.stack([t, t1], dim=-1)
                    t = t.contiguous()
                    keep.append(t)
                    setattr(io, field, _ptr(t))
        opts = self._opts(T)
        self._check(self._lib.mdpp_discrete_rollout(
            self._ctx, C.byref(self._state), C.byref(io), C.byref(opts),
            self._stream()))
        self._step_index += T
        if fast_key is not None:  # (holds the tensors, so the pointers stay valid)
            self._io_cache = (fast_key, io, actions, dict(out))
        return out

    # ------------------------------------------------------------------
    # CUDA-graph step: the gym-style path without per-step launch overhead
    # ------------------------------------------------------------------
    def _state_tensors(self):
        names = ("_cur", "_cur_irr", "_key", "_t", "_episode", "_ring", "_history",
                 "_stats", "_derivs", "_emitted", "_reached", "_pos", "_prev",
                 "_hist_line")
        return [getattr(self, n) for n in names
                if getattr(self, n, None) is not None]

    def make_graphed_step(self):
        """Capture one step() -- the step kernel, the renderer when images
        are on, and the advance of the Philox step counter -- into a CUDA
        graph.  Returns `fn(actions) -> (obs, reward, terminated, truncated,
        info)` with the same meaning as step(); the returned tensors are
        static buffers that the next call overwrites.  `fn.actions` is the
        graph's own input buffer: filling it in place and passing it to `fn`
        avoids the device copy of the actions.  Philox noise only."""
        assert self.noise == "philox", "graphed step needs noise='philox'"
        N, dev = self.num_envs, self.device
        cont = self.spec.kind == "continuous"
        grid = self.spec.kind == "grid"
        D = self.spec.state_space_dim
        if grid:
            a_shape = (1, N, len(self.spec.grid_shape))
        else:
            a_shape = (1, N, D) if cont else ((1, N, 2) if self._irr else (1, N))
        static_a = torch.zeros(a_shape, dtype=self._real if cont else (
            torch.int64 if grid else torch.int32), device=dev)
        if cont:
            out = {"obs": torch.empty((1, N, D), dtype=self._real, device=dev),
                   "reward": torch.empty((1, N), dtype=self._real, device=dev)}
        else:
            out = {"obs": torch.empty(a_shape, dtype=torch.int64, device=dev),
                   "reward": torch.empty((1, N), dtype=torch.float64, device=dev)}
        out["terminated"] = torch.empty((1, N), dtype=torch.bool, device=dev)
        out["truncated"] = torch.empty((1, N), dtype=torch.bool, device=dev)
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

    def _draw_numpy(self, T):
        assert not self.autoreset, \
            "noise='numpy' needs explicit resets (draw order is host-driven)"
        N = self.num_envs
        rep = {}
        if self.has_pnoise:
            rep["transition_u"] = np.array(
                [[self._rng_S[i].random() for i in range(N)] for _ in range(T)])
        if self.has_rnoise:
            std = self.spec.reward_noise_std
            rep["reward_noise"] = np.array(
                [[self._rng_E[i].normal(0, std) for i in range(N)]
                 for _ in range(T)])
        if self.has_pnoise and self._irr:  # S' stream (:2075)
            rep["irr_transition_u"] = np.array(
                [[self._rng_S1[i].random() for i in range(N)] for _ in range(T)])
        return rep

    # ------------------------------------------------------------------
    # continuous backend (move_to_a_point)
    # ------------------------------------------------------------------
    def _continuous_cfg(self, sp, config, np_dt):
        """mdpp_continuous_config of one parsed config (one group)."""
        D = sp.state_space_dim
        c = _lib.ContinuousConfig()
        c.dim, c.order = D, sp.dynamics_order
        c.n_relevant = len(sp.relevant_indices)
        c.delay, c.reward_every_n_steps = sp.delay, sp.reward_every_n_steps
        c.dense = int(sp.make_denser)
        c.has_transition_noise = int(sp.has_transition_noise)
        c.has_reward_noise = int(sp.has_reward_noise)
        c.image_mode = int(sp.image_representations)
        c.target_is_f64 = int("target_point" not in config
                              and sp.reward_function == "move_to_a_point")
        c.is_f64 = int(np_dt == np.float64)
        # inertia: float, or one value per dimension (rl_toy_env.py:519-537); a
        # list / float64 array promotes `action / inertia` to float64 (:1654)
        if np.ndim(sp.inertia) == 0:
            c.inertia, c.inertia_mode = float(sp.inertia), 0
        else:
            iv = np.asarray(sp.inertia)
            if iv.shape != (D,):
                raise ValueError(f"inertia must be a scalar or have shape ({D},)")
            c.inertia = 1.0
            c.inertia_mode = 1 if iv.dtype == np_dt else 2
            for k in range(D):
                c.inertia_vec[k] = float(iv[k])
        c.time_unit = float(sp.time_unit)
        c.state_space_max = float(sp.state_space_max)
        c.action_space_max = float(sp.action_space_max)
        c.target_radius = float(sp.target_radius)
        c.action_loss_weight = float(sp.action_loss_weight)
        c.transition_noise_std = sp.transition_noise
        c.reward_noise_std = sp.reward_noise_std
        c.reward_scale, c.reward_shift = sp.reward_scale, sp.reward_shift
        c.term_state_reward = sp.term_state_reward
        for k, i in enumerate(sp.relevant_indices):
            c.relevant_indices[k] = i
        line = sp.reward_function == "move_along_a_line"
        c.reward_kind = _lib.MDPP_REWARD_LINE if line else _lib.MDPP_REWARD_POINT
        c.sequence_length = sp.sequence_length
        if line:
            if sp.sequence_length > 128:
                raise NotImplementedError("move_along_a_line: sequence_length <= 128")
            if sp.image_representations:
                raise NotImplementedError("move_along_a_line with image observations")
        else:
            tp = np.asarray(sp.target_point, dtype=np.float64)
            assert tp.shape[0] == c.n_relevant, \
                "target_point must have one entry per relevant index"
            for k in range(c.n_relevant):
                c.target_point[k] = float(tp[k])
        # terminal hypercubes (:895-952); Box casts its bounds to dtype_s
        term_lows, term_highs = [], []
        for centre in (sp.terminal_centres or []):
            lo = np.array([x - sp.term_state_edge / 2 for x in centre]).astype(np_dt)
            hi = np.array([x + sp.term_state_edge / 2 for x in centre]).astype(np_dt)
            term_lows.append(lo)
            term_highs.append(hi)
        if len(term_lows) > _lib.MDPP_MAX_TERM_BOXES:
            raise NotImplementedError("at most 8 terminal regions")
        c.n_term_boxes = len(term_lows)
        for b, (lo, hi) in enumerate(zip(term_lows, term_highs)):
            for k in range(c.n_relevant):
                c.term_low[b * _lib.MDPP_MAX_DIM + k] = float(lo[k])
                c.term_high[b * _lib.MDPP_MAX_DIM + k] = float(hi[k])
        return c, term_lows, term_highs

    def _init_continuous(self):
        sp = self.spec
        D, N, dev = sp.state_space_dim, self.num_envs, self.device
        if D > _lib.MDPP_MAX_DIM or sp.dynamics_order > _lib.MDPP_MAX_ORDER:
            raise NotImplementedError("state_space_dim <= 16 and order <= 4")
        np_dt = np.dtype(sp.dtype_s)
        if np_dt not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise NotImplementedError("continuous dtype_s must be float32/64")
        self._real = torch.float64 if np_dt == np.float64 else torch.float32
        self._np_real = np_dt.type
        self.observation_space = BoxSpace(
            -sp.state_space_max, sp.state_space_max, (D,), np_dt,
            seed=self.seed_dict.get("state_space"))
        self.action_space = BoxSpace(
            -sp.action_space_max, sp.action_space_max, (D,), np_dt,
            seed=self.seed_dict.get("action_space"))
        specs = self._group_specs
        G = len(specs)
        cfgs = []
        for gi, s_ in enumerate(specs):
            if (s_.state_space_dim != D
                    or list(s_.relevant_indices) != list(sp.relevant_indices)
                    or np.dtype(s_.dtype_s) != np_dt
                    or s_.reward_function != sp.reward_function
                    or s_.image_representations != sp.image_representations):
                raise ValueError(
                    "config_groups of continuous envs must agree on state_space_dim, "
                    "relevant_indices, dtype_s, "
                    "reward_function and image_representations (group %d)" % gi)
            cfgs.append(self._continuous_cfg(s_, s_.config, np_dt))
        c, self._term_lows, self._term_highs = cfgs[0]
        line = sp.reward_function == "move_along_a_line"
        self.has_pnoise = any(s_.has_transition_noise for s_ in specs)
        self.has_rnoise = any(s_.has_reward_noise for s_ in specs)
        max_delay = max(s_.delay for s_ in specs)

        def ring64(cc):
            return bool(self._real == torch.float32 and (
                (cc.target_is_f64 and cc.dense) or line))
        if G > 1:
            if sp.image_representations or self.noise == "numpy":
                raise NotImplementedError(
                    "config_groups of continuous envs: no images, no noise='numpy'")
            if len({ring64(cc) for cc, _, _ in cfgs}) != 1 or (
                    line and len({s_.sequence_length for s_ in specs}) != 1):
                raise ValueError(
                    "config_groups of continuous envs must agree on make_denser / "
                    "default target_point (the reward FIFO's dtype) and, for "
                    "move_along_a_line, on sequence_length")
            from .sharding import group_id_bases
            id_bases = group_id_bases(self._group_sizes, *self._shard)
            groups = (_lib.ContinuousGroup * G)()
            begin = 0
            self.group_slices = []
            for gi, (cc, _, _) in enumerate(cfgs):
                groups[gi].cfg = cc
                groups[gi].env_begin, groups[gi].env_count = begin, self._group_sizes[gi]
                groups[gi].global_id_base = id_bases[gi]
                self.group_slices.append(slice(begin, begin + self._group_sizes[gi]))
                begin += self._group_sizes[gi]
            assert begin == N
            if self._shard[1] > 1:  # (ids come from the groups, not from the offset)
                self.env_id_offset -= self._shard[0] * self.num_envs
            self._check(self._lib.mdpp_set_continuous_groups(self._ctx, groups, G))
        else:
            self._check(self._lib.mdpp_set_continuous_config(self._ctx, C.byref(c)))
        self.n_groups = G
        real = self._real
        self._max_order = max(s_.dynamics_order for s_ in specs)
        self._derivs = torch.zeros((self._max_order + 1, D, N), dtype=real,
                                   device=dev)
        self._emitted = torch.zeros((D, N), dtype=real, device=dev)
        self._t = torch.zeros(N, dtype=torch.int32, device=dev)
        self._episode = torch.zeros(N, dtype=torch.int32, device=dev)
        self._reached = torch.zeros(N, dtype=torch.uint8, device=dev)
        # (fp32 env + default float64 target_point + dense reward: the reward is
        # a python float all the way through the reference's reward_buffer)
        ring_dt = torch.float64 if ring64(c) else real
        # move_along_a_line: the last sequence_length emitted relevant states
        self._hist_line = torch.zeros((sp.sequence_length, c.n_relevant, N),
                                      dtype=real, device=dev) if line else None
        self._ring = torch.zeros((max_delay, N), dtype=ring_dt, device=dev) \
            if max_delay > 0 else None
        self._stats = torch.zeros((_lib.STATS_SLOTS, G, _lib.MDPP_N_STATS),
                                  dtype=torch.float64, device=dev)
        st = _lib.ContinuousState()
        st.n_envs = N
        st.derivs, st.emitted = _ptr(self._derivs), _ptr(self._emitted)
        st.t_episode, st.episode = _ptr(self._t), _ptr(self._episode)
        st.reached, st.ring = _ptr(self._reached), _ptr(self._ring)
        st.stats = _ptr(self._stats)
        st.stats_slots = _lib.STATS_SLOTS
        st.hist = _ptr(self._hist_line)
        self._state = st
        self._history = None
        if self.noise == "numpy":
            self._rng_F = [np_random(None if self.seed_dict.get("state_space") is None
                                     else self.seed_dict["state_space"] + i)[0]
                           for i in range(N)]
            self._rng_E = [None] * N

    def _host_box_sample(self, rng):
        """gymnasium Box.sample of the feature space + the reference's
        rejection of terminal regions (rl_toy_env.py:2284-2307)."""
        sp = self.spec
        D = sp.state_space_dim
        rel = sp.relevant_indices
        while True:
            if np.isinf(sp.state_space_max):
                s = rng.normal(size=(D,))
            else:
                hi = np.full((D,), sp.state_space_max).astype(self._np_real)
                s = rng.uniform(low=-hi, high=hi, size=(D,))
            s = s.astype(self._np_real)
            if not any(np.all(s[rel] >= lo) and np.all(s[rel] <= hi)
                       for lo, hi in zip(self._term_lows, self._term_highs)):
                return s

    def _reset_continuous(self, seed, options):
        N, dev, D = self.num_envs, self.device, self.spec.state_space_dim
        mask = options.get("mask")
        if mask is not None:
            mask = torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
        init = options.get("init_state")
        if self.noise == "numpy" and init is None:
            if seed is not None:
                for i in range(N):
                    self._rng_E[i], _ = np_random(seed + i)
            elif self._rng_E[0] is None:
                for i in range(N):
                    self._rng_E[i], _ = np_random(None)
            m = None if mask is None else mask.cpu().numpy()
            init = self._emitted.t().cpu().numpy().copy()
            for i in range(N):
                if m is None or m[i]:
                    init[i] = self._host_box_sample(self._rng_F[i])
        elif (seed is not None and self.noise == "philox"
              and not options.get("_ctor")):
            self._reseed(seed, mask, rewind=mask is None)
        if init is not None:
            init = torch.as_tensor(init, device=dev).to(self._real).reshape(
                N, D).contiguous()
        elif self.noise == "replay" and not options.get("_ctor"):
            raise ValueError("replay mode: pass options['init_state'] to reset()")
        obs = torch.empty((N, D), dtype=self._real, device=dev)
        opts = self._opts(1, _lib.MDPP_NOISE_PHILOX)
        self._check(self._lib.mdpp_continuous_reset(
            self._ctx, C.byref(self._state), _ptr(mask), _ptr(init), _ptr(obs),
            C.byref(opts), self._stream()))
        self.curr_obs = self._observe(obs, options.get("image_params"), reset=True,
                                      ctor=bool(options.get("_ctor")))
        return self.curr_obs, {}

    def _continuous_actions(self, actions):
        """Box.contains needs np.can_cast(action dtype, dtype_s): anything else
        (float64 actions for a float32 env, int32 / int64) is 'not in the
        action space' and the reference freezes the state for that step
        (:1640, :1671-1679).  strict (default): raise instead."""
        real = self._real
        if actions.dtype == real:
            return actions.contiguous()
        np_from = np.dtype(str(actions.dtype).replace("torch.", ""))
        if np.can_cast(np_from, np.dtype(self.spec.dtype_s)):
            return actions.to(real).contiguous()
        if self.strict:
            raise TypeError(f"actions must be {real}, got {actions.dtype} "
                            "(strict=False freezes the state like the reference)")
        if self.spec.action_loss_weight:
            raise NotImplementedError(
                "strict=False with action_loss_weight: the reference still "
                "charges the norm of the rejected action")
        # NaN fails every bound test in the kernel: frozen state, derivatives kept
        return torch.full(actions.shape, float("nan"), dtype=real,
                          device=actions.device)

    def _grid_actions(self, actions):
        """Non-integer grid actions: the reference applies a no-op and still
        tests the target (:1730-1733).  strict (default): raise instead."""
        if not actions.dtype.is_floating_point:
            return actions.to(torch.int64).contiguous()
        if self.strict:
            raise TypeError(f"grid actions must be integers, got {actions.dtype} "
                            "(strict=False applies a no-op like the reference)")
        noop = torch.zeros(actions.shape, dtype=torch.int64, device=actions.device)
        noop[..., 0] = 2  # out of range: the kernel's no-op that tests the target
        return noop

    def _rollout_continuous(self, n_steps, actions, replay, out, want_final_obs):
        T, N, dev = int(n_steps), self.num_envs, self.device
        D, real = self.spec.state_space_dim, self._real
        if actions is None:
            raise ValueError("continuous rollout needs an actions tensor [T,N,D]")
        actions = self._continuous_actions(torch.as_tensor(actions, device=dev))
        assert actions.shape == (T, N, D), (actions.shape, (T, N, D))
        if out is None:
            out = {
                "obs": torch.empty((T, N, D), dtype=real, device=dev),
                "reward": torch.empty((T, N), dtype=real, device=dev),
                "terminated": torch.empty((T, N), dtype=torch.bool, device=dev),
                "truncated": torch.empty((T, N), dtype=torch.bool, device=dev),
            }
            if want_final_obs:
                out["final_obs"] = torch.empty((T, N, D), dtype=real, device=dev)
        io = _lib.ContinuousIO()
        io.actions = _ptr(actions)
        io.obs, io.reward = _ptr(out.get("obs")), _ptr(out.get("reward"))
        io.final_obs = _ptr(out.get("final_obs"))
        io.terminated = _ptr(out.get("terminated"))
        io.truncated = _ptr(out.get("truncated"))
        keep = []
        if self.noise == "numpy":
            assert not self.autoreset, \
                "noise='numpy' needs explicit resets (draw order is host-driven)"
            replay = {}
            sn = np.zeros((T, N, D))
            rn = np.zeros((T, N))
            for t in range(T):
                for i in range(N):
                    if self.has_pnoise:
                        sn[t, i] = self._rng_E[i].normal(
                            0, self.spec.transition_noise, (D,))
                    if self.has_rnoise:
                        rn[t, i] = self._rng_E[i].normal(
                            0, self.spec.reward_noise_std)
            replay["state_noise"], replay["reward_noise"] = sn, rn
        if self.noise in ("replay", "numpy"):
            replay = replay or {}
            for name, field, dt, shp in (
                    ("state_noise", "replay_state_noise", torch.float64, (T, N, D)),
                    ("reward_noise", "replay_reward_noise", torch.float64, (T, N)),
                    ("reset_state", "replay_reset_state", real, (T, N, D))):
                if replay.get(name) is not None:
                    t_ = torch.as_tensor(replay[name], device=dev).to(dt).reshape(
                        shp).contiguous()
                    keep.append(t_)
                    setattr(io, field, _ptr(t_))
        opts = self._opts(T)
        if not (self.has_pnoise or self.has_rnoise) and self.noise == "philox" \
                and not self.autoreset:
            opts.noise_mode = _lib.MDPP_NOISE_OFF
        self._check(self._lib.mdpp_continuous_rollout(
            self._ctx, C.byref(self._state), C.byref(io), C.byref(opts),
            self._stream()))
        self._step_index += T
        return out


    # ------------------------------------------------------------------
    # grid backend (move_to_a_point on a 2-D grid)
    # ------------------------------------------------------------------
    def _init_grid(self):
        """rl_toy_env.py:780-812: cells are int64 rows [x, y(, x_irr, y_irr)],
        actions unit moves (GridActionSpace)."""
        sp, N, dev = self.spec, self.num_envs, self.device
        nd = len(sp.grid_shape)
        self._irr = False
        self._nd = nd
        hi = np.array(sp.grid_shape, dtype=np.int64)
        self.observation_space = BoxSpace(0 * hi, hi, (nd,), np.dtype(np.int64),
                                          seed=self.seed_dict.get("state_space"))
        self.action_space = BoxSpace(-np.ones(nd, dtype=np.int64),
                                     np.ones(nd, dtype=np.int64), (nd,),
                                     np.dtype(np.int64),
                                     seed=self.seed_dict.get("action_space"))
        specs = self._group_specs
        G = len(specs)
        self.has_pnoise = any(bool(s_.transition_noise) for s_ in specs)
        self.has_rnoise = any(s_.has_reward_noise for s_ in specs)

        def grid_cfg(s_):
            c = _lib.GridConfig()
            c.n_dims, c.dense = nd, int(s_.make_denser)
            c.reward_every_n_steps = s_.reward_every_n_steps
            c.has_transition_noise = int(bool(s_.transition_noise))
            c.has_reward_noise = int(s_.has_reward_noise)
            for k in range(nd):
                c.shape[k] = s_.grid_shape[k]
            c.target[0], c.target[1] = s_.target_point[0], s_.target_point[1]
            c.transition_noise = s_.transition_noise
            c.reward_noise_std = s_.reward_noise_std
            c.reward_scale, c.reward_shift = s_.reward_scale, s_.reward_shift
            c.term_state_reward = s_.term_state_reward
            return c
        if G > 1:
            # one launch for a whole sweep: every CTA steps its group's envs
            # under that group's scalars (csrc/grid.cu GROUPS); the groups may
            # differ in everything but the number of coordinates per cell
            if any(len(s_.grid_shape) != nd for s_ in specs):
                raise ValueError("config_groups of grid envs must agree on the "
                                 "number of grid dimensions (irrelevant_features)")
            if sp.image_representations or self.noise == "numpy":
                raise NotImplementedError(
                    "config_groups of grid envs: no images, no noise='numpy'")
            from .sharding import group_id_bases
            id_bases = group_id_bases(self._group_sizes, *self._shard)
            groups = (_lib.GridGroup * G)()
            begin = 0
            self.group_slices = []
            for gi, s_ in enumerate(specs):
                groups[gi].cfg = grid_cfg(s_)
                groups[gi].env_begin, groups[gi].env_count = begin, self._group_sizes[gi]
                groups[gi].global_id_base = id_bases[gi]
                self.group_slices.append(slice(begin, begin + self._group_sizes[gi]))
                begin += self._group_sizes[gi]
            assert begin == N
            if self._shard[1] > 1:  # (ids come from the groups, not from the offset)
                self.env_id_offset -= self._shard[0] * self.num_envs
            self._check(self._lib.mdpp_set_grid_groups(self._ctx, groups, G))
        else:
            c = grid_cfg(sp)
            self._check(self._lib.mdpp_set_grid_config(self._ctx, C.byref(c)))
        self.n_groups = G
        self._pos = torch.zeros((nd, N), dtype=torch.int32, device=dev)
        self._t = torch.zeros(N, dtype=torch.int32, device=dev)
        self._episode = torch.zeros(N, dtype=torch.int32, device=dev)
        self._reached = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._stats = torch.zeros((_lib.STATS_SLOTS, G, _lib.MDPP_N_STATS),
                                  dtype=torch.float64, device=dev)
        st = _lib.GridState()
        st.n_envs = N
        st.pos, st.t_episode = _ptr(self._pos), _ptr(self._t)
        st.episode, st.reached = _ptr(self._episode), _ptr(self._reached)
        st.stats = _ptr(self._stats)
        st.stats_slots = _lib.STATS_SLOTS
        self._prev = torch.full((2, N), -1, dtype=torch.int32, device=dev) \
            if self.track_history else None
        st.prev = _ptr(self._prev)
        self._state = st
        self._history = None
        if self.noise == "numpy":  # lane i: the reference seeded with seed + i
            def lanes(key):
                s = self.seed_dict.get(key)
                return [np_random(None if s is None else s + i)[0]
                        for i in range(N)]
            self._rng_F, self._rng_A = lanes("state_space"), lanes("action_space")
            self._rng_E = [None] * N

    def _reset_grid(self, seed, options):
        N, dev, nd = self.num_envs, self.device, self._nd
        mask = options.get("mask")
        if mask is not None:
            mask = torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
        init = options.get("init_state")
        if self.noise == "numpy" and init is None:
            if seed is not None:
                for i in range(N):
                    self._rng_E[i], _ = np_random(seed + i)
            elif self._rng_E[0] is None:
                for i in range(N):
                    self._rng_E[i], _ = np_random(None)
            m = None if mask is None else mask.cpu().numpy()
            init = self._pos.t().cpu().numpy().astype(np.int64)
            hi = np.array(self.spec.grid_shape, dtype=np.int64) + 1
            for i in range(N):
                if m is None or m[i]:  # gymnasium's int Box: floor(U(0, shape+1))
                    init[i] = np.floor(self._rng_F[i].uniform(
                        low=np.zeros(nd), high=hi, size=(nd,))).astype(np.int64)
        elif (seed is not None and self.noise == "philox"
              and not options.get("_ctor")):
            self._reseed(seed, mask, rewind=mask is None)
        if init is not None:
            init = torch.as_tensor(init, device=dev).to(torch.int64).reshape(
                N, nd).contiguous()
        elif self.noise == "replay" and not options.get("_ctor"):
            raise ValueError("replay mode: pass options['init_state'] to reset()")
        obs = torch.empty((N, nd), dtype=torch.int64, device=dev)
        opts = self._opts(1, _lib.MDPP_NOISE_PHILOX)
        self._check(self._lib.mdpp_grid_reset(
            self._ctx, C.byref(self._state), _ptr(mask), _ptr(init), _ptr(obs),
            C.byref(opts), self._stream()))
        self.curr_obs = self._observe(obs, None, reset=True,
                                      ctor=bool(options.get("_ctor")))
        return self.curr_obs, {}

    def _grid_numpy_draws(self, actions):
        """The reference's draws for one step of every lane (:1734-1750 E
        uniform + GridActionSpace samples, :1982 E normal), host side."""
        N, nd = self.num_envs, self._nd
        acts = actions.cpu().numpy().reshape(N, nd)
        rep = {"noise_u": np.ones(N), "noise_action": acts.copy(),
               "reward_noise": np.zeros(N)}
        for i in range(N):
            a = acts[i]
            valid = bool(np.all((a >= -1) & (a <= 1)) and np.abs(a).sum() <= 1)
            if valid and self.has_pnoise:
                rep["noise_u"][i] = u = self._rng_E[i].uniform()
                if u < self.spec.transition_noise:
                    while True:
                        new = np.zeros(nd, dtype=np.int64)
                        ind = self._rng_A[i].integers(nd).item()
                        new[ind] = self._rng_A[i].integers(3).item() - 1
                        if not np.array_equal(new, a):
                            rep["noise_action"][i] = new
                            break
            if self.has_rnoise:
                rep["reward_noise"][i] = self._rng_E[i].normal(
                    0, self.spec.reward_noise_std)
        return {k: v[None] for k, v in rep.items()}

    def _rollout_grid(self, n_steps, actions, replay, out, want_final_obs):
        """actions: int64 [T, N, n_dims] unit moves; returns obs / final_obs
        int64 [T, N, n_dims], reward float64 [T, N], terminated, truncated."""
        T, N, dev, nd = int(n_steps), self.num_envs, self.device, self._nd
        if actions is None:
            raise ValueError("grid rollout needs an actions tensor [T, N, n_dims]")
        actions = self._grid_actions(torch.as_tensor(actions, device=dev))
        assert actions.shape == (T, N, nd), (actions.shape, (T, N, nd))
        if out is None:
            out = {
                "obs": torch.empty((T, N, nd), dtype=torch.int64, device=dev),
                "reward": torch.empty((T, N), dtype=torch.float64, device=dev),
                "terminated": torch.empty((T, N), dtype=torch.bool, device=dev),
                "truncated": torch.empty((T, N), dtype=torch.bool, device=dev),
            }
            if want_final_obs:
                out["final_obs"] = torch.empty((T, N, nd), dtype=torch.int64,
                                               device=dev)
        io = _lib.GridIO()
        io.actions = _ptr(actions)
        io.obs, io.reward = _ptr(out.get("obs")), _ptr(out.get("reward"))
        io.final_obs = _ptr(out.get("final_obs"))
        io.terminated = _ptr(out.get("terminated"))
        io.truncated = _ptr(out.get("truncated"))
        keep = []
        if self.noise == "numpy":
            assert not self.autoreset and T == 1, \
                "noise='numpy' steps one at a time with explicit resets"
            replay = self._grid_numpy_draws(actions)
        if self.noise in ("replay", "numpy"):
            replay = replay or {}
            for name, field, dt, shp in (
                    ("noise_u", "replay_noise_u", torch.float64, (T, N)),
                    ("noise_action", "replay_noise_action", torch.int64, (T, N, nd)),
                    ("reward_noise", "replay_reward_noise", torch.float64, (T, N)),
                    ("reset_state", "replay_reset_state", torch.int64, (T, N, nd))):
                if replay.get(name) is not None:
                    t_ = torch.as_tensor(replay[name], device=dev).to(dt).reshape(
                        shp).contiguous()
                    keep.append(t_)
                    setattr(io, field, _ptr(t_))
        opts = self._opts(T)
        self._check(self._lib.mdpp_grid_rollout(
            self._ctx, C.byref(self._state), C.byref(io), C.byref(opts),
            self._stream()))
        self._step_index += T
        return out

    # ------------------------------------------------------------------
    def get_augmented_state(self):
        if self.spec.kind == "grid":
            # :2159-2164: augmented_state = [cell before the last step (NaN
            # right after a reset), current relevant cell], float64 [N, 2, 2]
            d = {"curr_state": self._pos.t().to(torch.int64).contiguous(),
                 "curr_obs": self.curr_obs}
            if self._prev is not None:
                prev = self._prev.t().to(torch.float64)
                prev = torch.where(prev < 0, torch.full_like(prev, float("nan")), prev)
                cur = self._pos[:2].t().to(torch.float64)
                d["augmented_state"] = torch.stack([prev, cur], dim=1)
            return d
        if self.spec.kind == "continuous":
            return {"curr_state": self._emitted.t().contiguous(),
                    "curr_obs": self.curr_obs,
                    "state_derivatives": self._derivs.permute(2, 0, 1).contiguous()}
        """Batched analogue of RLToyEnv.get_augmented_state (:2127):
        curr_state int64[N], curr_obs, augmented_state float64[N, L+d+1]
        (NaN where the reference has NaN)."""
        if self._history is None:
            raise RuntimeError("construct with track_history=True to use "
                               "get_augmented_state()")
        H = self._hist_depth
        idx = (self._step_index - torch.arange(H - 1, -1, -1,
                                               device=self.device)) % H
        hist = self._history[idx].to(torch.float64).t().contiguous()  # [N, H]
        age = torch.arange(H - 1, -1, -1, device=self.device)[None, :]
        hist = torch.where(age <= self._t[:, None].to(torch.int64), hist,
                           torch.full_like(hist, float("nan")))
        cur = self._cur.to(torch.int64)
        if self._irr:  # (relevant, irrelevant); the window holds relevant states
            cur = torch.stack([cur, self._cur_irr.to(torch.int64)], dim=-1)
        return {"curr_state": cur,
                "curr_obs": self.curr_obs, "augmented_state": hist}

    def set_augmented_state(self, state):
        """Batched analogue of RLToyEnv.set_augmented_state (:2168): accepts
        the dict returned by get_augmented_state() or a bare state tensor
        ([N] discrete, [N, D] continuous; then the window holds only that state
        and continuous derivatives are zeroed).  Like the reference it does not
        touch the reward-delay FIFO or the RNG streams."""
        dev, N = self.device, self.num_envs
        if self.spec.kind == "grid":
            # the dict of get_augmented_state() or a bare [N, n_dims] cell
            # tensor (then the window holds only that cell, :2203-2208)
            cells = torch.as_tensor(state["curr_state"] if isinstance(state, dict)
                                    else state, device=dev).reshape(N, self._nd)
            self._pos.copy_(cells.t().to(torch.int32))
            if self._prev is not None:
                prev = torch.full((N, 2), float("nan"), dtype=torch.float64, device=dev)
                if isinstance(state, dict) and "augmented_state" in state:
                    prev = torch.as_tensor(state["augmented_state"], device=dev).to(
                        torch.float64).reshape(N, 2, 2)[:, 0]
                self._prev.copy_(torch.nan_to_num(prev, nan=-1.0).t().to(torch.int32))
            self.curr_obs = self._observe(cells.to(torch.int64), reset=True, ctor=True)
            return
        if self.spec.kind == "continuous":
            D, order = self.spec.state_space_dim, self._max_order
            if isinstance(state, dict):
                cur = torch.as_tensor(state["curr_state"], device=dev).to(self._real)
                sd = torch.as_tensor(state["state_derivatives"], device=dev).to(
                    self._real).reshape(N, order + 1, D)
            else:
                cur = torch.as_tensor(state, device=dev).to(self._real)
                sd = torch.zeros((N, order + 1, D), dtype=self._real, device=dev)
                sd[:, 0] = cur.reshape(N, D)
            self._emitted.copy_(cur.reshape(N, D).t())
            self._derivs.copy_(sd.permute(1, 2, 0))
            self.curr_obs = self._observe(cur.reshape(N, D), reset=True, ctor=True)
            return
        if self._history is None:
            raise RuntimeError("construct with track_history=True to use "
                               "set_augmented_state()")
        H, L = self._hist_depth, self.spec.sequence_length
        if self._irr:
            full = torch.as_tensor(state["curr_state"] if isinstance(state, dict)
                                   else state, device=dev).reshape(N, 2)
            self._check_column(full[:, 1:], irr=True, what="irrelevant state")
            if not isinstance(state, dict):
                state = full[:, 0]
        if isinstance(state, dict):
            aug = torch.as_tensor(state["augmented_state"], device=dev).to(
                torch.float64).reshape(N, H)
        else:
            aug = torch.full((N, H), float("nan"), dtype=torch.float64, device=dev)
            aug[:, -1] = torch.as_tensor(state, device=dev).to(torch.float64)
        valid = ~torch.isnan(aug)
        n_valid = valid.to(torch.int32).sum(dim=1)          # trailing entries
        states = torch.nan_to_num(aug, nan=0.0).to(torch.int64)
        self._check_column(states, irr=False, what="augmented_state entry")
        if self._irr:  # (only once both columns have passed the checks)
            self._cur_irr.copy_(full[:, 1].to(torch.int32))
        self._cur.copy_(states[:, -1].to(torch.int32))
        bits = max(1, int(np.ceil(np.log2(max(self.tables.n_states, 2)))))
        key = torch.zeros(N, dtype=torch.int64, device=dev)
        for j in range(L):  # oldest of the last L first, newest lowest
            key = (key << bits) | states[:, H - L + j]
        mask = (1 << (bits * L)) - 1
        self._key.copy_(key & mask)
        # t such that the kernel's NaN gate (t >= L) sees the same window; a
        # full window keeps the current count when it is already large enough
        t_new = (n_valid - 1).clamp(min=0)
        keep = (n_valid == H) & (self._t >= H - 1)
        self._t.copy_(torch.where(keep, self._t, t_new))
        idx = (self._step_index - torch.arange(H - 1, -1, -1, device=dev)) % H
        self._history[idx] = states.t().to(torch.int32)
        cur = self._cur.to(torch.int64)
        if self._irr:
            cur = torch.stack([cur, self._cur_irr.to(torch.int64)], dim=-1)
        self.curr_obs = self._observe(cur, reset=True, ctor=True)

    def seed(self, seed=None):
        """RLToyEnv.seed (:2379): re-keys the environment's noise stream."""
        if self.noise == "numpy":
            for i in range(self.num_envs):
                self._rng_E[i], _ = np_random(None if seed is None else seed + i)
        elif seed is not None:
            self._reseed(seed)
        return seed

    def episode_stats(self, reduce=False):
        """Per-group counters of rl_toy_env.py:2360-2369 summed over envs and
        episodes; `reduce=True` all-reduces over torch.distributed ranks."""
        from . import sharding
        total = self._stats.sum(dim=0)  # the kernels spread atomics over slots
        stats = sharding.reduce_stats(total) if reduce else total
        return sharding.summarize_stats(stats)
