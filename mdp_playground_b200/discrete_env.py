"""DiscreteEnv: the discrete state spaces of VectorRLToyEnv.

States index per-group host-built tables (tables.py); every launch runs the
envs as config groups, laid out group-major.  With irrelevant_features a
second, reward-free sub-MDP rides along: states, actions and observations
become rows (relevant, irrelevant), the reference's tuples
(rl_toy_env.py:2085-2088).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import _ptr
from .spaces import DiscreteSpace
from .tables import build_discrete_tables
from .vector_env import VectorRLToyEnv


def _host_ptrs(arrays):
    return [None if a is None else a.ctypes.data_as(C.c_void_p) for a in arrays]


class DiscreteEnv(VectorRLToyEnv):
    _FP64_NORMAL = _lib.MDPP_NORMAL_ZIGGURAT
    _STATE_TENSORS = ("_cur", "_cur_irr", "_key", "_t", "_episode", "_ring",
                      "_history", "_stats")
    _IO = _lib.DiscreteIO
    _random_policy = True
    _renders_in_step = True
    _REPLAY_RESET = "options['reset_u'] or options['init_state']"
    _state_dtype = torch.int64
    _replay_fields = tuple((name, "replay_" + name, torch.float64, ())
                           for name in ("transition_u", "reward_noise", "reset_u"))
    _OBS_CODES = {torch.int64: _lib.MDPP_OBS_I64, torch.int32: _lib.MDPP_OBS_I32,
                  torch.uint8: _lib.MDPP_OBS_U8}

    def _init_kind(self):
        """One configuration group per entry of self._group_specs (a single
        one for the plain drop-in use)."""
        sp = self.spec
        N, dev = self.num_envs, self.device
        specs = self._group_specs
        G = len(specs)
        self.group_tables = [build_discrete_tables(s_) for s_ in specs]
        self.tables = tb = self.group_tables[0]
        self.transition_matrix = tb.transition
        self.rewardable_sequences = tb.rewardable_sequences
        self.reward_matrix = tb.reward_matrix
        self.observation_space = DiscreteSpace(
            tb.n_states, seed=self.seed_dict.get("relevant_state_space"))
        self.action_space = DiscreteSpace(
            tb.n_actions, seed=self.seed_dict.get("relevant_action_space"))
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
        self._row = (2,) if self._irr else ()
        self._adt = torch.int32
        self._obs_dtype_override = None  # set_obs_dtype()
        self._io_cache = None            # rollout()'s last marshalled launch
        groups = self._group_array(_lib.DiscreteGroup)
        self._host_keep = []
        for g, s_, t_ in zip(groups, specs, self.group_tables):
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
            (g.transition, g.terminal, g.init_cdf, g.noise_cdf, g.sequences,
             g.sequence_rewards, g.reward_matrix) = _host_ptrs(keep)
            if t_.n_states_irr:
                g.n_states_irr, g.n_actions_irr = t_.n_states_irr, t_.n_actions_irr
                keep_irr = [t_.transition_irr, t_.init_cdf_irr, t_.noise_cdf_irr]
                keep.extend(keep_irr)
                (g.transition_irr, g.init_cdf_irr,
                 g.noise_cdf_irr) = _host_ptrs(keep_irr)
        self._check(self._lib.mdpp_set_discrete_groups(self._ctx, groups, G))
        max_delay = max(s_.delay for s_ in specs)

        self._cur = torch.zeros(N, dtype=torch.int32, device=dev)
        self._cur_irr = torch.zeros(N, dtype=torch.int32, device=dev) \
            if self._irr else None
        self._key = torch.zeros(N, dtype=torch.int64, device=dev)
        self._ring = torch.zeros((max_delay, N), dtype=torch.float64,
                                 device=dev) if max_delay > 0 else None
        self._hist_depth = sp.sequence_length + sp.delay + 1
        if G > 1:
            self.track_history = False  # augmented_state differs per group
        self._history = torch.zeros((self._hist_depth, N), dtype=torch.int32,
                                    device=dev) if self.track_history else None
        st = self._new_state(_lib.DiscreteState)
        st.cur_state, st.seq_key = _ptr(self._cur), _ptr(self._key)
        st.ring = _ptr(self._ring)
        st.ring_depth = max_delay
        st.history_depth = self._hist_depth
        st.history = _ptr(self._history)
        st.cur_state_irr = _ptr(self._cur_irr)
        self._state = st
        self._rollout_fn = self._lib.mdpp_discrete_rollout
        self._reset_fn = self._lib.mdpp_discrete_reset
        if self.noise == "numpy":
            assert G == 1, "noise='numpy' is a single-configuration mode"
            self._init_numpy_streams()

    def _init_numpy_streams(self):
        """Per-lane PCG64 streams; lane 0 = the reference's own (appendix C):
        S continues after the P-table draws, E is re-seeded at the first reset."""
        sd = self.seed_dict
        from .tables import _next_set_probabilities, sub_space_rngs
        rng0, rng1 = sub_space_rngs(self.spec)
        self._rng_S = [rng0] + self._numpy_lanes(sd.get("relevant_state_space"), 1)
        if self._irr:
            self._rng_S1 = [rng1] + self._numpy_lanes(
                sd.get("irrelevant_state_space"), 1)
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

    # ------------------------------------------------------------------
    def _init_states(self, init):
        init = torch.as_tensor(init, device=self.device).to(torch.int32).contiguous()
        self._check_state_range(init)
        return init

    def _numpy_reset_draws(self, mask):
        N = self.num_envs
        reset_u = np.zeros((N, 2) if self._irr else N)
        for i in range(N):
            if mask is None or mask[i]:  # one E draw per sub-space (:2255-2264)
                reset_u[i] = [self._rng_E[i].random() for _ in range(2)] \
                    if self._irr else self._rng_E[i].random()
        return reset_u

    def _reset_inputs(self, init, draws, options):
        reset_u = options.get("reset_u") if draws is None else draws
        if reset_u is not None:
            reset_u = torch.as_tensor(reset_u, dtype=torch.float64,
                                      device=self.device).contiguous()
        row = (self.num_envs,) + self._row
        if init is not None:
            assert tuple(init.shape) == row, (tuple(init.shape), row)
        if reset_u is not None:
            assert tuple(reset_u.shape) == row, (tuple(reset_u.shape), row)
        mode = _lib.MDPP_NOISE_REPLAY if reset_u is not None \
            else _lib.MDPP_NOISE_PHILOX
        return mode, (init, reset_u)

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

    # ------------------------------------------------------------------
    # observation dtype
    # ------------------------------------------------------------------
    def _obs_torch_dtype(self):
        """dtype the discrete kernels write observations in: the config's
        dtype_o (rl_toy_env.py:571, :611-614) when it is int64 / int32 / uint8
        (written in-kernel), else int64 followed by a cast."""
        forced = self._obs_dtype_override
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
        target = self._obs_dtype_override or getattr(
            torch, np.dtype(self.spec.dtype_o).name)
        return obs if obs.dtype == target else obs.to(target)

    # ------------------------------------------------------------------
    # stepping
    # ------------------------------------------------------------------
    def _coerce_actions(self, actions):
        return actions.to(torch.int32).contiguous()

    def _io(self, actions, out):
        # the kernels write observations in the dtype of the caller's buffer
        odt = out["obs"].dtype if out.get("obs") is not None else torch.int64
        if odt not in self._OBS_CODES or (
                out.get("final_obs") is not None and out["final_obs"].dtype != odt):
            raise TypeError("obs / final_obs buffers must both be int64, int32 or uint8")
        io = super()._io(actions, out)
        io.obs_dtype = self._OBS_CODES[odt]
        return io

    def _replay_tensor(self, replay, name, dtype, shape):
        t = torch.as_tensor(replay[name], dtype=dtype, device=self.device).reshape(shape)
        if self._irr and name != "reward_noise":
            # the irrelevant sub-space's draw rides in the same row
            t1 = replay.get("irr_" + name)
            t1 = torch.zeros_like(t) if t1 is None else torch.as_tensor(
                t1, dtype=dtype, device=self.device).reshape(shape)
            t = torch.stack([t, t1], dim=-1)
        return t.contiguous()

    def _draw_numpy(self, T, actions):
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

    def _step_render(self, state):
        if not self.spec.image_representations:
            return state, None
        # the renderer runs as a programmatic dependent of the step kernel
        # (its zero fill overlaps it), marshalled once as well
        dev = self.device
        M = state.numel()
        img = torch.empty(tuple(state.shape[:1]) + self.obs_shape,
                          dtype=torch.uint8, device=dev)
        prm = torch.empty((M, 5), dtype=torch.int32, device=dev)
        ropts = self._opts(1)
        ropts.flags = _lib.MDPP_LAUNCH_OVERLAP_PREVIOUS
        args = self._render_tables() + (_ptr(state), None, _ptr(prm), _ptr(img),
                                        M, self.num_envs, 3, C.byref(ropts))
        return img, (self._render_fn(), ropts, args, prm)

    def rollout(self, n_steps, actions=None, replay=None, out=None,
                want_final_obs=True):
        T = int(n_steps)
        # step()-granularity callers repeat the same launch (same action and
        # output buffers): reuse the marshalled I/O struct -- the Python side is
        # what bounds a T = 1 call (a 5 us kernel)
        fast_key = None
        if (out is not None and self.noise == "philox" and torch.is_tensor(actions)
                and actions.dtype == torch.int32 and actions.is_cuda
                and actions.is_contiguous()):
            fast_key = (T, actions.data_ptr(), tuple(actions.shape)) + tuple(
                (k, v.data_ptr(), v.dtype) for k, v in out.items())
            hit = self._io_cache
            if hit is not None and hit[0] == fast_key:
                opts = self._opts(T)
                self._check(self._lib.mdpp_discrete_rollout(
                    self._ctx, C.byref(self._state), C.byref(hit[1]),
                    C.byref(opts), self._stream()))
                self._step_index += T
                return out
        io, actions, out = self._launch_rollout(T, actions, replay, out, want_final_obs)
        if fast_key is not None:  # (holds the tensors, so the pointers stay valid)
            self._io_cache = (fast_key, io, actions, dict(out))
        return out

    # ------------------------------------------------------------------
    # image observations
    # ------------------------------------------------------------------
    @staticmethod
    def _image_key(sp):
        """What a discrete renderer table set depends on besides the state
        count: the transforms and their parameters."""
        tr = sp.image_transforms
        flags = tuple(t in tr for t in ("scale", "shift", "rotate", "flip"))
        return flags + (int(sp.image_sh_quant or 1), int(sp.image_ro_quant or 1),
                        tuple(sp.image_scale_range) if flags[0] else None)

    def _init_images(self):
        """Renderer tables: one set per distinct image configuration of the
        config groups (a sweep whose cells do not vary the images builds one),
        for the largest state count of the groups that share it."""
        from . import image_tables as it
        sp, dev = self.spec, self.device
        W, H = sp.image_width, sp.image_height
        self._img_keep = []

        def up(a, dtype):
            t = torch.as_tensor(np.ascontiguousarray(a)).to(dtype).to(dev).contiguous()
            self._img_keep.append(t)
            return _ptr(t)
        keys = [self._image_key(s_) for s_ in self._group_specs]
        n_states = {}
        for k, t_ in zip(keys, self.group_tables):
            n_states[k] = max(n_states.get(k, 0), t_.n_states, t_.n_states_irr or 0)
        # irrelevant_features: one polygon image per sub-state, stacked
        # along x (image_multi_discrete.py:272-288)
        self._n_sub = 2 if self._irr else 1
        self.image_table_sets = {}  # image key -> (host tables, struct)
        for k, s_ in zip(keys, self._group_specs):
            if k in self.image_table_sets:
                continue
            tb = it.build_discrete_image_tables(
                n_states[k], W, H, s_.image_transforms,
                s_.image_sh_quant, s_.image_ro_quant, s_.image_scale_range)
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
            c.n_sub_images = self._n_sub
            self.image_table_sets[k] = (tb, c)
        self.image_tables, self._img_cfg = self.image_table_sets[keys[0]]
        # (replay mode needs image_params when any group draws transforms)
        self._img_random = any(tb.has_scale or tb.has_shift or tb.has_rotate
                               or tb.has_flip
                               for tb, _ in self.image_table_sets.values())
        if self.n_groups > 1:
            groups = self._group_array(_lib.ImageDiscreteGroup)
            for g, k in zip(groups, keys):
                g.tb = self.image_table_sets[k][1]
            self._check(self._lib.mdpp_set_image_discrete_groups(
                self._ctx, groups, self.n_groups))
        self.obs_shape = (W * self._n_sub, H, 1)
        if self.noise == "numpy":
            self._rng_I = self._numpy_lanes(self.seed_dict.get("image_representations"))

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
        """State tensor -> uint8 image observations on the GPU:
        int64 [..., N] -> [..., N, W, H, 1] ([..., N, 2] rows -> 2W-wide
        images with irrelevant_features)."""
        dev, N = self.device, self.num_envs
        opts = self._opts(1)
        if self._use_dev_counter:  # observation after the step: index + 1 = the device counter
            opts.step_index = 0
        elif step_index is not None:
            opts.step_index = step_index
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
        elif self.noise == "replay" and not allow_philox and self._img_random:
            raise ValueError("replay mode: pass image_params [N, 5]")
        out = torch.empty(lead + self.obs_shape, dtype=torch.uint8, device=dev)
        self.last_image_params = torch.empty((M, 5), dtype=torch.int32,
                                             device=dev)
        if self._overlap_render and st.data_ptr() == state.data_ptr():
            # (no cast / copy kernel sits between the step and this launch)
            opts.flags = _lib.MDPP_LAUNCH_OVERLAP_PREVIOUS
        self._check(self._render_fn()(
            self._ctx, *self._render_tables(), _ptr(st), _ptr(image_params),
            _ptr(self.last_image_params), _ptr(out), M, N,
            6 if reset else 3, C.byref(opts), self._stream()))
        return out

    def _render_fn(self):
        """The renderer entry point: one table set, or each group's own."""
        return self._lib.mdpp_render_discrete_groups if self.n_groups > 1 \
            else self._lib.mdpp_render_discrete

    def _render_tables(self):
        """The entry point's table argument (none for the grouped one: the
        context holds the groups' tables)."""
        return () if self.n_groups > 1 else (C.byref(self._img_cfg),)

    # ------------------------------------------------------------------
    def get_augmented_state(self):
        """Batched analogue of RLToyEnv.get_augmented_state (:2127):
        curr_state int64[N], curr_obs, augmented_state float64[N, L+d+1]
        (NaN where the reference has NaN)."""
        if self._history is None:
            raise RuntimeError("construct with track_history=True to use "
                               "get_augmented_state()")
        H = self._hist_depth
        hist = self._history[self._history_rows()].to(
            torch.float64).t().contiguous()  # [N, H]
        age = torch.arange(H - 1, -1, -1, device=self.device)[None, :]
        hist = torch.where(age <= self._t[:, None].to(torch.int64), hist,
                           torch.full_like(hist, float("nan")))
        return {"curr_state": self._cur_state(),
                "curr_obs": self.curr_obs, "augmented_state": hist}

    def _history_rows(self):
        """Rows of the history ring holding the window, oldest first."""
        H = self._hist_depth
        return (self._step_index - torch.arange(H - 1, -1, -1, device=self.device)) % H

    def _cur_state(self):
        cur = self._cur.to(torch.int64)
        if self._irr:  # (relevant, irrelevant); the window holds relevant states
            cur = torch.stack([cur, self._cur_irr.to(torch.int64)], dim=-1)
        return cur

    def set_augmented_state(self, state):
        """Batched analogue of RLToyEnv.set_augmented_state (:2168): accepts
        the dict returned by get_augmented_state() or a bare state tensor [N]
        (then the window holds only that state).  Like the reference it does
        not touch the reward-delay FIFO or the RNG streams."""
        dev, N = self.device, self.num_envs
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
        self._history[self._history_rows()] = states.t().to(torch.int32)
        self.curr_obs = self._observe(self._cur_state(), reset=True, ctor=True)
