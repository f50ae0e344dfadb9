"""ContinuousEnv: the continuous state spaces of VectorRLToyEnv
(move_to_a_point and move_along_a_line): real [N, D] states driven by
dynamics of order 1-4, with terminal hypercubes."""
import numpy as np
import torch

from . import _lib
from ._lib import _ptr
from .spaces import BoxSpace
from .vector_env import VectorRLToyEnv


class ContinuousEnv(VectorRLToyEnv):
    _STATE_TENSORS = ("_t", "_episode", "_ring", "_stats", "_derivs", "_emitted",
                      "_reached", "_hist_line")
    _IO = _lib.ContinuousIO

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

    def _init_kind(self):
        sp = self.spec
        D, N, dev = sp.state_space_dim, self.num_envs, self.device
        if D > _lib.MDPP_MAX_DIM or sp.dynamics_order > _lib.MDPP_MAX_ORDER:
            raise NotImplementedError("state_space_dim <= 16 and order <= 4")
        np_dt = np.dtype(sp.dtype_s)
        if np_dt not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise NotImplementedError("continuous dtype_s must be float32/64")
        self._real = real = torch.float64 if np_dt == np.float64 else torch.float32
        self._np_real = np_dt.type
        self._row = (D,)
        self._adt = self._state_dtype = self._reward_dtype = real
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
        self._group_terms = [(lo, hi) for _, lo, hi in cfgs]  # (the images')
        line = sp.reward_function == "move_along_a_line"
        # (the key's presence, not its value, turns transition noise on here)
        self.has_pnoise = any(s_.has_transition_noise for s_ in specs)
        max_delay = max(s_.delay for s_ in specs)

        def ring64(cc):
            return bool(self._real == torch.float32 and (
                (cc.target_is_f64 and cc.dense) or line))
        if G > 1:
            if self.noise == "numpy":
                raise NotImplementedError(
                    "config_groups of continuous envs: no noise='numpy'")
            if len({ring64(cc) for cc, _, _ in cfgs}) != 1 or (
                    line and len({s_.sequence_length for s_ in specs}) != 1):
                raise ValueError(
                    "config_groups of continuous envs must agree on make_denser / "
                    "default target_point (the reward FIFO's dtype) and, for "
                    "move_along_a_line, on sequence_length")
        self._set_configs([cc for cc, _, _ in cfgs], _lib.ContinuousGroup,
                          self._lib.mdpp_set_continuous_groups,
                          self._lib.mdpp_set_continuous_config)
        self._max_order = max(s_.dynamics_order for s_ in specs)
        self._derivs = torch.zeros((self._max_order + 1, D, N), dtype=real,
                                   device=dev)
        self._emitted = torch.zeros((D, N), dtype=real, device=dev)
        self._reached = torch.zeros(N, dtype=torch.uint8, device=dev)
        # (fp32 env + default float64 target_point + dense reward: the reward is
        # a python float all the way through the reference's reward_buffer)
        ring_dt = torch.float64 if ring64(c) else real
        # move_along_a_line: the last sequence_length emitted relevant states
        self._hist_line = torch.zeros((sp.sequence_length, c.n_relevant, N),
                                      dtype=real, device=dev) if line else None
        self._ring = torch.zeros((max_delay, N), dtype=ring_dt, device=dev) \
            if max_delay > 0 else None
        st = self._new_state(_lib.ContinuousState)
        st.derivs, st.emitted = _ptr(self._derivs), _ptr(self._emitted)
        st.reached, st.ring = _ptr(self._reached), _ptr(self._ring)
        st.hist = _ptr(self._hist_line)
        self._state = st
        self._rollout_fn = self._lib.mdpp_continuous_rollout
        self._reset_fn = self._lib.mdpp_continuous_reset
        self._replay_fields = (
            ("state_noise", "replay_state_noise", torch.float64, (D,)),
            ("reward_noise", "replay_reward_noise", torch.float64, ()),
            ("reset_state", "replay_reset_state", real, (D,)))
        if not (self.has_pnoise or self.has_rnoise) and self.noise == "philox" \
                and not self.autoreset:
            self._noise_mode = _lib.MDPP_NOISE_OFF
        if self.noise == "numpy":
            self._rng_F = self._numpy_lanes(self.seed_dict.get("state_space"))

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

    def _numpy_reset_draws(self, mask):
        init = self._emitted.t().cpu().numpy().copy()
        for i in range(self.num_envs):
            if mask is None or mask[i]:
                init[i] = self._host_box_sample(self._rng_F[i])
        return init

    def _coerce_actions(self, actions):
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

    def _draw_numpy(self, T, actions):
        assert not self.autoreset, \
            "noise='numpy' needs explicit resets (draw order is host-driven)"
        N, D = self.num_envs, self.spec.state_space_dim
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
        return {"state_noise": sn, "reward_noise": rn}

    # ------------------------------------------------------------------
    def _init_images(self):
        """One renderer configuration per config group: its own target,
        terminal regions and feature bounds (state_space_max)."""
        D = self.spec.state_space_dim
        if D not in (2, 4):
            raise NotImplementedError(
                "continuous image observations: 2 relevant (+ 0 or 2 "
                "irrelevant) dimensions")
        dt = self._np_real
        cfgs = []
        for s_, (lows, highs) in zip(self._group_specs, self._group_terms):
            assert np.isfinite(s_.state_space_max), \
                "image observations need a bounded state space"
            cfgs.append(self._box_image_cfg(
                s_, D, np.full((2,), -s_.state_space_max).astype(dt),
                np.full((2,), s_.state_space_max).astype(dt),
                list(zip(lows, highs)),
                np.asarray(s_.target_point, dtype=dt), self._real == torch.float64))
        self._set_image_groups(cfgs)

    def _render_states(self, state):
        return state.to(self._real).contiguous()

    # ------------------------------------------------------------------
    def get_augmented_state(self):
        return {"curr_state": self._emitted.t().contiguous(),
                "curr_obs": self.curr_obs,
                "state_derivatives": self._derivs.permute(2, 0, 1).contiguous()}

    def set_augmented_state(self, state):
        """Batched analogue of RLToyEnv.set_augmented_state (:2168): accepts
        the dict returned by get_augmented_state() or a bare state tensor
        [N, D] (then the derivatives are zeroed).  Like the reference it does
        not touch the reward-delay FIFO or the RNG streams."""
        dev, N = self.device, self.num_envs
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
