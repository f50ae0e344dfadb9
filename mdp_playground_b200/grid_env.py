"""GridEnv: the grid state spaces of VectorRLToyEnv (move_to_a_point on a
2-D grid, rl_toy_env.py:780-812): cells are int64 rows [x, y(, x_irr,
y_irr)], actions unit moves (GridActionSpace)."""
import numpy as np
import torch

from . import _lib
from ._lib import _ptr
from .spaces import BoxSpace
from .vector_env import VectorRLToyEnv


class GridEnv(VectorRLToyEnv):
    _STATE_TENSORS = ("_t", "_episode", "_stats", "_reached", "_pos", "_prev")
    _IO = _lib.GridIO
    _state_dtype = torch.int64

    def _init_kind(self):
        sp, N, dev = self.spec, self.num_envs, self.device
        nd = len(sp.grid_shape)
        self._nd = nd
        self._row = (nd,)
        self._adt = torch.int64
        hi = np.array(sp.grid_shape, dtype=np.int64)
        self.observation_space = BoxSpace(0 * hi, hi, (nd,), np.dtype(np.int64),
                                          seed=self.seed_dict.get("state_space"))
        self.action_space = BoxSpace(-np.ones(nd, dtype=np.int64),
                                     np.ones(nd, dtype=np.int64), (nd,),
                                     np.dtype(np.int64),
                                     seed=self.seed_dict.get("action_space"))
        specs = self._group_specs

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
        if len(specs) > 1:
            # one launch for a whole sweep: every CTA steps its group's envs
            # under that group's scalars (csrc/grid.cu GROUPS); the groups may
            # differ in everything but the number of coordinates per cell
            if any(len(s_.grid_shape) != nd for s_ in specs):
                raise ValueError("config_groups of grid envs must agree on the "
                                 "number of grid dimensions (irrelevant_features)")
            if self.noise == "numpy":
                raise NotImplementedError(
                    "config_groups of grid envs: no noise='numpy'")
        self._set_configs([grid_cfg(s_) for s_ in specs], _lib.GridGroup,
                          self._lib.mdpp_set_grid_groups,
                          self._lib.mdpp_set_grid_config)
        self._pos = torch.zeros((nd, N), dtype=torch.int32, device=dev)
        self._reached = torch.zeros(N, dtype=torch.uint8, device=dev)
        st = self._new_state(_lib.GridState)
        st.pos, st.reached = _ptr(self._pos), _ptr(self._reached)
        self._prev = torch.full((2, N), -1, dtype=torch.int32, device=dev) \
            if self.track_history else None
        st.prev = _ptr(self._prev)
        self._state = st
        self._rollout_fn = self._lib.mdpp_grid_rollout
        self._reset_fn = self._lib.mdpp_grid_reset
        self._replay_fields = (
            ("noise_u", "replay_noise_u", torch.float64, ()),
            ("noise_action", "replay_noise_action", torch.int64, (nd,)),
            ("reward_noise", "replay_reward_noise", torch.float64, ()),
            ("reset_state", "replay_reset_state", torch.int64, (nd,)))
        if self.noise == "numpy":
            self._rng_F = self._numpy_lanes(self.seed_dict.get("state_space"))
            self._rng_A = self._numpy_lanes(self.seed_dict.get("action_space"))

    def _numpy_reset_draws(self, mask):
        nd = self._nd
        init = self._pos.t().cpu().numpy().astype(np.int64)
        hi = np.array(self.spec.grid_shape, dtype=np.int64) + 1
        for i in range(self.num_envs):
            if mask is None or mask[i]:  # gymnasium's int Box: floor(U(0, shape+1))
                init[i] = np.floor(self._rng_F[i].uniform(
                    low=np.zeros(nd), high=hi, size=(nd,))).astype(np.int64)
        return init

    def _coerce_actions(self, actions):
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

    def _draw_numpy(self, T, actions):
        """The reference's draws for one step of every lane (:1734-1750 E
        uniform + GridActionSpace samples, :1982 E normal), host side."""
        assert not self.autoreset and T == 1, \
            "noise='numpy' steps one at a time with explicit resets"
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

    # ------------------------------------------------------------------
    def _init_images(self):
        """One renderer configuration per config group (its own grid lines,
        target and terminal cells)."""
        self._set_image_groups([self._grid_image_cfg(s_) for s_ in self._group_specs])

    def _grid_image_cfg(self, sp):
        # ImageContinuous with grid_shape (image_continuous.py:139-207):
        # white grid lines, black terminal cells, green target and blue
        # agent discs at the cell centres (+0.5), per sub-grid
        W, H = sp.image_width, sp.image_height
        nd, gs = self._nd, sp.grid_shape
        if W > 256 or H > 256:
            raise NotImplementedError("grid images: width, height <= 256")
        cells = sp.terminal_cells or []
        if len(cells) > _lib.MDPP_MAX_TERM_BOXES:
            raise NotImplementedError("at most 8 terminal cells in images")
        corners = [np.array(cell, dtype=np.float64).astype(np.int64) for cell in cells]
        # (image_continuous.py:248-277 over Box(0, shape))
        c = self._box_image_cfg(sp, nd, np.zeros(2, dtype=np.int64),
                                np.array(gs[:2], dtype=np.int64),
                                [(lo_, lo_ + 1.0) for lo_ in corners],
                                np.array(sp.target_point, dtype=float) + 0.5, True)
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
        return c

    def _render_states(self, state):
        return (state.to(torch.float64) + 0.5).contiguous()  # cell centres

    # ------------------------------------------------------------------
    def get_augmented_state(self):
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

    def set_augmented_state(self, state):
        """The dict of get_augmented_state() or a bare [N, n_dims] cell
        tensor (then the window holds only that cell, :2203-2208)."""
        dev, N = self.device, self.num_envs
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
