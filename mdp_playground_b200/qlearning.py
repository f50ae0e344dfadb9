"""Tabular Q-learning inside the discrete and grid rollout kernels.

`TabularQLearner(env)` gives every env of a discrete VectorRLToyEnv its own
Q-table, float64 [N, S_max, A_max] on the device, and trains all of them in
one fused launch per `learn(T)` call (mdpp_discrete_qlearn,
include/mdpp_b200.h): epsilon-greedy action selection, the env step and the
one-step Q-learning update, T steps per launch.  `GridQLearner(env)` does the
same for a grid env (mdpp_grid_qlearn).  Each env is one independent
training run (one seed); in a grouped env each config group is one cell of an
experiment grid.

Discrete envs explore with the random policy's own draw (`rollout(actions=
None)` at the same global step), so with epsilon = 1 `learn` takes exactly
the actions a random rollout would take.  Grid envs explore with a stream of
their own; a grid state is the cell's row-major index over [0, shape_k] (the
cell one past the grid that reset draws included), an action the index of a
GridActionSpace member (grid_action_rows).  The env's step counter advances
by T, like rollout(), so later rollout / step / reseed calls behave as they
would after a rollout of T steps.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import _ptr


def grid_action_rows(nd):
    """The kernel's grid action indices as rows: 0 = no-op, 1 + 2k = -1 on
    dim k, 2 + 2k = +1 on dim k.  int64 [2 nd + 1, nd]."""
    rows = np.zeros((2 * nd + 1, nd), dtype=np.int64)
    for k in range(nd):
        rows[1 + 2 * k, k], rows[2 + 2 * k, k] = -1, 1
    return rows


def grid_cells(shape):
    """Q-table rows of a grid: prod_k (shape_k + 1)."""
    return int(np.prod([int(n) + 1 for n in shape]))


def _unit(name, x):
    x = float(x)
    if not 0.0 <= x <= 1.0:
        raise ValueError(f"{name} must lie in [0, 1], got {x}")
    return x


class EpisodeReturns:
    """The base of the learners that run inside a rollout kernel
    (TabularQLearner, GridQLearner, ars.LinearARS): the checks they share,
    the per-env return bookkeeping (ep_return, the running episode's;
    ret_sum / ret_count, the episodes that ended in an auto-reset; all [N]
    on the device next to self.env) and the launch of a learn call."""

    def __init__(self, env):
        if env.noise != "philox":
            raise ValueError(f"{type(self).__name__} needs noise='philox' "
                             f"(got {env.noise!r})")
        if any(s_.image_representations for s_ in env._group_specs):
            raise ValueError(f"{type(self).__name__} does not support "
                             "image_representations")
        self.env = env
        N, dev = env.num_envs, env.device
        self.ep_return = torch.zeros(N, dtype=torch.float64, device=dev)
        self.ret_sum = torch.zeros(N, dtype=torch.float64, device=dev)
        self.ret_count = torch.zeros(N, dtype=torch.int32, device=dev)

    def _new_params(self, struct):
        """A new parameter struct (_lib.QlearnParams / ArsParams) pointing
        at the return counters."""
        p = struct()
        p.ep_return, p.ret_sum = _ptr(self.ep_return), _ptr(self.ret_sum)
        p.ret_count = _ptr(self.ret_count)
        return p

    def _learn(self, entry, params, T, record, action_shape, action_dtype):
        """One launch of the learner's entry point over T steps; with record,
        the outputs and the actions taken ([T, N, *action_shape])."""
        env = self.env
        out = {}
        if record:
            out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
            out["actions"] = torch.empty((T, env.num_envs) + action_shape,
                                         dtype=action_dtype, device=env.device)
            params.actions_taken = _ptr(out["actions"])
        io = env._io(None, out)
        opts = env._opts(T, noise_mode=_lib.MDPP_NOISE_PHILOX)
        env._check(entry(env._ctx, C.byref(env._state), C.byref(io), C.byref(params),
                         C.byref(opts), env._stream()))
        env._step_index += T
        return out if record else None

    # -- evaluation -------------------------------------------------------------
    def _check_eval_env(self, eval_env):
        """ValueError unless eval_env has the training env's layout: class,
        env count, group sizes and the learner's per-group shapes
        (_check_eval_layout), Philox noise, no images, autoreset and a
        horizon (which bounds every episode, so E * horizon steps complete
        E episodes)."""
        env, name = self.env, type(self).__name__
        if type(eval_env) is not type(env):
            raise ValueError(f"{name}.evaluate: eval_env is a {type(eval_env).__name__}, "
                             f"the learner's env a {type(env).__name__}")
        if eval_env.num_envs != env.num_envs or \
                list(eval_env._group_sizes) != list(env._group_sizes):
            raise ValueError(f"{name}.evaluate: eval_env has {eval_env.num_envs} envs in "
                             f"groups {list(eval_env._group_sizes)}, the learner's env "
                             f"{env.num_envs} in {list(env._group_sizes)}")
        self._check_eval_layout(eval_env)
        if eval_env.noise != "philox":
            raise ValueError(f"{name}.evaluate: eval_env needs noise='philox' "
                             f"(got {eval_env.noise!r})")
        if any(s_.image_representations for s_ in eval_env._group_specs):
            raise ValueError(f"{name}.evaluate: eval_env has image_representations")
        if not eval_env.autoreset or eval_env.horizon < 1:
            raise ValueError(f"{name}.evaluate: eval_env needs autoreset=True and a "
                             "horizon >= 1")

    def _evaluate(self, eval_env, episodes, entry, params, per_env):
        """One evaluation launch of `entry` with `params` (an _lib.EvalParams
        holding the policy) on eval_env, after eval_env.reset()."""
        E = int(episodes)
        if E < 1:
            raise ValueError(f"episodes must be >= 1, got {episodes}")
        self._check_eval_env(eval_env)
        eval_env.reset()
        N, dev = eval_env.num_envs, eval_env.device
        T = E * eval_env.horizon
        ret_sum = torch.empty(N, dtype=torch.float64, device=dev)
        ret_count = torch.empty(N, dtype=torch.int32, device=dev)
        len_sum = torch.empty(N, dtype=torch.int64, device=dev)
        params.episodes = E
        params.ret_sum, params.ret_count = _ptr(ret_sum), _ptr(ret_count)
        params.len_sum = _ptr(len_sum)
        io = eval_env._io(None, {})
        opts = eval_env._opts(T, noise_mode=_lib.MDPP_NOISE_PHILOX)
        eval_env._check(entry(eval_env._ctx, C.byref(eval_env._state), C.byref(io),
                              C.byref(params), C.byref(opts), eval_env._stream()))
        eval_env._step_index += T
        # every episode is at most `horizon` steps long, so E * horizon steps
        # complete E of them in every env
        if not bool((ret_count == E).all()):
            raise RuntimeError(f"evaluate: an env completed {int(ret_count.min())} of "
                               f"{E} episodes in {T} steps")
        group = torch.repeat_interleave(
            torch.arange(eval_env.n_groups, device=dev),
            torch.tensor(eval_env._group_sizes, device=dev))
        per_group = torch.zeros((3, eval_env.n_groups), dtype=torch.float64, device=dev)
        per_group[0].index_add_(0, group, ret_count.to(torch.float64))
        per_group[1].index_add_(0, group, ret_sum)
        per_group[2].index_add_(0, group, len_sum.to(torch.float64))
        ep, tot, length = per_group.cpu().numpy()
        out = {"episodes": ep, "episode_reward_mean": tot / ep,
               "episode_len_mean": length / ep}
        if per_env:
            out.update(ret_sum=ret_sum, ret_count=ret_count, len_sum=len_sum)
        return out

    def episode_returns(self, clear=False):
        """Per config group: "episodes" completed by an auto-reset since the
        last clear, and their mean return "episode_reward_mean" (NaN when
        none completed).  clear=True starts the next count (the running
        episodes carry on)."""
        env, dev = self.env, self.ret_sum.device
        group = torch.repeat_interleave(
            torch.arange(env.n_groups, device=dev),
            torch.tensor(env._group_sizes, device=dev))
        per_group = torch.zeros((2, env.n_groups), dtype=torch.float64, device=dev)
        per_group[0].index_add_(0, group, self.ret_count.to(torch.float64))
        per_group[1].index_add_(0, group, self.ret_sum)
        ep, tot = per_group.cpu().numpy()
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = np.where(ep > 0, tot / np.maximum(ep, 1), np.nan)
        if clear:
            self.ret_sum.zero_()
            self.ret_count.zero_()
        return {"episodes": ep, "episode_reward_mean": mean}


class TabularQLearner(EpisodeReturns):
    """Per-env tabular Q-learning on a discrete env (Philox noise, no
    irrelevant features, no image observations).  Grid envs train with
    GridQLearner.

    q: float64 [N, S_max, A_max] device tensor (S_max / A_max over the config
    groups; entries beyond an env's own S or A stay at q_init)."""

    def __init__(self, env, alpha=0.1, gamma=0.99, epsilon=0.1, q_init=0.0):
        self._check_env(env)
        super().__init__(env)
        self.alpha = _unit("alpha", alpha)
        self.gamma = _unit("gamma", gamma)
        self.epsilon = _unit("epsilon", epsilon)
        S, A = self._table_shape()
        self.q = torch.full((env.num_envs, S, A), float(q_init), dtype=torch.float64,
                            device=env.device)

    # -- what differs between the env kinds -----------------------------------
    def _check_env(self, env):
        from .discrete_env import DiscreteEnv
        if not isinstance(env, DiscreteEnv):
            raise ValueError("TabularQLearner needs a discrete env (got "
                             f"{type(env).__name__}; grid envs train with GridQLearner)")
        if env._irr:
            raise ValueError("TabularQLearner does not support irrelevant_features")

    def _table_shape(self):
        tables = self.env.group_tables
        return max(t.n_states for t in tables), max(t.n_actions for t in tables)

    def _check_eval_layout(self, eval_env):
        if eval_env._irr:
            raise ValueError("TabularQLearner.evaluate: eval_env has irrelevant_features")
        shapes = [[(t.n_states, t.n_actions) for t in e.group_tables]
                  for e in (self.env, eval_env)]
        if shapes[0] != shapes[1]:
            raise ValueError("TabularQLearner.evaluate: eval_env's groups have (S, A) "
                             f"{shapes[1]}, the learner's {shapes[0]}")

    def _entry(self):
        return self.env._lib.mdpp_discrete_qlearn

    def _eval_entry(self):
        return self.env._lib.mdpp_discrete_qeval

    def _before_launch(self):
        pass

    def _actions_out(self, idx):
        return idx

    def learn(self, n_steps, record=False, alpha=None, gamma=None, epsilon=None):
        """T steps of acting, stepping and learning in one launch.  Returns
        None, or with record=True a dict of time-major [T, N] tensors: obs
        (state after the step and any auto-reset), reward, terminated,
        truncated and the actions taken (GridQLearner: int64 [T, N, n_dims]
        action rows, which env.rollout(actions=...) accepts).  alpha / gamma
        / epsilon override the constructor's values for this call (e.g.
        epsilon=0, alpha=0 for a greedy run that leaves q unchanged; evaluate()
        measures the greedy policy on a separate evaluation env)."""
        T = int(n_steps)
        self._before_launch()
        qp = self._new_params(_lib.QlearnParams)
        qp.alpha = self.alpha if alpha is None else _unit("alpha", alpha)
        qp.gamma = self.gamma if gamma is None else _unit("gamma", gamma)
        qp.epsilon = self.epsilon if epsilon is None else _unit("epsilon", epsilon)
        qp.q = _ptr(self.q)
        qp.q_states, qp.q_actions = self.q.shape[1], self.q.shape[2]
        out = self._learn(self._entry(), qp, T, record, (), torch.int32)
        if record:
            out["actions"] = self._actions_out(out["actions"])
        return out

    def evaluate(self, eval_env, episodes=10, per_env=False):
        """The greedy policy of the current q (argmax, lowest index on ties;
        no exploration, q only read) on eval_env, an env built like the
        learner's (typically without its noises): eval_env.reset(), then one
        launch of episodes * eval_env.horizon steps in which the first
        `episodes` episodes of every env are counted.  Leaves q, the
        training env and episode_returns untouched.  Returns per config
        group (numpy [G]): "episodes" counted, and their mean return
        "episode_reward_mean" and mean length "episode_len_mean"; with
        per_env=True also the per-env device tensors "ret_sum", "ret_count"
        and "len_sum"."""
        ep = _lib.EvalParams()
        ep.q = _ptr(self.q)
        ep.q_states, ep.q_actions = self.q.shape[1], self.q.shape[2]
        return self._evaluate(eval_env, episodes, self._eval_entry(), ep, per_env)


class GridQLearner(TabularQLearner):
    """Per-env tabular Q-learning on a grid env (Philox noise, no image
    observations; 2-D grids and irrelevant_features), one fused launch of
    mdpp_grid_qlearn per learn(T).  The state is the cell's row-major index
    over [0, shape_k], one past the grid included (grid_cells), the action
    the index of a GridActionSpace member (grid_action_rows).

    q: float64 [N, S_max, A], S_max = prod_k (shape_k + 1) over the config
    groups, A = 8 for 2-D grids (one 64-byte row; 5 actions are used) and 9
    for 4-D ones.  learn() raises ValueError when a cell lies outside
    [0, shape_k] (e.g. one set by set_augmented_state): it has no table row."""

    def _check_env(self, env):
        from .grid_env import GridEnv
        if not isinstance(env, GridEnv):
            raise ValueError(f"GridQLearner needs a grid env (got {type(env).__name__})")
        dev = env.device
        self._action_rows = torch.as_tensor(grid_action_rows(env._nd), device=dev)
        # [nd, N] largest coordinate of each env's cells
        self._cell_max = torch.repeat_interleave(
            torch.tensor([list(s_.grid_shape) for s_ in env._group_specs],
                         dtype=torch.int32), torch.tensor(env._group_sizes),
            dim=0).t().contiguous().to(dev)

    def _table_shape(self):
        env = self.env
        return (max(grid_cells(s_.grid_shape) for s_ in env._group_specs),
                8 if env._nd == 2 else 9)

    def _check_eval_layout(self, eval_env):
        shapes = [[tuple(s_.grid_shape) for s_ in e._group_specs]
                  for e in (self.env, eval_env)]
        if shapes[0] != shapes[1]:
            raise ValueError(f"GridQLearner.evaluate: eval_env's grid shapes {shapes[1]} "
                             f"differ from the learner's {shapes[0]}")

    def _entry(self):
        return self.env._lib.mdpp_grid_qlearn

    def _eval_entry(self):
        return self.env._lib.mdpp_grid_qeval

    def _before_launch(self):
        pos = self.env._pos
        if bool(((pos < 0) | (pos > self._cell_max)).any()):
            raise ValueError("GridQLearner: a grid cell lies outside [0, grid_shape] "
                             "(set_augmented_state / reset(init_state=...))")

    def _actions_out(self, idx):
        T, N = idx.shape
        return torch.index_select(self._action_rows, 0,
                                  idx.reshape(-1)).reshape(T, N, -1)
