"""Tabular Q-learning inside the discrete rollout kernel.

`TabularQLearner(env)` gives every env of a discrete VectorRLToyEnv its own
Q-table, float64 [N, S_max, A_max] on the device, and trains all of them in
one fused launch per `learn(T)` call (mdpp_discrete_qlearn,
include/mdpp_b200.h): epsilon-greedy action selection, the env step and the
one-step Q-learning update, T steps per launch.  Each env is one independent
training run (one seed); in a grouped env each config group is one cell of an
experiment grid.

The exploring action is the random policy's own draw (`rollout(actions=None)`
at the same global step), so with epsilon = 1 `learn` takes exactly the
actions a random rollout would take.  The env's step counter advances by T,
like rollout(), so later rollout / step / reseed calls behave as they would
after a rollout of T steps.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import _ptr


def _unit(name, x):
    x = float(x)
    if not 0.0 <= x <= 1.0:
        raise ValueError(f"{name} must lie in [0, 1], got {x}")
    return x


class TabularQLearner:
    """Per-env tabular Q-learning on a discrete env (Philox noise, no
    irrelevant features, no image observations).

    q: float64 [N, S_max, A_max] device tensor (S_max / A_max over the config
    groups; entries beyond an env's own S or A stay at q_init)."""

    def __init__(self, env, alpha=0.1, gamma=0.99, epsilon=0.1, q_init=0.0):
        from .discrete_env import DiscreteEnv
        if not isinstance(env, DiscreteEnv):
            raise ValueError("TabularQLearner needs a discrete env "
                             f"(got {type(env).__name__})")
        if env.noise != "philox":
            raise ValueError("TabularQLearner needs noise='philox' "
                             f"(got {env.noise!r})")
        if env._irr:
            raise ValueError("TabularQLearner does not support irrelevant_features")
        if any(s_.image_representations for s_ in env._group_specs):
            raise ValueError("TabularQLearner does not support image_representations")
        self.env = env
        self.alpha = _unit("alpha", alpha)
        self.gamma = _unit("gamma", gamma)
        self.epsilon = _unit("epsilon", epsilon)
        N, dev = env.num_envs, env.device
        S = max(t.n_states for t in env.group_tables)
        A = max(t.n_actions for t in env.group_tables)
        self.q = torch.full((N, S, A), float(q_init), dtype=torch.float64, device=dev)
        # return of each env's running episode, and sum / count of the returns
        # of the episodes that ended in an auto-reset
        self.ep_return = torch.zeros(N, dtype=torch.float64, device=dev)
        self.ret_sum = torch.zeros(N, dtype=torch.float64, device=dev)
        self.ret_count = torch.zeros(N, dtype=torch.int32, device=dev)

    def learn(self, n_steps, record=False, alpha=None, gamma=None, epsilon=None):
        """T steps of acting, stepping and learning in one launch.  Returns
        None, or with record=True a dict of time-major [T, N] tensors: obs
        (state after the step and any auto-reset), reward, terminated,
        truncated and the actions taken.  alpha / gamma / epsilon override
        the constructor's values for this call (e.g. epsilon=0, alpha=0 for a
        greedy evaluation that leaves q unchanged)."""
        env = self.env
        T = int(n_steps)
        qp = _lib.QlearnParams()
        qp.alpha = self.alpha if alpha is None else _unit("alpha", alpha)
        qp.gamma = self.gamma if gamma is None else _unit("gamma", gamma)
        qp.epsilon = self.epsilon if epsilon is None else _unit("epsilon", epsilon)
        qp.q = _ptr(self.q)
        qp.q_states, qp.q_actions = self.q.shape[1], self.q.shape[2]
        qp.ep_return, qp.ret_sum = _ptr(self.ep_return), _ptr(self.ret_sum)
        qp.ret_count = _ptr(self.ret_count)
        out = {}
        if record:
            out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
            out["actions"] = torch.empty((T, env.num_envs), dtype=torch.int32,
                                         device=env.device)
            qp.actions_taken = _ptr(out["actions"])
        io = env._io(None, out)
        opts = env._opts(T)
        env._check(env._lib.mdpp_discrete_qlearn(
            env._ctx, C.byref(env._state), C.byref(io), C.byref(qp),
            C.byref(opts), env._stream()))
        env._step_index += T
        return out if record else None

    def episode_returns(self, clear=False):
        """Per config group: "episodes" completed by an auto-reset since the
        last clear, and their mean return "episode_reward_mean" (NaN when
        none completed).  clear=True starts the next count (the running
        episodes carry on)."""
        env, dev = self.env, self.q.device
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
