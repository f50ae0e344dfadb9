"""Augmented random search (ARS V1 / V1-t; Mania, Guy & Recht 2018) inside
the continuous rollout kernel.

`LinearARS(env)` trains one linear policy a = W [obs; 1] per config group of
a continuous VectorRLToyEnv (one group: the whole env).  The group's envs are
the perturbation population: local envs 2p and 2p + 1 act with
theta + noise_std * delta_p and theta - noise_std * delta_p, where delta_p is
regenerated on the device from a Philox counter (global id of the + member,
iteration), so no action array and no perturbation is stored.  `learn(T)`
runs T fused steps (mdpp_continuous_ars, include/mdpp_b200.h) and adds each
returned reward to the env's fitness; `update()` applies one ARS step per
group from the fitness gathered since the last update
(mdpp_continuous_ars_update) and starts the next iteration.  The env's step
counter advances by T per learn call, like rollout().
"""
import ctypes as C
import math

import torch

from . import _lib
from ._lib import _ptr
from .qlearning import EpisodeReturns


def _positive(name, x, allow_zero=False):
    x = float(x)
    if not math.isfinite(x) or x < 0.0 or (x == 0.0 and not allow_zero):
        raise ValueError(f"{name} must be finite and {'>=' if allow_zero else '>'} 0, "
                         f"got {x}")
    return x


class LinearARS(EpisodeReturns):
    """ARS on a continuous env (Philox noise, no image observations, even
    config-group sizes).

    theta: float64 [G, D, D + 1] device tensor, the groups' master weights
    (row d: the weights of action d on (obs_0, ..., obs_{D-1}, 1)).
    fitness: float64 [N], each env's reward sum since the last update().
    iteration: the update count (the counter word of the perturbations).
    top_directions: pairs kept per update (None: every pair)."""

    def __init__(self, env, step_size=0.02, noise_std=0.03, top_directions=None,
                 theta_init=0.0):
        from .continuous_env import ContinuousEnv
        if not isinstance(env, ContinuousEnv):
            raise ValueError(f"LinearARS needs a continuous env (got {type(env).__name__})")
        super().__init__(env)
        sizes = list(env._group_sizes)
        if any(n % 2 or n < 2 for n in sizes):
            raise ValueError("LinearARS needs an even number (>= 2) of envs per "
                             f"config group (got {sizes})")
        self.step_size = _positive("step_size", step_size)
        self.noise_std = _positive("noise_std", noise_std, allow_zero=True)
        pairs = min(sizes) // 2
        b = pairs if top_directions is None else int(top_directions)
        if not 1 <= b <= pairs:
            raise ValueError(f"top_directions must lie in [1, {pairs}] (the smallest "
                             f"group's pairs), got {top_directions}")
        self.top_directions = b
        N, dev, D = env.num_envs, env.device, env.spec.state_space_dim
        self.D = D
        self.theta = torch.empty((env.n_groups, D, D + 1), dtype=torch.float64, device=dev)
        self.theta[:] = torch.as_tensor(theta_init, dtype=torch.float64)
        self.fitness = torch.zeros(N, dtype=torch.float64, device=dev)
        self.iteration = 0

    def _params(self, noise_std=None):
        env = self.env
        ap = self._new_params(_lib.ArsParams)
        ap.step_size = self.step_size
        ap.noise_std = self.noise_std if noise_std is None else \
            _positive("noise_std", noise_std, allow_zero=True)
        ap.theta, ap.fitness = _ptr(self.theta), _ptr(self.fitness)
        ap.top_directions = self.top_directions
        ap.iteration = self.iteration
        ap.seed = env.philox_seed
        ap.env_id_offset = env.env_id_offset
        return ap

    def learn(self, n_steps, record=False, noise_std=None):
        """T steps of every env acting with its perturbed policy, in one
        launch.  Returns None, or with record=True a dict of time-major
        tensors: obs (state after the step and any auto-reset), reward,
        terminated, truncated and the actions taken ([T, N, D] in dtype_s,
        which env.rollout(actions=...) accepts).  noise_std overrides the
        constructor's for this call (0: every env acts with theta)."""
        env = self.env
        T = int(n_steps)
        return self._learn(env._lib.mdpp_continuous_ars, self._params(noise_std), T, record,
                           (self.D,), env._real)

    def _check_eval_layout(self, eval_env):
        if eval_env.spec.state_space_dim != self.D or eval_env._real != self.env._real:
            raise ValueError(f"LinearARS.evaluate: eval_env has D = "
                             f"{eval_env.spec.state_space_dim} in {eval_env._real}, the "
                             f"learner's env D = {self.D} in {self.env._real}")

    def evaluate(self, eval_env, episodes=10, per_env=False):
        """theta itself (no perturbation) on eval_env, an env built like the
        learner's (typically without its noises): eval_env.reset(), then one
        launch of episodes * eval_env.horizon steps in which the first
        `episodes` episodes of every env are counted.  Leaves theta,
        fitness, iteration, the training env and episode_returns untouched.
        Returns what TabularQLearner.evaluate returns."""
        ep = _lib.EvalParams()
        ep.theta = _ptr(self.theta)
        return self._evaluate(eval_env, episodes, self.env._lib.mdpp_continuous_ars_eval,
                              ep, per_env)

    def update(self):
        """One ARS step per config group from the fitness since the last
        update; then fitness restarts at 0 and the iteration advances.
        Returns per group (numpy [G]): "fitness_mean" and "sigma_R" of the
        kept returns and "updated" (False when sigma_R is 0 or not finite:
        theta is left as it was)."""
        env = self.env
        ap = self._params()
        stats = torch.empty((env.n_groups, 3), dtype=torch.float64, device=env.device)
        ap.group_stats = _ptr(stats)
        env._check(env._lib.mdpp_continuous_ars_update(
            env._ctx, env.num_envs, C.byref(ap), env._stream()))
        self.iteration += 1
        st = stats.cpu().numpy()
        return {"fitness_mean": st[:, 0], "sigma_R": st[:, 1],
                "updated": st[:, 2] != 0.0}

    def perturbations(self):
        """The current iteration's delta as the device computes it: float64
        [N / 2, D, D + 1], row p = pair p (local envs 2p, 2p + 1 of its
        group; pairs in env order)."""
        env = self.env
        ap = self._params()
        delta = torch.empty((env.num_envs // 2, self.D, self.D + 1), dtype=torch.float64,
                            device=env.device)
        ap.delta_out = _ptr(delta)
        env._check(env._lib.mdpp_continuous_ars_perturbations(
            env._ctx, env.num_envs, C.byref(ap), env._stream()))
        return delta

