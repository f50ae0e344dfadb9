"""Experiment-grid front end (SURVEY.md 8f row N4): run a reference experiment
file's environment grid as ONE heterogeneous VectorRLToyEnv.

The reference expands `var_env_configs` of an `experiments/*.py` module into
a Cartesian grid (config_processor.get_grid_of_configs,
config_processor/config_processor.py:492-517), merges every cell over the
static `env_config["env_config"]` and hands each to a separate Ray trial
(scripts/run_experiments.py:231-276).  Here every cell becomes one
configuration group of a single batched env, stepped by one kernel launch,
and the per-cell episode statistics are written in the reference's CSV layout
(config_processor.py:241-259, :340-373) so its analysis code can read them.
Continuous and grid experiment files run the same way, image observations
included: each cell renders with its own image settings (discrete transforms
and their quantisation, continuous / grid targets, terminal regions and
bounds).  Only cells that cannot share one launch (different state dimension
/ dtype, image size) get one batched env per cell instead.  `run` steps a
uniform random policy (or one supplied by the caller); `train` (discrete
experiments) and `train_grid` (grid-world experiments) train a tabular
Q-learning agent per env inside the step kernel (qlearning.py), and
`train_continuous` (continuous experiments) one linear ARS policy per cell
(ars.py); each writes a learning curve per cell, one CSV row per (training
iteration, cell) like the reference's stats files.
"""
import copy
import importlib.util
import itertools
import os
import sys
import types
from collections import OrderedDict

import numpy as np


def _ray_stub():
    """The experiment files do `from ray import tune` and only use
    `tune.grid_search([...])` in agent configs; ray itself is not needed to
    read the environment grid."""
    ray = types.ModuleType("ray")
    tune = types.ModuleType("ray.tune")
    tune.grid_search = lambda values: {"grid_search": list(values)}
    tune.choice = lambda values: {"choice": list(values)}
    tune.uniform = lambda a, b: {"uniform": (a, b)}
    tune.function = lambda f: f  # old Ray API the eval configs still use
    ray.tune = tune
    return {"ray": ray, "ray.tune": tune}


def load_experiment(path):
    """Import an experiment module (stubbing `ray` if it is not installed)."""
    path = os.path.abspath(path)
    if not path.endswith(".py"):
        path += ".py"
    stubs = {}
    try:
        import ray  # noqa: F401
    except ModuleNotFoundError:
        stubs = _ray_stub()
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        spec = importlib.util.spec_from_file_location(
            "mdpp_experiment_" + os.path.basename(path)[:-3], path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


def expand_grid(var_configs):
    """get_grid_of_configs (:492-517): Cartesian product of every leaf list,
    in the dict's iteration order.  Returns (keys, list of value tuples) with
    keys as (config_type, key) pairs."""
    keys, values = [], []
    for config_type, config_dict in var_configs.items():
        for key, leaf in config_dict.items():
            assert isinstance(leaf, list), (
                "var_configs should be a dict of dicts with lists as the leaf "
                "values to allow each configuration option to take multiple "
                "possible values")
            keys.append((config_type, key))
            values.append(leaf)
    cells = list(itertools.product(*values)) if values else []
    return keys, cells


def env_grid(module):
    """(var env keys, list of per-cell env config dicts) of an experiment."""
    var_configs = getattr(module, "var_configs", None)
    if var_configs is None:
        var_configs = OrderedDict({"env": module.var_env_configs})
    keys, cells = expand_grid(var_configs)
    static = copy.deepcopy(module.env_config.get("env_config", {}))
    env_keys = [k for t, k in keys if t == "env"]
    out = []
    for cell in cells:
        cfg = copy.deepcopy(static)
        for (t, k), v in zip(keys, cell):
            if t == "env":
                cfg[k] = v
        out.append(cfg)
    return env_keys, out


class _NormalProbe:
    """Stands in for the numpy Generator that the reference passes to a noise
    callable: records every call made on it."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def record(*args, **kwargs):
            self.calls.append((name, args, kwargs))
            return self
        return record


def noise_std(key, f):
    """The sigma of a noise callable of the reference's evaluation configs,
    `tune.function(lambda a: a.normal(0, sigma))`: one `normal(0, sigma)`
    call with constant arguments, whose draw is the callable's value.
    Anything else raises NotImplementedError naming `key`."""
    probe = _NormalProbe()
    try:
        out = f(probe)
    except Exception as e:
        raise NotImplementedError(
            f"evaluation env_config[{key!r}]: only lambda a: a.normal(0, sigma) is "
            f"supported (calling it raised {type(e).__name__})") from None
    ok = out is probe and len(probe.calls) == 1 and probe.calls[0][0] == "normal"
    if ok:
        _, args, kwargs = probe.calls[0]
        names = ("loc", "scale")
        ok = len(args) <= 2 and set(kwargs) <= set(names[len(args):])
        if ok:
            vals = dict(zip(names, args), **kwargs)
            loc, scale = vals.get("loc", 0.0), vals.get("scale", 1.0)
            ok = all(isinstance(v, (int, float, np.integer, np.floating))
                     and not isinstance(v, bool) for v in (loc, scale)) \
                and float(loc) == 0.0 and np.isfinite(scale) and float(scale) >= 0.0
    if not ok:
        raise NotImplementedError(
            f"evaluation env_config[{key!r}]: only lambda a: a.normal(0, sigma) with "
            f"constant sigma >= 0 is supported (got calls {probe.calls})")
    return float(scale)


# keys of the reference's evaluation_config that configure the agent, not the env
_AGENT_EVAL_KEYS = ("explore",)


def eval_settings(module, evaluation, horizon):
    """The evaluation of an experiment: the module's `eval_config` (the
    reference's RLlib layout: top-level "evaluation_interval", and in
    "evaluation_config" "evaluation_num_episodes", "horizon" and the
    "env_config" overrides; agent keys such as "explore" and
    "exploration_*" are ignored), with the entries of a dict `evaluation`
    on top (the same four names, "env_config" merged key by key).
    Noise callables become their sigma (noise_std).  Returns a dict of
    "interval", "episodes", "horizon" and "env_config"."""
    ec = copy.deepcopy(getattr(module, "eval_config", None) or {})
    inner = ec.get("evaluation_config", {}) or {}
    out = {"interval": ec.get("evaluation_interval", 1),
           "episodes": inner.get("evaluation_num_episodes",
                                 ec.get("evaluation_num_episodes", 10)),
           "horizon": inner.get("horizon", horizon),
           "env_config": dict(inner.get("env_config", {}) or {})}
    if isinstance(evaluation, dict):
        known = {"evaluation_interval", "evaluation_num_episodes", "horizon", "env_config"}
        if set(evaluation) - known:
            raise ValueError(f"evaluation: unknown keys {sorted(set(evaluation) - known)} "
                             f"(known: {sorted(known)})")
        out["interval"] = evaluation.get("evaluation_interval", out["interval"])
        out["episodes"] = evaluation.get("evaluation_num_episodes", out["episodes"])
        out["horizon"] = evaluation.get("horizon", out["horizon"])
        out["env_config"].update(evaluation.get("env_config", {}) or {})
    for key in ("interval", "episodes", "horizon"):
        v = out[key]
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or v < 1:
            raise ValueError(f"evaluation {key} must be an integer >= 1, got {v!r}")
        out[key] = int(v)
    env_cfg = {}
    for k, v in out["env_config"].items():
        if k in _AGENT_EVAL_KEYS or k.startswith("exploration_"):
            continue
        env_cfg[k] = noise_std(k, v) if callable(v) else v
    out["env_config"] = env_cfg
    return out


def eval_cell_configs(cell_configs, env_config):
    """Each cell's config with the evaluation's env overrides on top."""
    return [dict(copy.deepcopy(c), **copy.deepcopy(env_config)) for c in cell_configs]


class Sweep:
    """All cells of an experiment's env grid in one VectorRLToyEnv."""

    def __init__(self, experiment, envs_per_cell=64, horizon=None, device=None,
                 shard=(0, 1), **env_kwargs):
        from .vector_env import VectorRLToyEnv
        self.module = load_experiment(experiment) if isinstance(experiment, str) \
            else experiment
        self.env_keys, self.cell_configs = env_grid(self.module)
        self.n_cells = len(self.cell_configs)
        if horizon is None:
            horizon = int(self.module.env_config.get("horizon", 100))
        self.envs_per_cell = int(envs_per_cell)
        self.world = int(shard[1])
        kinds = {str(c.get("state_space_type", "")).lower()
                 for c in self.cell_configs}
        assert len(kinds) == 1, "one state_space_type per experiment file"
        self.kind = kinds.pop()
        self._env_args = (device, shard, env_kwargs)
        if self.kind == "discrete":
            # the whole grid is ONE heterogeneous env: one launch per rollout
            self.env = VectorRLToyEnv(
                self.n_cells * self.envs_per_cell, device=device, autoreset=True,
                horizon=horizon, config_groups=self.cell_configs,
                group_sizes=[self.envs_per_cell] * self.n_cells, shard=shard,
                **env_kwargs)
            self.envs = [self.env]
        elif self._try_grouped(VectorRLToyEnv, device, horizon, shard, env_kwargs):
            pass  # the whole grid is ONE heterogeneous env here too
        else:
            # cells that differ in what shapes the state arrays (continuous:
            # dimension or dtype; grid: irrelevant_features) take one
            # configuration per context: one env per cell, launched back to
            # back on the same stream
            self.envs = self._per_cell_envs(self.cell_configs, horizon)
            self.env = self.envs[0]
        self.timesteps = 0
        self._returned = np.zeros(self.n_cells)
        self.agents = None  # one learner per env of self.envs
        self.algorithm = None  # the learner's name in write_csv once one has trained
        self.train_results = []  # one dict per training iteration
        self.eval_envs = None  # evaluation envs, laid out like self.envs
        self.evaluation = None  # eval_settings() of the first train(evaluation=...)
        self.eval_results = []  # one dict per evaluated training iteration

    def _per_cell_envs(self, cell_configs, horizon):
        from .vector_env import VectorRLToyEnv
        device, (rank, world), env_kwargs = self._env_args
        return [VectorRLToyEnv(
            self.envs_per_cell, device=device, autoreset=True,
            horizon=horizon,
            env_id_offset=(i * world + rank) * self.envs_per_cell,
            **env_kwargs, **copy.deepcopy(c))
            for i, c in enumerate(cell_configs)]

    def _build_eval_envs(self, evaluation):
        """The evaluation envs, once: the layout of self.envs (one grouped
        env, or one env per cell with the same env ids), each cell's config
        with the evaluation's env overrides on top."""
        if self.eval_envs is not None:
            return
        from .vector_env import VectorRLToyEnv
        self.evaluation = eval_settings(self.module, evaluation, self.env.horizon)
        cfgs = eval_cell_configs(self.cell_configs, self.evaluation["env_config"])
        horizon = self.evaluation["horizon"]
        device, shard, env_kwargs = self._env_args
        if self.kind == "discrete" or getattr(self, "grouped", False):
            self.eval_envs = [VectorRLToyEnv(
                self.n_cells * self.envs_per_cell, device=device, autoreset=True,
                horizon=horizon, config_groups=cfgs,
                group_sizes=[self.envs_per_cell] * self.n_cells, shard=shard,
                **env_kwargs)]
        else:
            self.eval_envs = self._per_cell_envs(cfgs, horizon)

    def _try_grouped(self, Env, device, horizon, shard, env_kwargs):
        """Continuous cells that share dim / dtype / reward function, and grid
        cells that share the number of coordinates, run as config groups of
        one env: one launch per rollout for the whole grid
        (e.g. experiments/sac_move_to_a_point_p_order_2.py:10-30), and one
        render launch per observation when the cells have images."""
        try:
            self.env = Env(
                self.n_cells * self.envs_per_cell, device=device, autoreset=True,
                horizon=horizon, config_groups=copy.deepcopy(self.cell_configs),
                group_sizes=[self.envs_per_cell] * self.n_cells, shard=shard,
                **env_kwargs)
        except (ValueError, NotImplementedError):
            return False
        self.envs = [self.env]
        self.grouped = True
        if self.kind == "grid":
            return True
        import torch
        amax = torch.tensor([float(c.get("action_space_max", np.inf))
                             for c in self.cell_configs], device=self.env.device)
        self._amax = amax.repeat_interleave(self.envs_per_cell).to(self.env._real)
        return True

    def run(self, steps_per_env, chunk=256, actions_fn=None):
        """Random-policy (or `actions_fn(t0, T) -> int32[T, N]`) rollouts."""
        import torch
        done = 0
        while done < steps_per_env:
            T = min(chunk, steps_per_env - done)
            if self.kind == "discrete" or getattr(self, "grouped", False):
                acts = None if actions_fn is None else actions_fn(done, T)
                if acts is None and self.kind == "continuous":
                    acts = self._random_actions_grouped(T, done)
                elif acts is None and self.kind == "grid":
                    acts = self._random_actions(self.env, T, done)
                out = self.env.rollout(T, actions=acts, want_final_obs=False)
                r = out["reward"].sum(dim=0).reshape(self.n_cells,
                                                     self.envs_per_cell)
                self._returned += r.sum(dim=1).to(torch.float64).cpu().numpy()
            else:
                for i, env in enumerate(self.envs):
                    acts = self._random_actions(env, T, done) \
                        if actions_fn is None else actions_fn(done, T, i)
                    out = env.rollout(T, actions=acts, want_final_obs=False)
                    self._returned[i] += float(out["reward"].sum())
            done += T
        self.timesteps += steps_per_env
        return self.results()

    def train(self, iterations, steps_per_iteration, alpha=0.1, gamma=0.99,
              epsilon=0.1, chunk=256, evaluation=None):
        """Tabular Q-learning (one agent per env; envs_per_cell seeds per
        cell), `iterations` times `steps_per_iteration` steps per env.  Each
        iteration appends to `train_results`, per cell: the cumulative
        timesteps_total, episode_reward_mean (mean return of the episodes
        completed in the iteration; NaN if none) and episode_len_mean (from
        the episode counters' change over the iteration).  Discrete grids
        only (grid-world experiments: train_grid).  Calling train again
        continues with the same Q-tables.

        evaluation: None (none), True (the experiment file's eval_config) or
        a dict overriding it (eval_settings).  Every evaluation_interval-th
        iteration then evaluates every agent's greedy policy
        (TabularQLearner.evaluate) on evaluation envs built once like the
        training envs, with the evaluation's env_config on top of each
        cell's config, and appends to `eval_results`, per cell: the
        training_iteration, its timesteps_total, and the evaluation
        episodes' episode_reward_mean and episode_len_mean (write_eval_csv).
        The settings and envs of the first evaluating call are kept.
        Rank-local, like train_results."""
        return self._train_q(
            "discrete", "Sweep.train: tabular Q-learning runs on discrete grids only "
            "(grid-world experiments: Sweep.train_grid)",
            iterations, steps_per_iteration, alpha, gamma, epsilon, chunk, evaluation)

    def train_grid(self, iterations, steps_per_iteration, alpha=0.1, gamma=0.99,
                   epsilon=0.1, chunk=256, evaluation=None):
        """train() for grid-world experiments (GridQLearner): one learner on
        the grouped env, or one per cell when the cells differ in
        irrelevant_features; results in cell order either way."""
        return self._train_q("grid", "Sweep.train_grid: runs grid-world experiments only",
                             iterations, steps_per_iteration, alpha, gamma, epsilon, chunk,
                             evaluation)

    def _train_q(self, kind, refusal, iterations, steps_per_iteration, alpha, gamma,
                 epsilon, chunk, evaluation=None):
        """train / train_grid: `refusal` is the NotImplementedError message
        for experiments of another kind than `kind`."""
        if self.kind != kind:
            raise NotImplementedError(refusal)
        from .qlearning import GridQLearner, TabularQLearner
        learner = GridQLearner if kind == "grid" else TabularQLearner
        kw = dict(alpha=alpha, gamma=gamma, epsilon=epsilon)
        return self._train(lambda e: learner(e, **kw), iterations, steps_per_iteration,
                           chunk, kw, "TabularQLearning", evaluation=evaluation)

    def train_continuous(self, iterations, steps_per_iteration, step_size=0.02,
                         noise_std=0.03, top_directions=None, chunk=256, evaluation=None):
        """train() for continuous experiments: augmented random search
        (ars.LinearARS), one linear policy per cell whose envs_per_cell envs
        (an even number) are the perturbation population.  One learner on the
        grouped env, or one per cell when the cells differ in dimension or
        dtype.  Each iteration runs `steps_per_iteration` steps per env (the
        learn chunks), then one ARS update per cell, and appends the same
        per-cell results as train().  Calling it again continues with the
        same policies.  Not for sharded sweeps (the update is per rank).
        evaluation: as in train(), evaluating theta itself
        (LinearARS.evaluate)."""
        if self.kind != "continuous":
            raise NotImplementedError(
                "Sweep.train_continuous: runs continuous experiments only")
        if self.world > 1:
            raise NotImplementedError(
                "Sweep.train_continuous: a sharded sweep would need a cross-rank "
                "ARS update")
        from .ars import LinearARS
        return self._train(
            lambda e: LinearARS(e, step_size=step_size, noise_std=noise_std,
                                top_directions=top_directions),
            iterations, steps_per_iteration, chunk, {}, "ARS", update=True,
            evaluation=evaluation)

    def _train(self, make, iterations, steps_per_iteration, chunk, learn_kw,
               algorithm, update=False, evaluation=None):
        if self.agents is None:
            self.agents = [make(e) for e in self.envs]
        self.algorithm = algorithm
        evaluate = evaluation is not None and evaluation is not False
        if evaluate:
            self._build_eval_envs(evaluation)

        def per_cell(dicts, key):  # one value per group of each env, in cell order
            return np.concatenate([np.asarray(d[key]).reshape(-1) for d in dicts])
        for ag in self.agents:
            ag.episode_returns(clear=True)
        for _ in range(int(iterations)):
            before = [e.episode_stats() for e in self.envs]
            done = 0
            while done < steps_per_iteration:
                T = min(chunk, steps_per_iteration - done)
                for ag in self.agents:
                    ag.learn(T, **learn_kw)
                done += T
            if update:
                for ag in self.agents:
                    ag.update()
            self.timesteps += steps_per_iteration
            after = [e.episode_stats() for e in self.envs]
            ret = [ag.episode_returns(clear=True) for ag in self.agents]
            d_ep = per_cell(after, "episodes") - per_cell(before, "episodes")
            d_tr = per_cell(after, "transitions") - per_cell(before, "transitions")
            self.train_results.append({
                "training_iteration": len(self.train_results) + 1,
                "timesteps_total": per_cell(after, "transitions"),
                "episode_reward_mean": per_cell(ret, "episode_reward_mean"),
                "episode_len_mean": d_tr / np.maximum(d_ep, 1)})
            it = len(self.train_results)
            if evaluate and it % self.evaluation["interval"] == 0:
                ev = [ag.evaluate(e, self.evaluation["episodes"])
                      for ag, e in zip(self.agents, self.eval_envs)]
                self.eval_results.append({
                    "training_iteration": it,
                    "timesteps_total": per_cell(after, "transitions"),
                    "episode_reward_mean": per_cell(ev, "episode_reward_mean"),
                    "episode_len_mean": per_cell(ev, "episode_len_mean")})
        return self.train_results

    def _random_actions(self, env, T, t0):
        """Uniform random policy for the per-cell envs (continuous: uniform
        in the action box, or N(0, 1) when it is unbounded; grid: one unit
        move or the no-op), seeded per env and chunk."""
        import torch
        N, dev = env.num_envs, env.device
        gen = torch.Generator(dev).manual_seed(
            (env.philox_seed + 7919 * env.env_id_offset + t0) % (2**63))
        if self.kind == "grid":
            nd = env._nd
            acts = torch.zeros((T, N, nd), dtype=torch.int64, device=dev)
            dim = torch.randint(0, nd, (T, N, 1), device=dev, generator=gen)
            acts.scatter_(2, dim, torch.randint(-1, 2, (T, N, 1), device=dev,
                                                generator=gen))
            return acts
        D, amax = env.spec.state_space_dim, env.spec.action_space_max
        if np.isfinite(amax):
            u = torch.rand((T, N, D), device=dev, generator=gen, dtype=env._real)
            return (u * 2 - 1) * amax
        return torch.randn((T, N, D), device=dev, generator=gen, dtype=env._real)

    def _random_actions_grouped(self, T, t0):
        """Uniform in every cell's own action box (N(0, 1) where unbounded)."""
        import torch
        env = self.env
        N, D, dev = env.num_envs, env.spec.state_space_dim, env.device
        gen = torch.Generator(dev).manual_seed(
            (env.philox_seed + 7919 * (env._shard[0] + 1) + t0) % (2**63))
        u = torch.rand((T, N, D), device=dev, generator=gen, dtype=env._real) * 2 - 1
        z = torch.randn((T, N, D), device=dev, generator=gen, dtype=env._real)
        bounded = torch.isfinite(self._amax)[None, :, None]
        return torch.where(bounded, u * torch.nan_to_num(self._amax, posinf=1.0)[None, :, None], z)

    def results(self, reduce=False):
        if self.kind == "discrete" or getattr(self, "grouped", False):
            st = self.env.episode_stats(reduce=reduce)
        else:  # one single-group env per cell
            per = [e.episode_stats(reduce=reduce) for e in self.envs]
            st = {k: np.array([float(np.asarray(p[k]).reshape(-1)[0]) for p in per])
                  for k in ("episodes", "transitions", "noisy_transitions")}
        ep = np.maximum(st["episodes"], 1)
        returned = self._returned
        if reduce:  # the reward sums are rank-local like the counters
            import torch
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                dev = self.env.device if self.kind == "discrete" else self.envs[0].device
                use_cuda = dist.get_backend() == "nccl"
                t = torch.as_tensor(returned, dtype=torch.float64,
                                    device=dev if use_cuda else "cpu").clone()
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                returned = t.cpu().numpy()
        return {"episodes": st["episodes"], "transitions": st["transitions"],
                "episode_reward_mean": returned / ep,
                "episode_len_mean": st["transitions"] / ep,
                "noisy_transitions": st["noisy_transitions"]}

    def write_csv(self, path, algorithm=None):
        """The reference's stats-file layout: one row per grid cell, or, once
        `train` has run, one row per (training iteration, cell).  algorithm
        defaults to "RandomPolicy", or after training to the learner's name
        ("TabularQLearning", or "ARS" after `train_continuous`)."""
        if self.train_results:
            iters = self.train_results
            algorithm = algorithm or self.algorithm
        else:
            res = self.results()
            iters = [{"training_iteration": 1, "timesteps_total": res["transitions"],
                      "episode_reward_mean": res["episode_reward_mean"],
                      "episode_len_mean": res["episode_len_mean"]}]
            algorithm = algorithm or "RandomPolicy"
        return self._write_rows(path, iters, algorithm)

    def write_eval_csv(self, path, algorithm=None):
        """The evaluation results (eval_results) in write_csv's column
        layout: one row per (evaluated training iteration, cell) with the
        training iteration, its timesteps_total, and the evaluation
        episodes' mean return and mean length.  The reference's callbacks
        write evaluation episodes to a stats file of their own, which its
        analysis code loads next to the training file; whether that file
        has exactly these columns has not been checked against the
        reference.  Rank-local, like write_csv."""
        return self._write_rows(path, self.eval_results, algorithm or self.algorithm)

    def _write_rows(self, path, iters, algorithm):
        with open(path, "w") as f:
            f.write("# training_iteration, algorithm, "
                    + "".join(k + ", " for k in self.env_keys)
                    + "timesteps_total, episode_reward_mean, episode_len_mean\n")
            for it in iters:
                for i, cfg in enumerate(self.cell_configs):
                    row = [str(it["training_iteration"]), algorithm]
                    for k in self.env_keys:
                        v = cfg[k]
                        row.append("%.2e" % v if isinstance(v, float)
                                   else str(v).replace(" ", ""))
                    row += [str(int(it["timesteps_total"][i])),
                            "%.2e" % it["episode_reward_mean"][i],
                            "%.2e" % it["episode_len_mean"][i]]
                    f.write(" ".join(row) + "\n")
        return path
