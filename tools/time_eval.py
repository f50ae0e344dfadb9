"""Times the learners' evaluation launches (evaluate) against their learn
launches and the rollout of the same env.

    python tools/time_eval.py [--envs 65536] [--episodes 10] [--reps 5]

Workloads (horizon 100, E = --episodes, so T = 100 E steps per launch):
  #1, #2  BASELINE configs #1 and #2 at --envs envs (TabularQLearner)
  grid8   an 8 x 8 move_to_a_point grid at --envs envs (GridQLearner)
  ddpg12  the 12 cells of tests/fixtures/ddpg_move_to_a_point_like.py as one
          grouped env, --cell-envs envs per cell (LinearARS)
Arms alternated in one process after warm-up, CUDA events around `--reps`
calls of each:
  evaluate  learner.evaluate(eval_env, E): eval_env.reset(), the launch, the
            per-env episode count check and the per-group means (one sync)
  learn     learner.learn(T) on the training env (no [T, N] output)
  rollout   env.rollout(T, actions=None) (discrete: the device random
            policy) or, for ddpg12, env.rollout(T, actions=...) with actions
            recorded once and already on the device
The eval env is built like the training env.  Prints the card, its power
limit and its max SM clock first: a rate is only meaningful with them.
"""
import argparse
import os
import sys
import warnings

import torch

sys.path.insert(0, ".")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from mdp_playground_b200 import (GridQLearner, LinearARS, TabularQLearner,  # noqa: E402
                                 VectorRLToyEnv)
from mdp_playground_b200.sweep import Sweep  # noqa: E402
from time_qlearn import CONFIGS, card, report, time_arms  # noqa: E402

GRID8 = dict(seed=0, state_space_type="grid", grid_shape=(8, 8), target_point=[5, 5],
             reward_function="move_to_a_point", make_denser=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--cell-envs", type=int, default=65536)
    ap.add_argument("--episodes", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    H, E = 100, a.episodes
    T = H * E
    fixture = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests",
                           "fixtures", "ddpg_move_to_a_point_like.py")
    for label in ("#1", "#2", "grid8", "ddpg12"):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if label == "ddpg12":
                env, ev = (Sweep(fixture, envs_per_cell=a.cell_envs).env for _ in range(2))
            else:
                cfg = GRID8 if label == "grid8" else CONFIGS[label]
                env, ev = (VectorRLToyEnv(a.envs, autoreset=True, horizon=H, **cfg)
                           for _ in range(2))
        arms = {}
        if label == "ddpg12":
            ag = LinearARS(env)
            acts = ag.learn(T, record=True)["actions"]
            out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
            arms["rollout"] = lambda: env.rollout(T, actions=acts, out=out)
        else:
            ag = (GridQLearner if label == "grid8" else TabularQLearner)(env)
            ag.learn(T)  # a non-trivial table
            if label != "grid8":
                out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
                arms["rollout"] = lambda: env.rollout(T, out=out)
        arms["evaluate"] = lambda: ag.evaluate(ev, E)
        arms["learn"] = lambda: ag.learn(T)
        ms = time_arms(arms, a.reps)
        report(label, env.num_envs, T, ms)
        del env, ev, ag
        arms.clear()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
