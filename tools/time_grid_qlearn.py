"""Times the fused grid Q-learning launch (GridQLearner.learn on a grid
env) against the grid rollout with the same number of steps.

    python tools/time_grid_qlearn.py [--reps 10]

Two workloads, 8 x 8 grid, transition noise 0.25, reward noise 1.0 (the N1
grid row's configuration, tools/time_grid.py):
  65 536 envs x 1000 steps (the Q-tables are 340 MB: more than the L2)
  1 M envs x 100 steps (the N1 shape; 5.4 GB of Q-tables)
Three arms alternated in one process after warm-up, CUDA events around
`--reps` launches of each:
  learn          GridQLearner.learn(T): no [T, N] output at all
  learn_record   learn(T, record=True): obs, reward, flags and the action rows
  rollout        env.rollout(T, actions=...) with the action rows already on
                 the device
Prints the card and its power limit first: a rate is only meaningful with them.
"""
import argparse
import os
import sys
import warnings

import torch

sys.path.insert(0, ".")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from mdp_playground_b200 import GridQLearner, VectorRLToyEnv  # noqa: E402
from time_qlearn import card, report, time_arms  # noqa: E402

GRID = dict(seed=0, state_space_type="grid", grid_shape=(8, 8), target_point=[5, 5],
            delay=0, sequence_length=1, reward_function="move_to_a_point",
            make_denser=True, transition_noise=0.25, reward_noise=1.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    for label, N, T in (("64k", 65536, 1000), ("N1", 1 << 20, 100)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            env = VectorRLToyEnv(N, autoreset=True, horizon=100, **GRID)
        ag = GridQLearner(env, alpha=0.1, gamma=0.99, epsilon=0.1)
        acts = ag.learn(T, record=True)["actions"]  # the rows the learner takes
        out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
        ms = time_arms({
            "learn": lambda: ag.learn(T),
            "learn_record": lambda: ag.learn(T, record=True),
            "rollout": lambda: env.rollout(T, actions=acts, out=out),
        }, a.reps)
        report(label, N, T, ms)
        print(f"{label:>6} Q-tables: {ag.q.numel() * 8 / 1e6:.0f} MB", flush=True)
        del env, ag, out, acts
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
