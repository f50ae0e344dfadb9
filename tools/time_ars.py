"""Times the fused ARS launch (LinearARS.learn on a continuous env) against
the continuous rollout with the same actions, and the ARS update.

    python tools/time_ars.py [--reps 10]

Workloads (move_to_a_point, dense reward, order 2, horizon 100, float32):
  D2      1 M envs x 100 steps, state_space_dim 2
  D6      1 M envs x 100 steps, state_space_dim 6 (relevant dims 0, 1)
  ddpg12  the 12 cells of tests/fixtures/ddpg_move_to_a_point_like.py as
          one grouped env, 65 536 envs per cell, 100 steps
Four arms alternated in one process after warm-up, CUDA events around
`--reps` calls of each:
  learn          LinearARS.learn(T): no [T, N] output at all
  learn_record   learn(T, record=True): obs, reward, flags and the actions
  rollout        env.rollout(T, actions=...) with the recorded actions
                 already on the device (the AOT or NVRTC kernel the env picks)
  update         LinearARS.update() (its fitness is whatever the previous
                 arms left; the update's cost does not depend on it)
Prints the card and its power limit first: a rate is only meaningful with them.
"""
import argparse
import os
import sys
import warnings

import torch

sys.path.insert(0, ".")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from mdp_playground_b200 import LinearARS, VectorRLToyEnv  # noqa: E402
from mdp_playground_b200.sweep import Sweep  # noqa: E402
from time_qlearn import card, report, time_arms  # noqa: E402


def cont(D):
    return dict(seed=0, state_space_type="continuous", action_space_type="continuous",
                state_space_dim=D, action_space_dim=D, relevant_indices=[0, 1],
                irrelevant_features=D > 2, transition_dynamics_order=2, inertia=1.0,
                time_unit=0.5, target_radius=0.05, target_point=[0.0, 0.0],
                state_space_max=10.0, action_space_max=1.0,
                reward_function="move_to_a_point", make_denser=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--cell-envs", type=int, default=65536)
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    T = 100
    fixture = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests",
                           "fixtures", "ddpg_move_to_a_point_like.py")
    for label in ("D2", "D6", "ddpg12"):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if label == "ddpg12":
                env = Sweep(fixture, envs_per_cell=a.cell_envs).env
            else:
                env = VectorRLToyEnv(a.envs, autoreset=True, horizon=100,
                                     **cont(int(label[1:])))
        ag = LinearARS(env)
        acts = ag.learn(T, record=True)["actions"]
        out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
        ms = time_arms({
            "learn": lambda: ag.learn(T),
            "learn_record": lambda: ag.learn(T, record=True),
            "rollout": lambda: env.rollout(T, actions=acts, out=out),
            "update": ag.update,
        }, a.reps)
        report(label, env.num_envs, T, {k: v for k, v in ms.items() if k != "update"})
        print(f"{label:>6} {'update':>13}: {ms['update']:9.3f} ms  "
              f"({env.n_groups} group(s), {env.num_envs // 2} pairs, "
              f"P = {ag.theta[0].numel()})", flush=True)
        del env, ag, out, acts
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
