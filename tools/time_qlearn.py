"""Times the fused tabular Q-learning launch (TabularQLearner.learn) against
the random-policy rollout of the same env.

    python tools/time_qlearn.py [--envs 65536] [--steps 1000] [--reps 10]

BASELINE configs #1 and #2 at `--envs` envs x `--steps` steps per launch,
three arms alternated in one process after warm-up, CUDA events around
`--reps` launches of each:
  learn          TabularQLearner.learn(T): no [T, N] output at all
  learn_record   learn(T, record=True): obs, reward, flags and actions
  rollout        env.rollout(T, actions=None): the device random policy
and a 1000-cell grouped learn / rollout pair (BASELINE config #5 shape, 1 M
envs).  At 65 536 envs of 8 x 8 the Q-tables are 32 MB and stay in L2; at
1 M envs they are 512 MB and do not.  Prints the card and its power limit
first: a rate is only meaningful with them.
"""
import argparse
import subprocess
import sys
import warnings

import torch

sys.path.insert(0, ".")
from mdp_playground_b200 import TabularQLearner, VectorRLToyEnv  # noqa: E402

BASE = dict(seed=0, state_space_type="discrete", action_space_type="discrete",
            state_space_size=8, reward_density=0.25, terminal_state_density=0.25)
CONFIGS = {
    "#1": dict(BASE, action_space_size=5, sequence_length=1, delay=0),
    "#2": dict(BASE, action_space_size=8, sequence_length=3, delay=2,
               transition_noise=0.1, reward_noise=0.25, reward_every_n_steps=True),
}
C5 = [dict(BASE, action_space_size=8, delay=d, sequence_length=L,
           transition_noise=pn, reward_noise=rn, make_denser=md,
           reward_every_n_steps=True)
      for d in (0, 1, 2, 4, 8) for L in (1, 2, 3, 4)
      for pn in (0, 0.01, 0.02, 0.1, 0.25) for rn in (0, 1, 5, 10, 25)
      for md in (False, True)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return torch.cuda.get_device_name()


def time_arms(arms, reps, rounds=3):
    """ms per launch of each arm: `rounds` rounds of `reps` launches per arm,
    arms alternated, the minimum over rounds."""
    for fn in arms.values():  # warm-up (module load, smem opt-in)
        fn()
        fn()
    torch.cuda.synchronize()
    best = {k: float("inf") for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            best[k] = min(best[k], e0.elapsed_time(e1) / reps)
    return best


def report(label, N, T, ms):
    base = ms.get("rollout")
    for k, v in ms.items():
        rate = N * T / v * 1e3
        rel = f"  {v / base:.2f}x rollout time" if base and k != "rollout" else ""
        print(f"{label:>6} {k:>13}: {v:9.3f} ms  {rate:.3e} env-steps/s{rel}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--c5-envs", type=int, default=1 << 20)
    ap.add_argument("--c5-steps", type=int, default=100)
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    N, T = a.envs, a.steps
    for name, cfg in CONFIGS.items():
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            env = VectorRLToyEnv(N, autoreset=True, horizon=100, **cfg)
        ag = TabularQLearner(env, alpha=0.1, gamma=0.99, epsilon=0.1)
        out = env._alloc_out(T, env._obs_torch_dtype(), final_obs=False)
        ms = time_arms({
            "learn": lambda: ag.learn(T),
            "learn_record": lambda: ag.learn(T, record=True),
            "rollout": lambda: env.rollout(T, out=out),
        }, a.reps)
        report(name, N, T, ms)
        del env, ag, out
        torch.cuda.empty_cache()
    N5, T5 = a.c5_envs, a.c5_steps
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        env = VectorRLToyEnv(N5, autoreset=True, horizon=100, config_groups=C5)
    ag = TabularQLearner(env, alpha=0.1, gamma=0.99, epsilon=0.1)
    out = env._alloc_out(T5, env._obs_torch_dtype(), final_obs=False)
    ms = time_arms({"learn": lambda: ag.learn(T5),
                    "rollout": lambda: env.rollout(T5, out=out)}, a.reps)
    report("#5", N5, T5, ms)


if __name__ == "__main__":
    main()
