"""numpy restatement of the fused tabular Q-learning launch
(mdpp_discrete_qlearn, mdp_playground_b200/qlearning.py).  TEST INFRASTRUCTURE.

Built on the batched oracle of oracle/vector_oracle.py: every step draws the
random policy's STREAM_ACTION word (px.step_words), picks the epsilon-greedy
action, and hands it to the oracle's own `rollout` for one step; the float64
update follows in the kernel's order (each numpy float64 operation rounds on
its own, as the kernel's _rn intrinsics do).
"""
import numpy as np

from oracle import philox as px
from oracle.vector_oracle import VectorGroupedOracle


def new_accumulators(n):
    return {"ep_return": np.zeros(n), "ret_sum": np.zeros(n),
            "ret_count": np.zeros(n, dtype=np.int64)}


def _qlearn_part(ora, T, alpha, gamma, epsilon, q, acc):
    """T steps of one VectorDiscreteOracle; q [N, S_max, A_max] and the
    accumulators (views into the caller's arrays) are updated in place."""
    N, A = ora.N, ora.A
    rows = np.arange(N)
    thr = epsilon * 4294967296.0
    keys = ("obs", "final_obs", "reward", "terminated", "truncated")
    out = {k: [] for k in keys}
    out["actions"] = []
    for _ in range(T):
        w = px.step_words(ora.seed, ora.gid, ora.step_index, px.STREAM_ACTION)
        a_rand = px.mulhi32(w[0], A).astype(np.int64)
        explore = w[2].astype(np.float64) < thr
        s = ora.cur.copy()
        a = np.where(explore, a_rand, np.argmax(q[rows, s, :A], axis=1))
        o = ora.rollout(1, actions=a[None, :])
        r, nxt = o["reward"][0], o["final_obs"][0]
        done, trunc = o["terminated"][0], o["truncated"][0]
        q_next = q[rows, nxt, :A]
        m = q_next[rows, np.argmax(q_next, axis=1)]
        target = np.where(done, r, r + gamma * m)
        q_sa = q[rows, s, a]
        q[rows, s, a] = q_sa + alpha * (target - q_sa)
        acc["ep_return"][:] = acc["ep_return"] + r
        ended = (done | trunc) if ora.autoreset else np.zeros(N, dtype=bool)
        acc["ret_sum"][ended] = acc["ret_sum"][ended] + acc["ep_return"][ended]
        acc["ret_count"][ended] += 1
        acc["ep_return"][ended] = 0.0
        for k in keys:
            out[k].append(o[k][0])
        out["actions"].append(a)
    return {k: np.stack(v) for k, v in out.items()}


def qlearn(oracle, T, alpha, gamma, epsilon, q, acc=None):
    """T steps of epsilon-greedy tabular Q-learning on a VectorDiscreteOracle
    or a VectorGroupedOracle.  q: float64 [N, S_max, A_max], updated in
    place; acc: the episode-return accumulators (new_accumulators(N)),
    updated in place.  Returns the [T, N] outputs of a rollout plus the
    actions taken, and the accumulators under their names."""
    parts = oracle.parts if isinstance(oracle, VectorGroupedOracle) else [oracle]
    N = sum(p.N for p in parts)
    acc = new_accumulators(N) if acc is None else acc
    outs, begin = [], 0
    for p in parts:
        sl = slice(begin, begin + p.N)
        outs.append(_qlearn_part(p, T, alpha, gamma, epsilon, q[sl],
                                 {k: v[sl] for k, v in acc.items()}))
        begin += p.N
    res = {k: np.concatenate([o[k] for o in outs], axis=1) for k in outs[0]}
    res.update(acc)
    return res
