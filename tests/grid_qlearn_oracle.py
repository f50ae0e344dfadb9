"""numpy restatement of the fused grid Q-learning launch (mdpp_grid_qlearn,
mdp_playground_b200/qlearning.py).  TEST INFRASTRUCTURE.

Built on the batched grid oracle of oracle/vector_grid_oracle.py: every step
draws the learner's STREAM_GRID_ACTION words, picks the epsilon-greedy action
index, and hands its action row to the oracle's own `rollout` for one step;
the float64 update follows in the kernel's order (each numpy float64
operation rounds on its own, as the kernel's _rn intrinsics do).
"""
import numpy as np

from oracle import philox as px
from oracle.vector_grid_oracle import VectorGroupedGridOracle
from tests.qlearn_oracle import new_accumulators

STREAM_GRID_ACTION = 45


def action_rows(nd):
    """Action index -> row: 0 = no-op, 1 + 2k = -1 on dim k, 2 + 2k = +1."""
    rows = [[0] * nd]
    for k in range(nd):
        for v in (-1, 1):
            r = [0] * nd
            r[k] = v
            rows.append(r)
    return np.array(rows, dtype=np.int64)


def cell_index(pos, shape):
    """Row-major index of cells [..., nd] over [0, shape_k]."""
    pos = np.asarray(pos, dtype=np.int64)
    s = pos[..., 0]
    for k in range(1, len(shape)):
        s = s * (int(shape[k]) + 1) + pos[..., k]
    return s


def n_cells(shape):
    return int(np.prod([int(n) + 1 for n in shape]))


def _qlearn_part(ora, T, alpha, gamma, epsilon, q, acc):
    """T steps of one VectorGridOracle; q [N, S_max, A_max] and the
    accumulators (views into the caller's arrays) are updated in place."""
    N, nd = ora.N, ora.nd
    A = 2 * nd + 1
    rows_of = action_rows(nd)
    rows = np.arange(N)
    thr = epsilon * 4294967296.0
    keys = ("obs", "final_obs", "reward", "terminated", "truncated")
    out = {k: [] for k in keys}
    out["actions"], out["action_index"], out["state"] = [], [], []
    for _ in range(T):
        step = ora.step_index
        w = px.step_words(ora.seed, ora.gid, step >> 1, STREAM_GRID_ACTION)
        w_explore, w_action = (w[2], w[3]) if step & 1 else (w[0], w[1])
        explore = w_explore.astype(np.float64) < thr
        a_rand = px.mulhi32(w_action, A)
        s = cell_index(ora.pos, ora.shape)
        a = np.where(explore, a_rand, np.argmax(q[rows, s, :A], axis=1))
        o = ora.rollout(1, actions=rows_of[a][None])
        r = o["reward"][0]
        nxt = cell_index(o["final_obs"][0], ora.shape)
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
        out["actions"].append(rows_of[a])
        out["action_index"].append(a)
        out["state"].append(s)
    return {k: np.stack(v) for k, v in out.items()}


def qlearn(oracle, T, alpha, gamma, epsilon, q, acc=None):
    """T steps of epsilon-greedy tabular Q-learning on a VectorGridOracle or
    a VectorGroupedGridOracle.  q: float64 [N, S_max, A_max], updated in
    place; acc: the episode-return accumulators (new_accumulators(N)),
    updated in place.  Returns the [T, N] outputs of a rollout plus the
    action rows ("actions", [T, N, nd]), their indices ("action_index") and
    the cell index each step started from ("state"), and the accumulators."""
    parts = oracle.parts if isinstance(oracle, VectorGroupedGridOracle) else [oracle]
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
