"""numpy restatement of the evaluation launches (mdpp_discrete_qeval,
mdpp_grid_qeval, mdpp_continuous_ars_eval; the learners' evaluate()).
TEST INFRASTRUCTURE.

Built on the batched oracles: every step acts with the fixed policy (the
greedy action of q, or theta [obs; 1]) and hands the actions to the oracle's
own `rollout` for one step.  Of each env the first E episodes (an episode
ends on terminated or truncated) add their return and length.
`first_episodes` is the same bookkeeping as a plain per-env loop.
"""
import numpy as np

from tests import ars_oracle as ao
from tests import grid_qlearn_oracle as go


def parts_of(oracle):
    return list(getattr(oracle, "parts", [oracle]))


def _greedy_discrete(q, rows):
    def act(p, sl):
        return np.argmax(q[sl][rows[sl], p.cur, :p.A], axis=1)
    return act


def _greedy_grid(q, rows):
    def act(p, sl):
        A = 2 * p.nd + 1
        s = go.cell_index(p.pos, p.shape)
        return go.action_rows(p.nd)[np.argmax(q[sl][rows[sl], s, :A], axis=1)]
    return act


def _theta_policy(thetas):
    def act(p, sl, g):
        w = np.broadcast_to(thetas[g], (p.N,) + thetas[g].shape)
        return ao.policy_actions(w, p.em, p.R, p.e.action_space_max)
    return act


def evaluate(oracle, kind, policy, episodes, horizon):
    """E = episodes evaluation episodes of every env of a (grouped) batched
    oracle that the caller has reset.  kind: "discrete" / "grid" (policy: q
    [N, S_max, A_max]) or "continuous" (policy: theta [G, D, D + 1]).  Runs
    E * horizon steps; returns per env "ret_sum", "ret_count", "len_sum" and
    the [T, N] "reward" / "ended" / "actions" records."""
    parts = parts_of(oracle)
    N = sum(p.N for p in parts)
    rows = np.arange(N) - np.repeat(np.cumsum([0] + [p.N for p in parts])[:-1],
                                    [p.N for p in parts])
    T = int(episodes) * int(horizon)
    ret = np.zeros(N)
    ret_sum = np.zeros(N)
    length = np.zeros(N, dtype=np.int64)
    len_sum = np.zeros(N, dtype=np.int64)
    count = np.zeros(N, dtype=np.int64)
    rec = {"reward": [], "ended": [], "actions": []}
    for _ in range(T):
        rw, en, acts, begin = [], [], [], 0
        for g, p in enumerate(parts):
            sl = slice(begin, begin + p.N)
            if kind == "discrete":
                a = _greedy_discrete(policy, rows)(p, sl)
            elif kind == "grid":
                a = _greedy_grid(policy, rows)(p, sl)
            else:
                a = _theta_policy(policy)(p, sl, g)
            o = p.rollout(1, a[None])
            rw.append(np.asarray(o["reward"][0], dtype=np.float64))
            en.append(o["terminated"][0] | o["truncated"][0])
            acts.append(a)
            begin += p.N
        r, ended = np.concatenate(rw), np.concatenate(en)
        live = count < episodes
        ret = np.where(live, ret + r, ret)
        length = np.where(live, length + 1, length)
        fin = live & ended
        ret_sum[fin] = ret_sum[fin] + ret[fin]
        len_sum[fin] += length[fin]
        count[fin] += 1
        ret[fin] = 0.0
        length[fin] = 0
        rec["reward"].append(r)
        rec["ended"].append(ended)
        rec["actions"].append(np.concatenate(acts))
    out = {k: np.stack(v) for k, v in rec.items()}
    out.update(ret_sum=ret_sum, ret_count=count, len_sum=len_sum)
    return out


def first_episodes(reward, ended, episodes):
    """Per env of [T, N] rewards and episode ends: (return sum, count, length
    sum) of its first `episodes` episodes, summed in step order."""
    reward, ended = np.asarray(reward, dtype=np.float64), np.asarray(ended, dtype=bool)
    T, N = reward.shape
    ret_sum = np.zeros(N)
    count = np.zeros(N, dtype=np.int64)
    len_sum = np.zeros(N, dtype=np.int64)
    for i in range(N):
        ret, length = 0.0, 0
        for t in range(T):
            if count[i] == episodes:
                break
            ret += float(reward[t, i])
            length += 1
            if ended[t, i]:
                ret_sum[i] += ret
                len_sum[i] += length
                count[i] += 1
                ret, length = 0.0, 0
    return ret_sum, count, len_sum
