"""numpy restatement of augmented random search as mdpp_continuous_ars /
mdpp_continuous_ars_update run it (include/mdpp_b200.h, csrc/ars.cu), in the
same operation order, so the device agrees bit for bit wherever the inputs
do (the Box-Muller normals of delta agree to libm accuracy).  TEST ONLY.

Layout: D = state_space_dim, P = D (D + 1), theta / delta [D][D + 1]
row-major; local env 2p is the + member, 2p + 1 the - member of pair p."""
import math

import numpy as np

from oracle import philox as px

STREAM_ARS_DELTA = 0x20000


def perturbations(seed, gid_plus, iteration, D):
    """delta of the pairs whose + members have global ids `gid_plus`:
    float64 [n_pairs, D, D + 1]."""
    P = D * (D + 1)
    gid_plus = np.asarray(gid_plus, dtype=np.uint32)
    out = np.zeros((gid_plus.size, 4 * ((P + 3) // 4)))
    it = int(iteration)
    for c in range((P + 3) // 4):
        w = px.philox4x32_10(gid_plus, it & 0xFFFFFFFF, (it >> 32) & 0xFFFFFFFF,
                             STREAM_ARS_DELTA + c, seed)
        out[:, 4 * c], out[:, 4 * c + 1] = px.normal_pair_f64(w[0], w[1])
        out[:, 4 * c + 2], out[:, 4 * c + 3] = px.normal_pair_f64(w[2], w[3])
    return out[:, :P].reshape(-1, D, D + 1)


def env_weights(theta, delta, noise_std):
    """[2 n_pairs, D, D + 1]: theta + (s nu) delta, s = + for local env 2p,
    - for 2p + 1; one rounded product and one rounded sum per entry."""
    nu = float(noise_std)
    plus = theta[None] + nu * delta
    minus = theta[None] + (-nu) * delta
    return np.stack([plus, minus], axis=1).reshape((-1,) + theta.shape)


def policy_actions(w, obs, real, action_space_max):
    """a_d = sum_k w[d][k] phi_k, phi = (obs as float64, 1), from the k = 0
    product upward, every product and sum rounded on its own; cast to `real`
    and clipped to the action box when it is finite.  w [N, D, D + 1], obs
    [N, D] -> [N, D] of `real`."""
    obs = np.asarray(obs).astype(np.float64)
    D = obs.shape[1]
    acc = w[:, :, 0] * obs[:, None, 0]
    for k in range(1, D):
        acc = acc + w[:, :, k] * obs[:, None, k]
    acc = acc + w[:, :, D]
    a = acc.astype(real)
    if math.isfinite(action_space_max):
        amax = real(action_space_max)
        a = np.where(a < -amax, -amax, np.where(a > amax, amax, a)).astype(real)
    return a


def update(theta, fitness, delta, top_directions, step_size):
    """One group's update, in the device's order.  theta [D, D + 1],
    fitness [2 n_pairs], delta [n_pairs, D, D + 1].  Returns (new theta,
    m, sigma_R, updated)."""
    f = np.asarray(fitness, dtype=np.float64)
    n_pairs = f.size // 2
    b = int(top_directions)
    key = np.maximum(f[0::2], f[1::2])
    kept = []
    for p in range(n_pairs):
        rank = sum(1 for q in range(n_pairs)
                   if key[q] > key[p] or (key[q] == key[p] and q < p))
        kept.append(rank < b)
    n = float(2 * b)
    s = 0.0
    for p in range(n_pairs):
        if kept[p]:
            s = (s + float(f[2 * p])) + float(f[2 * p + 1])
    m = s / n
    v = 0.0
    for p in range(n_pairs):
        if kept[p]:
            d0, d1 = float(f[2 * p]) - m, float(f[2 * p + 1]) - m
            v = (v + d0 * d0) + d1 * d1
    sigma = math.sqrt(v / n)
    if not (math.isfinite(sigma) and sigma > 0.0):
        return theta.copy(), m, sigma, False
    fac = step_size / (float(b) * sigma)
    G = np.zeros(theta.size)
    flat = delta.reshape(n_pairs, -1)
    for p in range(n_pairs):
        if kept[p]:
            G = G + (float(f[2 * p]) - float(f[2 * p + 1])) * flat[p]
    return (theta.reshape(-1) + fac * G).reshape(theta.shape), m, sigma, True


def run(oracles, thetas, iterations, steps, step_size, noise_std, seed,
        top_directions=None):
    """ARS on VectorContinuousOracle groups (one per cell, each already
    reset; global ids from oracle.gid): `iterations` times `steps` steps,
    then an update per cell.  Returns (thetas, per-iteration list of the
    mean return of the episodes that ended in an auto-reset, per cell)."""
    curve = []
    ep_ret = [np.zeros(o.N) for o in oracles]
    for it in range(iterations):
        fitness = [np.zeros(o.N) for o in oracles]
        rsum = [0.0] * len(oracles)
        rcnt = [0] * len(oracles)
        deltas = [perturbations(seed, o.gid[0::2], it, o.D) for o in oracles]
        ws = [env_weights(th, dl, noise_std) for th, dl in zip(thetas, deltas)]
        for _ in range(steps):
            for i, o in enumerate(oracles):
                a = policy_actions(ws[i], o.em, o.R, o.e.action_space_max)
                out = o.rollout(1, a[None])
                r = out["reward"][0].astype(np.float64)
                fitness[i] = fitness[i] + r
                ep_ret[i] = ep_ret[i] + r
                end = out["terminated"][0] | out["truncated"][0]
                rsum[i] += float(ep_ret[i][end].sum())
                rcnt[i] += int(end.sum())
                ep_ret[i][end] = 0.0
        curve.append([s / c if c else float("nan") for s, c in zip(rsum, rcnt)])
        n_pairs = min(o.N for o in oracles) // 2
        b = n_pairs if top_directions is None else top_directions
        thetas = [update(th, f, dl, b, step_size)[0]
                  for th, f, dl in zip(thetas, fitness, deltas)]
    return thetas, curve
