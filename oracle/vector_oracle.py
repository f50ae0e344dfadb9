"""Batched numpy oracle for the discrete step path (TEST INFRASTRUCTURE ONLY).

N environments sharing the tables of one `ScalarRLToyEnv` (the scalar
oracle, itself pinned to the reference), stepped with the batched-API
semantics the CUDA path adds on top of the reference: same-step auto-reset,
`horizon` truncation, and noise from replayed arrays or from the Philox
streams of oracle/philox.py.  Per-env arithmetic follows
rl_toy_env.py:1602-1622 (transition), :1817-1846 + :1968-1990 (reward),
:2098-2109 (done / terminal reward), :2250-2278 (reset).  Plain Python loop
over time, numpy over environments.
"""
import numpy as np

from . import philox as px


class VectorDiscreteOracle:
    def __init__(self, scalar_env, num_envs, autoreset=False, horizon=0,
                 seed=0, env_id_offset=0, fast_normal=False, normal="ziggurat",
                 gids=None):
        e = scalar_env
        assert e.kind == "discrete"
        self.N = int(num_envs)
        self.S, self.A = int(e.state_space_size), int(e.action_space_size)
        self.L, self.d = e.sequence_length, e.delay
        self.every_n = int(e.reward_every_n_steps)
        self.P = np.array(e.transition_matrix, dtype=np.int64)
        self.term = np.zeros(self.S, dtype=bool)
        self.term[np.array(e.terminal_states, dtype=np.int64)] = True
        self.init_cdf = e.init_cdf
        self.custom = e.use_custom_mdp
        if self.custom:
            self.R = np.asarray(e.reward_matrix, dtype=np.float64)
        else:
            self.seq = {k: float(v) for k, v in e.rewardable_sequences.items()
                        if len(k) == self.L}
        self.has_pnoise = bool(e.transition_noise)
        self.noise_cdf = e.noise_cdf if self.has_pnoise else None
        self.pn_params = px.transition_noise_params(
            float(e.transition_noise) if self.has_pnoise else 0.0, self.S)
        self.has_rnoise = e.has_reward_noise and e.reward_noise_std is not None
        self.r_std = e.reward_noise_std
        self.scale, self.shift = e.reward_scale, e.reward_shift
        self.term_reward = e.term_state_reward
        # irrelevant_features (rl_toy_env.py:2062-2082, :2260-2264): a second,
        # reward-free chain; obs / actions become rows (relevant, irrelevant)
        self.irr = bool(getattr(e, "irrelevant_features", False))
        if self.irr:
            self.S1, self.A1 = int(e.state_space_size_irr), int(e.action_space_size_irr)
            self.P1 = np.array(e.transition_matrix_irr, dtype=np.int64)
            self.init_cdf1 = e.init_cdf_irr
            self.noise_cdf1 = e.noise_cdf_irr if self.has_pnoise else None
            self.pn_params1 = px.transition_noise_params(
                float(e.transition_noise) if self.has_pnoise else 0.0, self.S1)
        self.autoreset, self.horizon = autoreset, int(horizon)
        self.seed = int(seed)
        self.fast_normal = fast_normal
        # reward normals: "ziggurat" (the API default, normal_precision="fp64"),
        # "boxmuller" (fp64 Box-Muller) or fast_normal=True (fp32 SFU form)
        self.normal = None if fast_normal or normal == "boxmuller" else normal
        self.gid = (np.arange(self.N, dtype=np.int64) + env_id_offset).astype(
            np.uint32) if gids is None else np.asarray(gids).astype(np.uint32)
        assert self.gid.shape == (self.N,)
        self.step_index = 0
        self.cur = np.zeros(self.N, dtype=np.int64)
        self.cur1 = np.zeros(self.N, dtype=np.int64)
        self.t = np.zeros(self.N, dtype=np.int64)
        self.episode = np.zeros(self.N, dtype=np.int64)
        self.window = [[] for _ in range(self.N)]   # last L states
        # states since the reset, newest last, at most L + d + 1 (the window
        # of get_augmented_state)
        self.H = self.L + self.d + 1
        self.hist = [[] for _ in range(self.N)]
        self.fifo = [[0.0] * self.d for _ in range(self.N)]
        self.stats = dict(episodes=0, transitions=0, reward=0.0,
                          noisy_transitions=0, abs_reward_noise=0.0,
                          returned_reward=0.0, terminated=0)

    def load_state(self, cur, t, episode, key, ring, step_index, key_bits):
        """Adopt the per-env state of the CUDA path (the SoA arrays of
        mdp_playground_b200.VectorRLToyEnv: cur_state, t_episode, episode,
        seq_key, delay ring [d, N]) at global step `step_index`, so that a
        rollout can be checked from the middle of a long run."""
        self.step_index = int(step_index)
        self.cur = np.asarray(cur, dtype=np.int64).copy()
        self.t = np.asarray(t, dtype=np.int64).copy()
        self.episode = np.asarray(episode, dtype=np.int64).copy()
        mask = (1 << key_bits) - 1
        for i in range(self.N):
            n = min(int(self.t[i]) + 1, self.L)   # states seen since the reset
            k = int(key[i])
            self.window[i] = [(k >> (key_bits * j)) & mask for j in range(n - 1, -1, -1)]
            assert self.window[i][-1] == self.cur[i]
            # fifo[k] (oldest first) was written d - k steps ago: ring slot
            # (step - (d - k)) mod d; anything older than the reset reads 0
            self.fifo[i] = [
                float(ring[(self.step_index - (self.d - k)) % self.d][i])
                if self.d - k <= self.t[i] else 0.0 for k in range(self.d)]

    def reseed(self, seed, mask=None, rewind=False):
        """reset(seed=...) / seed() of the CUDA path: a new Philox key and
        the episode counters of the envs in `mask` (all when None) back to 0.
        `rewind` (an unmasked reset(seed=...)) also sets the global step back
        to 0; otherwise the step index carries on.  The per-env FIFO and
        window here have no phase, so they are the reference for envs that a
        reseed leaves running."""
        self.seed = int(seed) & (2**64 - 1)
        idx = np.arange(self.N) if mask is None else np.nonzero(mask)[0]
        self.episode[idx] = 0
        if rewind:
            self.step_index = 0

    def set_state(self, states):
        """set_augmented_state with bare states ([N], or [N, 2] rows with
        irrelevant_features): each env continues as from the start of an
        episode in that state; episode counters and statistics unchanged."""
        st = np.asarray(states, dtype=np.int64)
        for i in range(self.N):
            s = st[i]
            if self.irr:
                s, self.cur1[i] = int(s[0]), int(s[1])
            self.cur[i] = int(s)
            self.t[i] = 0
            self.window[i] = [int(s)]
            self.hist[i] = [int(s)]
            self.fifo[i] = [0.0] * self.d

    def augmented_state(self):
        """get_augmented_state()["augmented_state"]: [N, L + d + 1] float64,
        oldest first, NaN before the episode start."""
        out = np.full((self.N, self.H), np.nan)
        for i, h in enumerate(self.hist):
            out[i, self.H - len(h):] = h
        return out

    # -- draws -------------------------------------------------------------
    def _reset_u(self, idx):
        w = px.philox4x32_10(self.gid[idx], self.episode[idx].astype(np.uint32),
                             0, px.STREAM_RESET, self.seed)
        return px.uniform53(w[0], w[1]), px.uniform53(w[2], w[3])

    def _obs(self):
        return np.stack([self.cur, self.cur1], axis=-1) if self.irr \
            else self.cur.copy()

    def reset(self, mask=None, init_state=None, reset_u=None):
        """With irrelevant_features init_state / reset_u are [N, 2] rows."""
        idx = np.arange(self.N) if mask is None else np.nonzero(mask)[0]
        if init_state is not None:
            init = np.asarray(init_state, dtype=np.int64)[idx]
            s0, s1 = (init[:, 0], init[:, 1]) if self.irr else (init, None)
        else:
            if reset_u is None:
                u, u1 = self._reset_u(idx)
            else:
                ru = np.asarray(reset_u)[idx]
                u, u1 = (ru[:, 0], ru[:, 1]) if self.irr else (ru, None)
            s0 = np.minimum(np.searchsorted(self.init_cdf, u, side="right"),
                            self.S - 1)
            s1 = np.minimum(np.searchsorted(self.init_cdf1, u1, side="right"),
                            self.S1 - 1) if self.irr else None
        self.stats["episodes"] += int((self.t[idx] > 0).sum())
        for j, (i, s) in enumerate(zip(idx, s0)):
            self._reset_one(i, int(s))
            if self.irr:
                self.cur1[i] = int(s1[j])
        return self._obs()

    def _reset_one(self, i, s0):
        self.cur[i] = s0
        self.t[i] = 0
        self.episode[i] += 1
        self.window[i] = [s0]
        self.hist[i] = [s0]
        self.fifo[i] = [0.0] * self.d

    def rollout(self, T, actions=None, replay=None):
        N = self.N
        row = (T, N, 2) if self.irr else (T, N)
        obs = np.zeros(row, dtype=np.int64)
        final_obs = np.zeros(row, dtype=np.int64)
        reward = np.zeros((T, N), dtype=np.float64)
        term = np.zeros((T, N), dtype=bool)
        trunc = np.zeros((T, N), dtype=bool)
        for t in range(T):
            step = self.step_index + t
            a1 = None
            if actions is not None:
                a = np.asarray(actions[t], dtype=np.int64)
                if self.irr:
                    a, a1 = a[:, 0], a[:, 1]
            else:
                w = px.step_words(self.seed, self.gid, step, px.STREAM_ACTION)
                a = px.mulhi32(w[0], self.A)
                if self.irr:
                    a1 = px.mulhi32(w[1], self.A1)
            a = np.minimum(a, self.A - 1)
            if self.irr:  # the irrelevant chain: table walk + noisy redraw
                nxt1 = self.P1[self.cur1, np.minimum(a1, self.A1 - 1)]
                if self.has_pnoise and replay is None:
                    w1 = px.quad_word(self.seed, self.gid, step, px.STREAM_IRR_STEP)
                    nxt1 = px.noisy_next_state(w1, nxt1, self.pn_params1)
                elif self.has_pnoise:
                    u1 = np.asarray(replay["irr_transition_u"][t])
                    nxt1 = np.array([
                        min(int(np.searchsorted(self.noise_cdf1[nxt1[i]], u1[i],
                                                side="right")), self.S1 - 1)
                        for i in range(N)], dtype=np.int64)
                self.cur1 = nxt1.astype(np.int64)
            u_tr = n_rw = None
            if replay is not None:
                if self.has_pnoise:
                    u_tr = np.asarray(replay["transition_u"][t])
                if self.has_rnoise:
                    n_rw = np.asarray(replay["reward_noise"][t])
            elif self.has_pnoise or self.has_rnoise:
                u_tr, z = px.step_noise(self.seed, self.gid, step,
                                        want_normal=self.has_rnoise,
                                        fast=self.fast_normal, raw=True,
                                        normal=self.normal)
                if self.has_rnoise:
                    n_rw = self.r_std * z
            nxt = self.P[self.cur, a]
            if self.has_pnoise and replay is None:
                noisy = px.noisy_next_state(u_tr, nxt, self.pn_params)
                self.stats["noisy_transitions"] += int((noisy != nxt).sum())
                nxt = noisy
            elif self.has_pnoise:
                noisy = np.array([
                    min(int(np.searchsorted(self.noise_cdf[nxt[i]], u_tr[i],
                                            side="right")), self.S - 1)
                    for i in range(N)], dtype=np.int64)
                self.stats["noisy_transitions"] += int((noisy != nxt).sum())
                nxt = noisy
            for i in range(N):
                s_prev = int(self.cur[i])
                win = self.window[i]
                win.append(int(nxt[i]))
                if len(win) > self.L:
                    del win[0]
                self.t[i] += 1
                ti = int(self.t[i])
                if self.custom:
                    r = float(self.R[s_prev, a[i]])
                elif ti >= self.L:
                    r = self.seq.get(tuple(win), 0.0)
                else:
                    r = 0.0
                fifo = self.fifo[i]
                fifo.append(r)
                r = fifo.pop(0)
                if ti % self.every_n != 0:
                    r = 0.0
                self.stats["reward"] += r
                if self.has_rnoise:
                    self.stats["abs_reward_noise"] += abs(float(n_rw[i]))
                    r = r + float(n_rw[i])
                r = r * self.scale
                r = r + self.shift
                done = bool(self.term[nxt[i]])
                if done:
                    r = r + self.term_reward * self.scale
                tr = self.horizon > 0 and ti >= self.horizon
                reward[t, i], term[t, i], trunc[t, i] = r, done, tr
                final_obs[t, i] = (nxt[i], self.cur1[i]) if self.irr else nxt[i]
                self.cur[i] = nxt[i]
                self.stats["returned_reward"] += r
                self.stats["terminated"] += int(done)
                self.stats["transitions"] += 1
                if self.autoreset and (done or tr):
                    if replay is not None:
                        u = float(replay["reset_u"][t][i])
                    else:
                        u = float(px.autoreset_uniform(
                            self.seed, self.gid[i:i + 1], step)[0])
                    s0 = min(int(np.searchsorted(self.init_cdf, u,
                                                 side="right")), self.S - 1)
                    self._reset_one(i, s0)
                    self.stats["episodes"] += 1
                    if self.irr:
                        if replay is not None:
                            u1 = float(replay["irr_reset_u"][t][i])
                        else:
                            u1 = float(px.uniform32(px.quad_word(
                                self.seed, self.gid[i:i + 1], step,
                                px.STREAM_IRR_AUTORESET))[0])
                        self.cur1[i] = min(int(np.searchsorted(
                            self.init_cdf1, u1, side="right")), self.S1 - 1)
                obs[t, i] = (self.cur[i], self.cur1[i]) if self.irr else self.cur[i]
                if not (self.autoreset and (done or tr)):
                    self.hist[i] = (self.hist[i] + [int(self.cur[i])])[-self.H:]
        self.step_index += T
        return dict(obs=obs, final_obs=final_obs, reward=reward,
                    terminated=term, truncated=trunc)


class VectorGroupedOracle:
    """A heterogeneous launch (BASELINE config #5): envs laid out group-major,
    group g = `sizes[g]` envs with the tables of `scalar_envs[g]`; global Philox
    ids follow mdp_playground_b200/sharding.py (every group's envs contiguous
    over ranks, groups one after the other).  One VectorDiscreteOracle per
    group, outputs concatenated along the env axis."""

    def __init__(self, scalar_envs, sizes, autoreset=False, horizon=0, seed=0,
                 env_id_offset=0, rank=0, world=1, **kw):
        assert len(scalar_envs) == len(sizes)
        self.sizes = [int(n) for n in sizes]
        self.parts, gbegin = [], 0
        for e, n in zip(scalar_envs, self.sizes):
            gids = env_id_offset + gbegin + rank * n + np.arange(n, dtype=np.int64)
            gbegin += world * n
            self.parts.append(VectorDiscreteOracle(
                e, n, autoreset=autoreset, horizon=horizon, seed=seed, gids=gids, **kw))

    def _split(self, x):
        """Per-group slices of an env-major array (None stays None)."""
        if x is None:
            return [None] * len(self.parts)
        x, begin, out = np.asarray(x), 0, []
        for n in self.sizes:
            out.append(x[begin:begin + n])
            begin += n
        return out

    def reset(self, mask=None, init_state=None):
        return np.concatenate([
            p.reset(mask=m, init_state=s) for p, m, s in
            zip(self.parts, self._split(mask), self._split(init_state))])

    def reseed(self, seed, mask=None, rewind=False):
        for p, m in zip(self.parts, self._split(mask)):
            p.reseed(seed, mask=m, rewind=rewind)

    def rollout(self, T, actions=None):
        outs, begin = [], 0
        for p, n in zip(self.parts, self.sizes):
            a = None if actions is None else np.asarray(actions)[:, begin:begin + n]
            outs.append(p.rollout(T, actions=a))
            begin += n
        return {k: np.concatenate([o[k] for o in outs], axis=1) for k in outs[0]}

    @property
    def stats(self):
        return [dict(p.stats) for p in self.parts]
