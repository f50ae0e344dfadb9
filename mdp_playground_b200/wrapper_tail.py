"""VectorGymEnvTail: GymEnvWrapper's post-processing for N external envs.

The reference's `GymEnvWrapper` (envs/gym_env_wrapper.py) injects MDP
Playground's dimensions into ANY gym environment: around `env.step` it
replaces the action with probability `transition_noise` (discrete) or adds
N(0, sigma) noise to the observation (continuous) (:353-376, :405-406), delays
rewards through a FIFO that is flushed at episode end (:411-424), adds reward
noise, scale and shift (:430-436), and pastes image observations into a padded
canvas at a random quantised shift (:523-618).  This class is that tail for a
batch of environments stepped elsewhere (an external vector env), as three
calls into libmdpp_b200.so:

    tail = VectorGymEnvTail(N, n_actions=18, state_space_type="discrete",
                            delay=2, transition_noise=0.1, reward_noise=0.5)
    a = tail.actions(a)                       # before the external step
    obs, r, done = external_env.step(a)       # (not ours)
    obs, r = tail.post(obs, r, done)          # after it

Config keys and defaults are the wrapper's.  Noise is Philox (default) or
replayed (`noise="replay"`: the caller passes the draws -- how the reference's
golden vectors are replayed bit for bit).  Terminal steps: the reference
raises TypeError at HEAD (:414); see include/mdpp_b200.h for what is computed.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import _ptr


class VectorGymEnvTail:
    def __init__(self, num_envs, device=None, noise="philox", seed=0,
                 env_id_offset=0, n_actions=None, obs_dim=None,
                 obs_dtype=torch.float32, image_side=None, normal_precision="fp64",
                 **config):
        if not torch.cuda.is_available():
            raise RuntimeError("VectorGymEnvTail needs a CUDA device: there is "
                               "no CPU fallback")
        assert noise in ("philox", "replay")
        # native noise normals: fp64 Box-Muller (default) or fp32 on the SFU
        assert normal_precision in ("fp64", "fast")
        self._normal_mode = _lib.MDPP_NORMAL_FAST if normal_precision == "fast" \
            else _lib.MDPP_NORMAL_F64
        self._lib = _lib.load()
        self.num_envs, self.noise = int(num_envs), noise
        self.device = torch.device("cuda", torch.cuda.current_device()) \
            if device is None else torch.device(device)
        self.seed, self.env_id_offset = int(seed) & (2**64 - 1), int(env_id_offset)
        self._step_index = 0
        c = _lib.TailConfig()
        kind = config["state_space_type"]
        assert kind in ("discrete", "continuous")
        c.discrete = int(kind == "discrete")
        c.n_actions = int(n_actions or 0)
        c.obs_dim = int(obs_dim or 0)
        c.obs_is_f64 = int(obs_dtype == torch.float64)
        self._obs_dtype = obs_dtype
        c.delay = int(config.get("delay", 0))
        assert c.delay >= 0
        pn = config.get("transition_noise", None)
        if callable(pn) or callable(config.get("reward_noise", None)):
            raise NotImplementedError("callable noise cannot run on the device")
        c.has_transition_noise = int(bool(pn))
        c.transition_noise = float(pn or 0.0)
        if c.discrete and pn is not None:
            assert 0.0 <= pn <= 1.0, (
                "transition_noise must be a value in [0.0, 1.0] when env is "
                "discrete, it was:" + str(pn))
        c.has_reward_noise = int("reward_noise" in config)
        c.reward_noise_std = float(config.get("reward_noise", 0.0) or 0.0)
        c.reward_scale = float(config.get("reward_scale", 1.0))
        c.reward_shift = float(config.get("reward_shift", 0.0))
        c.term_state_reward = float(config.get("term_state_reward", 0.0))
        tr = config.get("image_transforms", False)
        self.image_transforms = tr
        if tr:
            assert kind == "discrete", (
                "Image transforms are only supported for discrete envs with "
                "image observations.")
            c.image_side, c.image_channels = int(image_side), 3
            c.image_padding = int(config.get("image_padding", 20))
            c.has_shift = int("shift" in tr)
            c.sh_quant = int(config.get("image_sh_quant", 1) or 1)
        self._cfg = c
        self._ctx = C.c_void_p()
        _lib.check(self._lib, None,
                   self._lib.mdpp_create(self.device.index, C.byref(self._ctx)))
        N, dev = self.num_envs, self.device
        self._ring = torch.zeros((max(c.delay, 1), N), dtype=torch.float64, device=dev)
        self._t = torch.zeros(N, dtype=torch.int32, device=dev)
        st = _lib.TailState()
        st.n_envs, st.ring, st.t_episode = N, _ptr(self._ring), _ptr(self._t)
        self._state = st

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.mdpp_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _opts(self):
        o = _lib.StepOpts()
        o.n_steps = 1
        o.noise_mode = _lib.MDPP_NOISE_REPLAY if self.noise == "replay" \
            else _lib.MDPP_NOISE_PHILOX
        o.seed, o.step_index = self.seed, self._step_index
        o.env_id_offset = self.env_id_offset
        o.normal_mode = self._normal_mode
        return o

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        _lib.check(self._lib, self._ctx, rc)

    def reset(self, mask=None):
        """The wrapper's reset(): a fresh reward FIFO for the masked envs (:466)."""
        if mask is None:
            self._t.zero_()
        else:
            self._t.masked_fill_(torch.as_tensor(mask, device=self.device).bool(), 0)

    def actions(self, actions, replay_u=None):
        """:353-366.  Continuous envs: actions pass through."""
        if not self._cfg.discrete:
            return actions
        a = torch.as_tensor(actions, device=self.device).to(torch.int32).contiguous()
        out = torch.empty_like(a)
        u = None if replay_u is None else torch.as_tensor(
            np.nan_to_num(np.asarray(replay_u, dtype=np.float64)), device=self.device)
        self._keep = (a, u)
        self._check(self._lib.mdpp_tail_actions(
            self._ctx, C.byref(self._cfg), _ptr(a), _ptr(out), _ptr(u),
            self.num_envs, C.byref(self._opts()), self._stream()))
        return out

    def post(self, obs, reward, done, replay_reward_noise=None,
             replay_obs_noise=None, replay_shift=None):
        """(obs', reward') after the external step; advances the step index."""
        dev, N, c = self.device, self.num_envs, self._cfg
        r = torch.as_tensor(reward, device=dev).to(torch.float64).contiguous()
        d = torch.as_tensor(done, device=dev).to(torch.uint8).contiguous()
        out_r = torch.empty(N, dtype=torch.float64, device=dev)
        o_in = o_out = None
        if not c.discrete:
            o_in = torch.as_tensor(obs, device=dev).to(self._obs_dtype).contiguous()
            assert o_in.shape == (N, c.obs_dim)
            o_out = torch.empty_like(o_in)

        def rep(x):
            return None if x is None else torch.as_tensor(
                np.nan_to_num(np.asarray(x, dtype=np.float64)), device=dev).contiguous()
        rn, on = rep(replay_reward_noise), rep(replay_obs_noise)
        self._check(self._lib.mdpp_tail_post(
            self._ctx, C.byref(c), C.byref(self._state), _ptr(o_in), _ptr(o_out),
            _ptr(r), _ptr(d), _ptr(out_r), _ptr(rn), _ptr(on),
            C.byref(self._opts()), self._stream()))
        if self.image_transforms:
            o_out = self.shift_images(obs, replay_shift)
        elif c.discrete:
            o_out = obs
        self._step_index += 1
        return o_out, out_r

    def shift_images(self, images, replay_shift=None):
        """:523-618: uint8 [N, side, side, 3] -> [N, side + 2 pad, side + 2 pad, 3]."""
        dev, N, c = self.device, self.num_envs, self._cfg
        img = torch.as_tensor(images, device=dev).to(torch.uint8).contiguous()
        assert img.shape == (N, c.image_side, c.image_side, 3), tuple(img.shape)
        tot = c.image_side + 2 * c.image_padding
        out = torch.empty((N, tot, tot, 3), dtype=torch.uint8, device=dev)
        sh = None if replay_shift is None else torch.as_tensor(
            np.asarray(replay_shift), device=dev).to(torch.int32).contiguous()
        self.last_shift = torch.empty((N, 2), dtype=torch.int32, device=dev)
        self._check(self._lib.mdpp_tail_image_shift(
            self._ctx, C.byref(c), _ptr(img), _ptr(out), _ptr(sh),
            _ptr(self.last_shift), N, C.byref(self._opts()), self._stream()))
        return out
