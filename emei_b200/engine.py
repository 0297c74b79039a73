"""Device-buffer owners behind the env classes: they hold the state tensors, build the POD
parameter structs and issue the C-ABI calls.  No arithmetic happens in Python.

HBM layout (DESIGN.md section 3):
  cart-pole / IP : state  [B,4] row-major (one 128-bit row per env), ping-pong pair of buffers;
                   IP keeps a separate obs buffer (theta wrapped) because the reference wraps only
                   the observation copy (inverted_pendulum.py:45-49).
  charged ball   : on_circle uint8[B], circle [B,2], free [B,4] (= observation), updated in place.
  outputs        : reward [B,1] (engine dtype), done uint8[B,1] viewed as torch.bool.
"""
import ctypes
import gc
import os
from typing import Optional

import numpy as np
import torch

from . import _lib

_ACTION_KIND = {
    torch.uint8: _lib.ACTION_DISCRETE_U8,
    torch.bool: _lib.ACTION_DISCRETE_U8,
    torch.int32: _lib.ACTION_DISCRETE_I32,
    torch.int64: _lib.ACTION_DISCRETE_I64,
    torch.float32: _lib.ACTION_CONTINUOUS_F32,
    torch.float64: _lib.ACTION_CONTINUOUS_F64,
}


def normalise_action(env, action, continuous: bool) -> torch.Tensor:
    """-> contiguous device tensor [num_envs] in one of the encodings of include/emei_b200.h.
    Mirrors base_control.py:62-66 (int -> array; action_space.contains) for a batch."""
    n = env.num_envs
    if isinstance(action, (int, np.integer)) and not continuous:
        action = torch.full((n,), int(action), dtype=torch.int64)
    a, _ = env._to_device(action)
    if a.numel() != n:
        raise AssertionError(f"{action!r} ({type(action)}) invalid: expected {n} actions, got shape {tuple(a.shape)}")
    a = a.reshape(n)
    if continuous:
        if a.dtype not in (torch.float32, torch.float64):
            a = a.to(torch.float32)
    else:
        if a.dtype.is_floating_point:
            raise AssertionError(f"{action!r} ({type(action)}) invalid: discrete action space needs integers")
        if a.dtype not in _ACTION_KIND:
            a = a.to(torch.int64)
    if env.validate_actions:  # device-side range check: one sync, off by default
        if continuous:
            lo, hi = float(env.action_space.low.min()), float(env.action_space.high.max())
            ok = bool(((a >= lo) & (a <= hi)).all())
        else:
            ok = bool(((a >= 0) & (a < env.action_space.n)).all())
        assert ok, f"{action!r} ({type(action)}) invalid"
    return a.contiguous()


class StepOutputs:
    """Ping-pong reward / done buffers of the zero-copy mode (``copy_outputs=False``): what step t returns stays valid
    until step t+2 overwrites it (the charged ball's observation is the live ``free`` array: valid until step t+1).
    The default ``copy_outputs=True`` returns fresh tensors instead, like the reference's ``state.copy()``."""

    def __init__(self, n, dtype, device):
        self.reward = [torch.empty((n, 1), dtype=dtype, device=device) for _ in range(2)]
        self.done = [torch.empty((n, 1), dtype=torch.uint8, device=device) for _ in range(2)]


class RolloutMixin:
    """Episode bookkeeping buffers + the call of a fused T-step rollout entry point.

    float32 without state noise: the packed kernels (emei_cartpole_rollout_f32 / emei_charged_ball_rollout_f32).
    float64 (reference-exact), the inverted double pendulum and obs_noise_params: the reference-arithmetic kernels
    (emei_cartpole_rollout_ref_* / emei_i2p_rollout_* / emei_charged_ball_rollout_ref_f64), one env per thread, the
    step entry points' own device functions -- records, rewards and episode returns then have the engine dtype."""

    ep_step = ep_return = ep_index = None
    t_global = 0
    obs_dim = 4

    def _alloc_episode(self):
        if self.ep_step is None:
            dev = self.env.device
            self.ep_step = torch.zeros(self.n, dtype=torch.int32, device=dev)
            self.ep_return = torch.zeros(self.n, dtype=torch.float32, device=dev)
            self.ep_index = torch.zeros(self.n, dtype=torch.int32, device=dev)
            self.t_global = 0

    def new_episodes(self, reseed: bool):
        """called when the env's state is (re)set from outside: every env starts a fresh episode."""
        if self.ep_step is not None:
            self.ep_step.zero_()
            self.ep_return.zero_()
            if reseed:
                self.ep_index.zero_()
                self.t_global = 0

    def _rollout(self, entry: str, state_ptrs, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor,
                 ref: bool = False, extra=()):
        """entry: C-ABI symbol (with the precision suffix); ref: a reference-arithmetic entry point (records, rewards
        and episode returns in the engine dtype); extra: its trailing arguments before the stream (noise / init tables)."""
        env = self.env
        if env.dtype != torch.float32 and not ref:
            raise NotImplementedError("the packed rollout kernels are float32")
        self._alloc_episode()
        rdt = env.dtype if ref else torch.float32
        if self.ep_return.dtype != rdt:  # the running return follows the kernel's real type
            self.ep_return = self.ep_return.to(rdt)
        T, n, dev, D = int(rp.horizon), self.n, env.device, self.obs_dim
        rp.t0 = self.t_global
        rec = {}
        if actions is not None:
            if tuple(actions.shape[:2]) != (T, n) and tuple(actions.shape) != (T, n):
                raise ValueError(f"actions must be [horizon={T}, num_envs={n}], got {tuple(actions.shape)}")
            actions = actions.reshape(T, n).contiguous()
            self.params.action_kind = _ACTION_KIND[actions.dtype]
            act_dtype = actions.dtype
        else:
            cont = len(env.action_space.shape) > 0
            act_dtype = torch.float32 if cont else torch.uint8
            self.params.action_kind = _ACTION_KIND[act_dtype]
        ptrs = [None] * 6
        if record:
            rec = dict(
                observations=torch.empty((T, n, D), dtype=rdt, device=dev),
                next_observations=torch.empty((T, n, D), dtype=rdt, device=dev),
                actions=torch.empty((T, n), dtype=act_dtype, device=dev),
                rewards=torch.empty((T, n), dtype=rdt, device=dev),
                dones=torch.empty((T, n), dtype=torch.uint8, device=dev),
                timeouts=torch.empty((T, n), dtype=torch.uint8, device=dev),
            )
            ptrs = [rec[k].data_ptr() for k in ("observations", "next_observations", "actions", "rewards", "dones", "timeouts")]
        with torch.cuda.device(dev):
            _lib.call(
                entry, *state_ptrs, self.ep_step.data_ptr(), self.ep_return.data_ptr(), self.ep_index.data_ptr(),
                actions.data_ptr() if actions is not None else None, *ptrs,
                rollout_stats.data_ptr(), n, ctypes.byref(self.params), ctypes.byref(rp), *extra, env._stream(),
            )
        self.t_global += T
        if record:
            rec["dones"] = rec["dones"].view(torch.bool)
            rec["timeouts"] = rec["timeouts"].view(torch.bool)
        return rec


class CartPoleEngine(RolloutMixin):
    """cart-pole family + analytic inverted pendulum (emei_cartpole_step_*)."""

    def __init__(self, env, params: _lib.CartPoleParams, separate_obs: bool):
        self.env = env
        self.params = params
        self.separate_obs = separate_obs
        self.n = env.num_envs
        self._bufs = None
        self._obs = None
        self._out = None
        self._cur = 0
        self.has_state = False

    def _alloc(self):
        if self._bufs is None:
            dev, dt = self.env.device, self.env.dtype
            self._bufs = [torch.empty((self.n, 4), dtype=dt, device=dev) for _ in range(2)]
            if self.separate_obs:
                self._obs = [torch.empty((self.n, 4), dtype=dt, device=dev) for _ in range(2)]
            self._out = StepOutputs(self.n, dt, dev)

    @property
    def state(self) -> Optional[torch.Tensor]:
        return self._bufs[self._cur] if self.has_state else None

    def set_state(self, state):
        self._alloc()
        s, _ = self.env._to_device(state, self.env.dtype)
        if tuple(s.shape) != (self.n, 4):
            raise ValueError(f"state must have shape {(self.n, 4)}, got {tuple(s.shape)}")
        self._bufs[self._cur].copy_(s)
        self.has_state = True
        self.new_episodes(reseed=False)

    def step(self, action: torch.Tensor, copy_obs: bool, noise: Optional[_lib.NoiseParams] = None):
        env = self.env
        self._alloc()
        src, dst = self._bufs[self._cur], self._bufs[1 - self._cur]
        nxt = 1 - self._cur
        obs = None
        if self.separate_obs:
            obs = self._obs[nxt] if not copy_obs else torch.empty_like(src)
        elif copy_obs:
            obs = torch.empty_like(src)
        reward, done = self._out.reward[nxt], self._out.done[nxt]
        if copy_obs:
            reward, done = torch.empty_like(reward), torch.empty_like(done)
        self.params.action_kind = _ACTION_KIND[action.dtype]
        ptrs = (src.data_ptr(), dst.data_ptr(), obs.data_ptr() if obs is not None else None, action.data_ptr(),
                reward.data_ptr(), done.data_ptr(), env.stats.data_ptr(), self.n, ctypes.byref(self.params))
        if noise is None:
            env._call("emei_cartpole_step", *ptrs, env._stream())
        else:  # obs_noise_params (mujoco_env.py:98-104): Gaussian state noise after every sub-step
            env._call("emei_ip_step_noisy", *ptrs, ctypes.byref(noise), env._stream())
        self._cur = nxt
        return (obs if obs is not None else dst), reward, done.view(torch.bool)

    def step_range(self, lo: int, hi: int, action: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, obs_out,
                   noise: Optional[_lib.NoiseParams] = None):
        """Launch the step kernel for envs [lo, hi) only (src -> dst of the CURRENT ping-pong pair, no flip):
        the building block of the chunked host pipeline.  Call ``flip()`` once all ranges are launched.
        ``noise``: the step's NoiseParams (obs_noise_params); the range draws the streams of its own global env ids."""
        env = self.env
        self._alloc()
        src, dst = self._bufs[self._cur], self._bufs[1 - self._cur]
        if self.separate_obs and obs_out is None:
            obs_out = self._obs[1 - self._cur]
        self.params.action_kind = _ACTION_KIND[action.dtype]
        es, ea = src.element_size() * 4, action.element_size()
        ptrs = (src.data_ptr() + lo * es, dst.data_ptr() + lo * es,
                (obs_out.data_ptr() + lo * es) if obs_out is not None else None, action.data_ptr() + lo * ea,
                reward.data_ptr() + lo * reward.element_size(), done.data_ptr() + lo, env.stats.data_ptr(), hi - lo,
                ctypes.byref(self.params))
        if noise is None:
            env._call("emei_cartpole_step", *ptrs, env._stream())
        else:
            z = _lib.NoiseParams()
            ctypes.memmove(ctypes.byref(z), ctypes.byref(noise), ctypes.sizeof(z))
            z.env_offset = noise.env_offset + lo
            env._call("emei_ip_step_noisy", *ptrs, ctypes.byref(z), env._stream())
        return obs_out if obs_out is not None else dst

    def flip(self):
        self._cur = 1 - self._cur

    # ---- fused T-step rollout (emei_cartpole_rollout_f32) ----------------------------------------
    def rollout(self, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, noise=None):
        self._alloc()
        state = self._bufs[self._cur]
        if self.env.dtype == torch.float32 and noise is None:
            return self._rollout("emei_cartpole_rollout_f32", [state.data_ptr()], rp, actions, record, rollout_stats)
        # float64 reference-exact mode / obs_noise_params: the step entry points' own arithmetic, one env per thread
        z = ctypes.byref(noise) if noise is not None else None
        return self._rollout("emei_cartpole_rollout_ref" + self.env._suffix, [state.data_ptr()], rp, actions, record, rollout_stats,
                             ref=True, extra=(z,))

    def next_obs_stateless(self, obs: torch.Tensor, action: torch.Tensor):
        """get_batch_next_obs: one dynamics step from caller-supplied observations (any batch size);
        the engine's own state is untouched."""
        env = self.env
        b = obs.shape[0]
        out = torch.empty_like(obs)
        obs_out = torch.empty_like(obs) if self.separate_obs else None
        reward = torch.empty((b, 1), dtype=env.dtype, device=env.device)
        done = torch.empty((b, 1), dtype=torch.uint8, device=env.device)
        self.params.action_kind = _ACTION_KIND[action.dtype]
        env._call(
            "emei_cartpole_step",
            obs.data_ptr(), out.data_ptr(), obs_out.data_ptr() if obs_out is not None else None, action.data_ptr(),
            reward.data_ptr(), done.data_ptr(), None, b, ctypes.byref(self.params), env._stream(),
        )
        return obs_out if obs_out is not None else out

    # freeze/unfreeze: device-side snapshot of the live state buffer (base_control.py:32-36)
    def snapshot(self):
        src = self._bufs[self._cur]
        snap = torch.empty_like(src)
        with torch.cuda.device(self.env.device):
            _lib.call("emei_snapshot_copy", snap.data_ptr(), src.data_ptr(), src.numel() * src.element_size(), self.env._stream())
        return snap

    def restore(self, snap: torch.Tensor):
        self._alloc()
        dst = self._bufs[self._cur]
        with torch.cuda.device(self.env.device):
            _lib.call("emei_snapshot_copy", dst.data_ptr(), snap.data_ptr(), snap.numel() * snap.element_size(), self.env._stream())
        self.has_state = True


class I2PEngine(RolloutMixin):
    """analytic inverted double pendulum (emei_i2p_step_*): state [B,6] ping-pong pair + observation buffers."""

    obs_dim = 6

    def rollout(self, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, noise=None):
        """emei_i2p_rollout_*: the four I2P tasks of zoo/conf/task/BI2P*.yaml through the collection loop of
        zoo/util.py:33-93, one launch; in-kernel resets = reset_model (init_qpos || init_qvel + N(0, sigma))."""
        self._alloc()
        state = self._bufs[self._cur]
        mean, sigma = self.env._init_tables()
        Arr = ctypes.c_double * 6
        z = ctypes.byref(noise) if noise is not None else None
        return self._rollout("emei_i2p_rollout" + self.env._suffix, [state.data_ptr()], rp, actions, record, rollout_stats,
                             ref=True, extra=(Arr(*mean), Arr(*sigma), z))

    def __init__(self, env, params: _lib.I2PParams):
        self.env = env
        self.params = params
        self.n = env.num_envs
        self._bufs = self._obs = self._out = None
        self._cur = 0
        self.has_state = False

    def _alloc(self):
        if self._bufs is None:
            dev, dt = self.env.device, self.env.dtype
            self._bufs = [torch.empty((self.n, 6), dtype=dt, device=dev) for _ in range(2)]
            self._obs = [torch.empty((self.n, 6), dtype=dt, device=dev) for _ in range(2)]
            self._out = StepOutputs(self.n, dt, dev)

    @property
    def state(self) -> Optional[torch.Tensor]:
        return self._bufs[self._cur] if self.has_state else None

    def set_state(self, state):
        self._alloc()
        s, _ = self.env._to_device(state, self.env.dtype)
        if tuple(s.shape) != (self.n, 6):
            raise ValueError(f"state must have shape {(self.n, 6)}, got {tuple(s.shape)}")
        self._bufs[self._cur].copy_(s)
        self.has_state = True
        self.new_episodes(reseed=False)

    def step(self, action: torch.Tensor, copy_obs: bool, noise: Optional[_lib.NoiseParams] = None):
        env = self.env
        self._alloc()
        nxt = 1 - self._cur
        src, dst = self._bufs[self._cur], self._bufs[nxt]
        obs, reward, done = self._obs[nxt], self._out.reward[nxt], self._out.done[nxt]
        if copy_obs:
            obs, reward, done = torch.empty_like(obs), torch.empty_like(reward), torch.empty_like(done)
        self.params.action_kind = _ACTION_KIND[action.dtype]
        ptrs = (src.data_ptr(), dst.data_ptr(), obs.data_ptr(), action.data_ptr(), reward.data_ptr(), done.data_ptr(),
                env.stats.data_ptr(), self.n, ctypes.byref(self.params))
        if noise is None:
            env._call("emei_i2p_step", *ptrs, env._stream())
        else:
            env._call("emei_i2p_step_noisy", *ptrs, ctypes.byref(noise), env._stream())
        self._cur = nxt
        return obs, reward, done.view(torch.bool)

    def step_range(self, lo: int, hi: int, action: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, obs_out,
                   noise: Optional[_lib.NoiseParams] = None):
        """Launch the step kernel for envs [lo, hi) only (src -> dst of the CURRENT ping-pong pair, no flip): the
        building block of the chunked host pipeline (``step_host``).  Call ``flip()`` once all ranges are launched."""
        env = self.env
        self._alloc()
        nxt = 1 - self._cur
        src, dst = self._bufs[self._cur], self._bufs[nxt]
        if obs_out is None:
            obs_out = self._obs[nxt]
        self.params.action_kind = _ACTION_KIND[action.dtype]
        es, ea = src.element_size() * 6, action.element_size()
        ptrs = (src.data_ptr() + lo * es, dst.data_ptr() + lo * es, obs_out.data_ptr() + lo * es, action.data_ptr() + lo * ea,
                reward.data_ptr() + lo * reward.element_size(), done.data_ptr() + lo, env.stats.data_ptr(), hi - lo,
                ctypes.byref(self.params))
        if noise is None:
            env._call("emei_i2p_step", *ptrs, env._stream())
        else:
            z = _lib.NoiseParams()
            ctypes.memmove(ctypes.byref(z), ctypes.byref(noise), ctypes.sizeof(z))
            z.env_offset = noise.env_offset + lo
            env._call("emei_i2p_step_noisy", *ptrs, ctypes.byref(z), env._stream())
        return obs_out

    def flip(self):
        self._cur = 1 - self._cur

    def next_obs_stateless(self, obs: torch.Tensor, action: torch.Tensor):
        """get_batch_next_obs: one dynamics step from caller-supplied STATES (the 6-d observation of this family
        does not determine the state: inverted_double_pendulum.py:56-60 is not a bijection); engine untouched."""
        b = obs.shape[0]
        out, o2 = torch.empty_like(obs), torch.empty_like(obs)
        r = torch.empty((b, 1), dtype=obs.dtype, device=obs.device)
        d = torch.empty((b, 1), dtype=torch.uint8, device=obs.device)
        self.params.action_kind = _ACTION_KIND[action.dtype]
        self.env._call("emei_i2p_step", obs.data_ptr(), out.data_ptr(), o2.data_ptr(), action.data_ptr(), r.data_ptr(),
                       d.data_ptr(), None, b, ctypes.byref(self.params), self.env._stream())
        return o2

    def snapshot(self):
        src = self._bufs[self._cur]
        snap = torch.empty_like(src)
        with torch.cuda.device(self.env.device):
            _lib.call("emei_snapshot_copy", snap.data_ptr(), src.data_ptr(), src.numel() * src.element_size(), self.env._stream())
        return snap

    def restore(self, snap: torch.Tensor):
        self._alloc()
        dst = self._bufs[self._cur]
        with torch.cuda.device(self.env.device):
            _lib.call("emei_snapshot_copy", dst.data_ptr(), snap.data_ptr(), snap.numel() * snap.element_size(), self.env._stream())
        self.has_state = True


class ChargedBallEngine(RolloutMixin):
    """charged ball (emei_charged_ball_step_*): three state arrays updated in place."""

    # step_host: the observation is the `free` state array itself, so it needs a copy anyway and kernel-side stores of
    # reward / done alone measured slower than the DMA path (16384 envs: 50.8 us against 41.5)
    zero_copy_ok = False

    def rollout(self, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, noise=None):
        ptrs = [self.on_circle.data_ptr(), self.circle.data_ptr(), self.free.data_ptr()]
        if self.env.dtype == torch.float32:
            return self._rollout("emei_charged_ball_rollout_f32", ptrs, rp, actions, record, rollout_stats)
        return self._rollout("emei_charged_ball_rollout_ref_f64", ptrs, rp, actions, record, rollout_stats, ref=True)

    def __init__(self, env, params: _lib.ChargedBallParams):
        self.env = env
        self.params = params
        self.n = env.num_envs
        self.on_circle = self.circle = self.free = None
        self._out = None
        self._flip = 0
        self.has_state = False

    def _alloc(self):
        if self.on_circle is None:
            dev, dt = self.env.device, self.env.dtype
            self.on_circle = torch.empty((self.n,), dtype=torch.uint8, device=dev)
            self.circle = torch.empty((self.n, 2), dtype=dt, device=dev)
            self.free = torch.empty((self.n, 4), dtype=dt, device=dev)
            self._out = StepOutputs(self.n, dt, dev)

    def set_state(self, on_circle, circle, free):
        self._alloc()
        env = self.env
        self.on_circle.copy_(env._to_device(on_circle, torch.uint8)[0].reshape(self.n))
        self.circle.copy_(env._to_device(circle, env.dtype)[0].reshape(self.n, 2))
        self.free.copy_(env._to_device(free, env.dtype)[0].reshape(self.n, 4))
        self.has_state = True
        self.new_episodes(reseed=False)

    def sample_initial(self, seed: int, env_offset: int):
        self._alloc()
        self.env._call(
            "emei_init_charged_ball", self.on_circle.data_ptr(), self.circle.data_ptr(), self.free.data_ptr(), self.n,
            float(self.params.radius), ctypes.c_uint64(seed), ctypes.c_uint64(env_offset), self.env._stream(),
        )
        self.has_state = True

    def step(self, action: torch.Tensor, copy_obs: bool):
        env = self.env
        self._flip ^= 1
        reward, done = self._out.reward[self._flip], self._out.done[self._flip]
        if copy_obs:
            reward, done = torch.empty_like(reward), torch.empty_like(done)
        self.params.action_kind = _ACTION_KIND[action.dtype]
        env._call(
            "emei_charged_ball_step",
            self.on_circle.data_ptr(), self.circle.data_ptr(), self.free.data_ptr(), action.data_ptr(),
            reward.data_ptr(), done.data_ptr(), env.stats.data_ptr(), self.n, ctypes.byref(self.params), env._stream(),
        )
        obs = self.free.clone() if copy_obs else self.free
        return obs, reward, done.view(torch.bool)

    def step_range(self, lo: int, hi: int, action: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, obs_out):
        env = self.env
        self.params.action_kind = _ACTION_KIND[action.dtype]
        es = self.free.element_size()
        env._call(
            "emei_charged_ball_step",
            self.on_circle.data_ptr() + lo, self.circle.data_ptr() + lo * 2 * es, self.free.data_ptr() + lo * 4 * es,
            action.data_ptr() + lo * action.element_size(), reward.data_ptr() + lo * es, done.data_ptr() + lo,
            env.stats.data_ptr(), hi - lo, ctypes.byref(self.params), env._stream(),
        )
        return self.free

    def flip(self):
        pass

    def snapshot(self):
        out = []
        with torch.cuda.device(self.env.device):
            for src in (self.on_circle, self.circle, self.free):
                snap = torch.empty_like(src)
                _lib.call("emei_snapshot_copy", snap.data_ptr(), src.data_ptr(), src.numel() * src.element_size(), self.env._stream())
                out.append(snap)
        return tuple(out)

    def restore(self, snaps):
        self._alloc()
        with torch.cuda.device(self.env.device):
            for dst, snap in zip((self.on_circle, self.circle, self.free), snaps):
                _lib.call("emei_snapshot_copy", dst.data_ptr(), snap.data_ptr(), snap.numel() * snap.element_size(), self.env._stream())
        self.has_state = True


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """The row loaders use 128-bit accesses: a contiguous view that starts at an odd offset (``obs[k:]`` of 12-byte
    action rows or 72-byte observation rows) is copied to a fresh, aligned allocation (the reference accepts any slice)."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _sumsq(env, a: torch.Tensor, group):
    """batch-wide sum of squared actions (hopper.py:98 / half_cheetah.py:61), all-reduced when the batch is sharded."""
    sumsq = torch.empty(1, dtype=torch.float64, device=env.device)
    ws = getattr(env, "_sumsq_ws", None)
    if ws is None:  # zero-filled once; the kernel leaves its ticket counter at zero
        ws = env._sumsq_ws = torch.zeros(_lib.SUMSQ_WORKSPACE_BYTES // 8, dtype=torch.float64, device=env.device)
    env._call("emei_sumsq", a.data_ptr(), a.numel(), sumsq.data_ptr(), ws.data_ptr(), env._stream())
    if getattr(env, "ctrl_cost_scope", "global") == "global":
        from .dist import all_reduce_sum_

        all_reduce_sum_(sumsq, group)
    return sumsq


def _score_cache_key(env, params, tensors, group):
    """Identity of one scoring call: same tensors (address, shape, torch version counter), same parameters, same
    stream, and NO emei kernel launched since the cached pass (our kernels write through raw pointers and do not
    bump torch's version counters)."""
    ident = tuple((t.data_ptr(), tuple(t.shape), t._version, t.dtype) if t is not None else None for t in tensors)
    return (ident, bytes(params), env._stream(), id(group))


def score(env, params: _lib.ScoringParams, obs, pre_obs=None, action=None, want="both", group=None):
    """Fused get_batch_reward + get_batch_terminal through emei_reward_terminal_* for any batch size.

    Hopper/HalfCheetah: pass 1 = emei_sumsq_* over the action batch (the reference sums the control
    cost over the WHOLE batch, hopper.py:98 / half_cheetah.py:61), optional all-reduce of that one
    double across ranks when the batch is sharded, pass 2 = the fused row kernel.  When ``pre_obs`` and
    ``obs`` are the two shifted views of one trajectory tensor (``seq[:-1]`` / ``seq[1:]``) the C side
    walks the trajectory and reads every observation row once (include/emei_b200.h).

    The reference's API has two calls (get_batch_reward, get_batch_terminal: mujoco_env.py:163-169 callers);
    a caller that makes them back to back on the SAME device tensors gets the second answer from the first
    call's fused pass (one row pass instead of two).
    Returns (reward [B,1] or None, done bool[B,1] or None, came_from_numpy)."""
    family = params.family
    o, was_np = env._to_device(obs, env.dtype)
    if o.dim() != 2 or o.shape[1] != _lib.lib.emei_family_obs_dim(family):
        raise ValueError(f"obs must be [B,{_lib.lib.emei_family_obs_dim(family)}], got {tuple(o.shape)}")
    b = o.shape[0]
    needs_pre = family in (_lib.HOPPER, _lib.HALFCHEETAH)
    p = a = None
    if needs_pre and (want != "terminal" or (pre_obs is not None and action is not None)):
        if pre_obs is None or action is None:
            raise TypeError("get_batch_reward of this env needs obs, pre_obs and action")
        p, _ = env._to_device(pre_obs, env.dtype)
        a, _ = env._to_device(action, env.dtype)
        if tuple(p.shape) != tuple(o.shape) or a.shape[0] != b:
            raise ValueError("obs / pre_obs / action batch shapes disagree")
    # ---- the other half of a reward / terminal pair asked for on the same tensors: reuse the fused pass
    # Only the COMPLEMENTARY half is ever served (reward after terminal, terminal after reward), once: repeating the
    # same call, or get_batch_reward_terminal, always runs the kernels.
    key = key_obs = None
    if not was_np and want in ("reward", "terminal"):
        key_obs = _score_cache_key(env, params, (o,), group)
        if not needs_pre or p is not None:
            key = _score_cache_key(env, params, (o, p, a), group)
        hit = getattr(env, "_score_cache", None)
        env._score_cache = None
        if hit is not None and hit[2] == _lib.launch_count and hit[5] != want:
            if key is not None and hit[0] == key:
                return hit[3], hit[4], was_np
            if key is None and want == "terminal" and hit[1] == key_obs:  # terminal with obs alone: the flags depend on obs only
                return None, hit[4], was_np
    sumsq = None
    if needs_pre and p is not None:
        sumsq = _sumsq(env, _aligned16(a), group)
        if p.data_ptr() % 16 != 0 or o.data_ptr() % 16 != 0:  # keep the seq[:-1] / seq[1:] address relation when both are aligned
            p = _aligned16(p)
    elif needs_pre:
        # terminal only: reward inputs are not needed; feed harmless placeholders
        p = o
        sumsq = torch.zeros(1, dtype=torch.float64, device=env.device)
    o = _aligned16(o)
    reward = torch.empty((b, 1), dtype=env.dtype, device=env.device)
    done = torch.empty((b, 1), dtype=torch.uint8, device=env.device)
    env._call(
        "emei_reward_terminal",
        o.data_ptr(), p.data_ptr() if p is not None else None, reward.data_ptr(), done.data_ptr(),
        env.stats.data_ptr() if getattr(env, "accumulate_scoring_stats", False) else None,
        sumsq.data_ptr() if sumsq is not None else None, b, ctypes.byref(params), env._stream(),
    )
    done = done.view(torch.bool)
    if key is not None and not getattr(env, "accumulate_scoring_stats", False):
        env._score_cache = (key, key_obs, _lib.launch_count, reward, done, want)
    return reward, done, was_np


def score_seq(env, params: _lib.ScoringParams, obs_seq, action=None, group=None):
    """Trajectory scoring through emei_reward_terminal_seq_*: ``obs_seq`` [T+1, n, D] (an imagined rollout),
    ``action`` [T, n, A] -> reward [T, n, 1], done bool [T, n, 1].  Equal to ``score`` on
    ``obs = obs_seq[1:], pre_obs = obs_seq[:-1]`` flattened; every observation row is read once."""
    family = params.family
    s, was_np = env._to_device(obs_seq, env.dtype)
    d = _lib.lib.emei_family_obs_dim(family)
    if s.dim() != 3 or s.shape[2] != d or s.shape[0] < 1:
        raise ValueError(f"obs_seq must be [T+1, n, {d}], got {tuple(s.shape)}")
    T, n = s.shape[0] - 1, s.shape[1]
    needs_pre = family in (_lib.HOPPER, _lib.HALFCHEETAH)
    a = sumsq = None
    if needs_pre:
        if action is None:
            raise TypeError("get_batch_reward of this env needs the actions")
        a, _ = env._to_device(action, env.dtype)
        if a.shape[0] != T or a.shape[1] != n:
            raise ValueError(f"action must be [T={T}, n={n}, A], got {tuple(a.shape)}")
    if (n * d * s.element_size()) % 16 != 0:
        # rows of t >= 1 would lose the loader's alignment: score the flat views, whose pass computes the sum of squares
        r, dn, _ = score(env, params, s[1:].reshape(T * n, d), s[:-1].reshape(T * n, d).clone(),
                         a.reshape(T * n, -1) if needs_pre else None, group=group)
        return r.reshape(T, n, 1), dn.reshape(T, n, 1), was_np
    if needs_pre:
        sumsq = _sumsq(env, _aligned16(a), group)
    s = _aligned16(s)
    reward = torch.empty((T, n, 1), dtype=env.dtype, device=env.device)
    done = torch.empty((T, n, 1), dtype=torch.uint8, device=env.device)
    env._call(
        "emei_reward_terminal_seq", s.data_ptr(), reward.data_ptr(), done.data_ptr(),
        env.stats.data_ptr() if getattr(env, "accumulate_scoring_stats", False) else None,
        sumsq.data_ptr() if sumsq is not None else None, n, T, ctypes.byref(params), env._stream(),
    )
    return reward, done.view(torch.bool), was_np


def time_fused_scoring(env, obs, pre_obs, action, reps=10):
    """CUDA-event duration (ms per launch) of the fused reward+terminal kernel alone, for the roofline
    of bench.py: the sum-of-squares pre-pass runs once outside the timed launches."""
    params = env._scoring_params()
    b = obs.shape[0]
    sumsq = torch.zeros(1, dtype=torch.float64, device=env.device)
    ws = torch.zeros(_lib.SUMSQ_WORKSPACE_BYTES // 8, dtype=torch.float64, device=env.device)
    env._call("emei_sumsq", action.data_ptr(), action.numel(), sumsq.data_ptr(), ws.data_ptr(), env._stream())
    reward = torch.empty((b, 1), dtype=env.dtype, device=env.device)
    done = torch.empty((b, 1), dtype=torch.uint8, device=env.device)

    def launch():
        env._call("emei_reward_terminal", obs.data_ptr(), pre_obs.data_ptr(), reward.data_ptr(), done.data_ptr(), None,
                  sumsq.data_ptr(), b, ctypes.byref(params), env._stream())

    launch()
    torch.cuda.synchronize(env.device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize(env.device)
    return e0.elapsed_time(e1) / reps


ZERO_COPY_MAX_ENVS = 65536  # measured: scripts/probe_zero_copy_small.py, profiles/r02_zero_copy_small.txt
ZERO_COPY_ACTION_MAX_ENVS = 8192  # = the small-batch kernel's limit (cartpole_tma.cuh): plain loads below it


class HostStaging:
    """Pinned host buffers + the copy choreography of ``step_host`` (the end-to-end path with HOST
    inputs and outputs).  The env batch is cut into ``chunks`` contiguous ranges, each on its own
    stream: H2D(actions) -> step kernel on the range -> D2H(obs, reward, done).  Envs are independent,
    so range k+1's upload and range k-1's download overlap range k's kernel, and PCIe runs in both
    directions at once.  One host synchronisation per call."""

    @staticmethod
    def plan_ranges(n: int, chunks: Optional[int] = None, fractions=None):
        """[(lo, hi), ...] tiling [0, n)."""
        if fractions is None:
            if chunks is None:
                # measured on the B200 box (scripts/probe_step_host.py, 2^20 cart-pole envs, graph replay): 1 range
                # 0.523 ms, 2: 0.506, 4: 0.512, 8: 0.547 -- every extra range adds 4 DMA transfers of fixed cost, so
                # ranges of ~2^19 envs, at most 16
                chunks = min(16, max(1, n >> 19))
            chunks = max(1, min(int(chunks), n // 131072 or 1))  # small batches: one range (latency-bound anyway)
            # a short first range starts the downloads early ([0.25, 0.75] measured 0.486 ms against 0.503 for halves)
            fractions = [1.0] if chunks == 1 else [0.5 / chunks] + [(1.0 - 0.5 / chunks) / (chunks - 1)] * (chunks - 1)
        acc, edges = 0.0, [0]
        for f in fractions:
            acc += f
            edges.append(min(n, int(round(acc * n)) // 16 * 16))  # interior edges on 16-env boundaries: every array
        edges[-1] = n                                             # of a range (uint8 flags included) stays 16-byte aligned
        return [(edges[i], edges[i + 1]) for i in range(len(edges) - 1) if edges[i + 1] > edges[i]]

    ALL_OUTPUTS = ("obs", "reward", "done")

    def __init__(self, env, chunks: Optional[int] = None, fractions=None):
        self.env = env
        self.outputs = self.ALL_OUTPUTS  # which results the current call downloads
        n = env.num_envs
        cont = len(env.action_space.shape) > 0
        dev = env.device
        self.a_host = torch.empty((n,), dtype=torch.float32 if cont else torch.uint8).pin_memory()
        self.a_dev = torch.empty_like(self.a_host, device=dev)
        obs_dim = env.observation_space.shape[0]
        self.obs_host = torch.empty((n, obs_dim), dtype=env.dtype).pin_memory()
        self.rew_host = torch.empty((n, 1), dtype=env.dtype).pin_memory()
        self.done_host = torch.empty((n, 1), dtype=torch.bool).pin_memory()
        self.rew_dev = torch.empty((n, 1), dtype=env.dtype, device=dev)
        self.done_dev = torch.empty((n, 1), dtype=torch.uint8, device=dev)
        self.h2d_bytes = self.a_host.numel() * self.a_host.element_size()
        self._out_bytes = {"obs": self.obs_host.numel() * self.obs_host.element_size(),
                           "reward": self.rew_host.numel() * self.rew_host.element_size(), "done": self.done_host.numel()}
        self.d2h_bytes = sum(self._out_bytes.values())
        self.ranges = self.plan_ranges(n, chunks, fractions)
        self.streams = [torch.cuda.Stream(dev) for _ in self.ranges]
        self.done_host_u8 = self.done_host.view(torch.uint8)
        self.use_graphs = True
        # kernel-side loads / stores of the pinned host arrays instead of DMA transfers (see _enqueue); EMEI_ZERO_COPY_MAX
        # overrides the batch-size limit (0 disables)
        self.zero_copy = n <= int(os.environ.get("EMEI_ZERO_COPY_MAX", ZERO_COPY_MAX_ENVS)) and getattr(env._engine, "zero_copy_ok", True)
        self._capture_stream = torch.cuda.Stream(dev)
        self._graphs, self._seen, self._keep, self._pinned = {}, {}, {}, {}
        self._np_views = None

    # ---- one host step ---------------------------------------------------------------------------
    def _enqueue(self, a_src, noise=None):
        """Queue the whole step on the CURRENT stream (+ one side stream per range): uploads, kernels, downloads.
        No host synchronisation: used eagerly and under CUDA-graph capture."""
        env, eng = self.env, self.env._engine
        cur = torch.cuda.current_stream(env.device)
        kw = {} if noise is None else {"noise": noise}
        want = self.outputs
        if len(self.ranges) == 1 and self.zero_copy:
            # Small batch: the host step is pure latency (a 4096-env step is three copy-engine transfers of a few KB
            # around a 2 us kernel, ~10 us each).  A page-locked host buffer IS device-addressable (UVA), so the kernel
            # reads the actions from the caller's pinned array and stores reward / done / obs straight into the pinned
            # result arrays: one launch, no DMA transfers.  Same bytes over PCIe, moved by the SMs' loads and stores.
            # (At 2^20 envs the copy engines win -- 0.49 ms against 0.55 -- so this is for small batches only.)
            act = a_src
            if env.num_envs >= ZERO_COPY_ACTION_MAX_ENVS:  # the large-batch step kernel stages its actions with bulk (TMA) copies:
                self.a_dev.copy_(a_src, non_blocking=True)  # those read device memory, so the actions take the DMA path there
                act = self.a_dev
            obs = eng.step_range(0, env.num_envs, act, self.rew_host if "reward" in want else self.rew_dev,
                                 self.done_host_u8 if "done" in want else self.done_dev, self.obs_host if "obs" in want else None, **kw)
            if "obs" in want and obs is not self.obs_host:  # families whose observation is the state array itself
                self.obs_host.copy_(obs, non_blocking=True)
            return
        if len(self.ranges) == 1:  # one range, copy engines: no side streams
            self.a_dev.copy_(a_src, non_blocking=True)
            obs = eng.step_range(0, env.num_envs, self.a_dev, self.rew_dev, self.done_dev, None, **kw)
            if "obs" in want:
                self.obs_host.copy_(obs, non_blocking=True)
            if "reward" in want:
                self.rew_host.copy_(self.rew_dev, non_blocking=True)
            if "done" in want:
                self.done_host_u8.copy_(self.done_dev, non_blocking=True)
            return
        start = torch.cuda.Event()
        start.record(cur)
        for (lo, hi), st in zip(self.ranges, self.streams):
            with torch.cuda.stream(st):
                st.wait_event(start)  # everything queued before this call (reset, set_state, ...) is visible
                self.a_dev[lo:hi].copy_(a_src[lo:hi], non_blocking=True)
                obs = eng.step_range(lo, hi, self.a_dev, self.rew_dev, self.done_dev, None, **kw)
                if "obs" in want:
                    self.obs_host[lo:hi].copy_(obs[lo:hi], non_blocking=True)
                if "reward" in want:
                    self.rew_host[lo:hi].copy_(self.rew_dev[lo:hi], non_blocking=True)
                if "done" in want:
                    self.done_host_u8[lo:hi].copy_(self.done_dev[lo:hi], non_blocking=True)
        for st in self.streams:
            cur.wait_stream(st)

    def _result(self):
        w = self.outputs
        v = self._np_views  # the numpy views of the pinned result arrays are made once (a small host step is latency)
        if v is None:
            v = self._np_views = {"obs": self.obs_host.numpy(), "reward": self.rew_host.numpy(), "done": self.done_host.numpy()}
        return (v["obs"] if "obs" in w else None, v["reward"] if "reward" in w else None, v["done"] if "done" in w else None, False, {})

    def step(self, action, outputs=None):
        """``outputs``: subset of ("obs", "reward", "done") to download (default: all three, the reference's step()
        contract); what is not asked for stays on the device (``env.state``) and comes back as None -- a caller that
        only consumes reward / done moves 5 bytes per env over PCIe instead of 21.

        Eager the first time a (caller buffer, ping-pong parity) pair is seen; captured into a CUDA graph the
        second time and replayed from then on: a host step is ~5 enqueues per range, and at 2^20 envs the host
        could not queue them as fast as PCIe drains them (0.52 ms per step against 0.42 ms of copies); one graph
        launch also lets the ranges be finer.  The graph bakes pointers in, so it is keyed by the action buffer's
        address and the engine's current ping-pong side."""
        env = self.env
        eng = env._engine
        assert eng is not None and eng.has_state, "Call reset before using step method."
        outs = self.ALL_OUTPUTS if outputs is None else tuple(o for o in self.ALL_OUTPUTS if o in outputs)
        if outputs is not None and (len(outs) != len(tuple(outputs)) or not outs):
            raise ValueError(f"outputs must be a non-empty subset of {self.ALL_OUTPUTS}, got {outputs!r}")
        if outs != self.outputs or self.d2h_bytes == 0:
            self.outputs = outs
            self.d2h_bytes = sum(self._out_bytes[o] for o in outs)
        a = torch.as_tensor(action)
        if a.is_cuda:
            raise TypeError("step_host takes host actions; use step() for device tensors")
        if a.dim() != 1:
            a = a.reshape(-1)
        if a.numel() != self.a_host.numel():
            raise ValueError(f"step_host: expected {self.a_host.numel()} actions, got {a.numel()}")
        ptr = a.data_ptr()
        if a.dtype == self.a_host.dtype and a.is_contiguous() and (ptr in self._pinned or a.is_pinned()):
            # is_pinned() is a driver query: asked once per buffer.  The cache keeps the tensor alive, so its address
            # cannot be handed to a pageable allocation while it is trusted (at most 32 caller buffers are remembered).
            if ptr not in self._pinned and len(self._pinned) < 32:
                self._pinned[ptr] = a
            a_src = a  # already page-locked in the wire dtype: DMA straight from the caller's buffer
        else:
            self.a_host.copy_(a)  # host-side cast into the pinned staging buffer (uint8 / float32)
            a_src = self.a_host
        cur = torch.cuda.current_stream(env.device)
        noise = getattr(env, "_next_obs_noise", lambda: None)()
        if noise is not None:  # obs_noise_params: the step counter changes every call, so nothing can be baked into a graph
            self._enqueue(a_src, noise)
            eng.flip()
            cur.synchronize()
            return self._result()
        key = (a_src.data_ptr(), getattr(eng, "_cur", 0), outs)
        graph = self._graphs.get(key) if self.use_graphs else None
        if graph is None and self.use_graphs and self._seen.get(key, 0) >= 1 and len(self._graphs) < 32:
            graph = torch.cuda.CUDAGraph()
            launches0 = _lib.launch_count
            # no garbage collection inside the capture: a dead CUDAGraph (an earlier env's) destroyed mid-capture
            # invalidates it
            gc.collect()
            gc_was_on = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(graph, stream=self._capture_stream, capture_error_mode="thread_local"):
                    self._enqueue(a_src)
            finally:
                if gc_was_on:
                    gc.enable()
            _lib.launch_count = launches0  # capture launches nothing
            self._graphs[key] = graph
            self._keep[key] = a_src  # the graph reads this buffer at every replay
        if graph is not None:
            graph.replay()
            _lib.launch_count += len(self.ranges)
        else:
            if len(self._seen) > 256:  # a caller that never reuses a buffer: nothing worth remembering
                self._seen.clear()
            self._seen[key] = self._seen.get(key, 0) + 1
            self._enqueue(a_src)
        eng.flip()
        cur.synchronize()
        return self._result()
