"""Device-buffer owners behind the env classes: they hold the state tensors, build the POD
parameter structs and issue the C-ABI calls.  No arithmetic happens in Python.

HBM layout (DESIGN.md section 3):
  cart-pole / IP : state  [B,4] row-major (one 128-bit row per env), ping-pong pair of buffers;
                   IP keeps a separate obs buffer (theta wrapped) because the reference wraps only
                   the observation copy (inverted_pendulum.py:45-49).
  I2P            : the same with [B,6] rows and obs buffers (RowStateEngine serves all three).
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

_KIND_DTYPE = {_lib.ACTION_DISCRETE_U8: torch.uint8, _lib.ACTION_DISCRETE_I32: torch.int32, _lib.ACTION_DISCRETE_I64: torch.int64,
               _lib.ACTION_CONTINUOUS_F32: torch.float32, _lib.ACTION_CONTINUOUS_F64: torch.float64}


def action_rule(env, a: torch.Tensor, continuous: bool) -> torch.Tensor:
    """The dtype and range rule of every action entry point (base_control.py:62-66 for a batch): device tensor ``a`` of
    any shape -> one of the encodings of include/emei_b200.h.  ``bool`` is read as its uint8 bytes."""
    if a.dtype == torch.bool:
        a = a.view(torch.uint8)
    if continuous:
        if a.dtype not in (torch.float32, torch.float64):
            a = a.to(torch.float32)
    elif a.dtype.is_floating_point:
        raise AssertionError(f"actions of dtype {a.dtype} invalid: discrete action space needs integers")
    elif a.dtype not in _ACTION_KIND:
        a = a.to(torch.int64)
    if env.validate_actions:  # device-side range check: one sync, off by default
        if continuous:
            lo, hi = float(env.action_space.low.min()), float(env.action_space.high.max())
            ok = bool(((a >= lo) & (a <= hi)).all())
        else:
            ok = bool(((a >= 0) & (a < env.action_space.n)).all())
        assert ok, "actions outside the action space"
    return a


def normalise_action(env, action, continuous: bool, n: int) -> torch.Tensor:
    """-> contiguous device tensor [n] of one step's actions for a batch of ``n`` rows (int -> array, as
    base_control.py:62-66; then ``action_rule``)."""
    if isinstance(action, (int, np.integer)) and not continuous:
        action = torch.full((n,), int(action), dtype=torch.int64)
    a, _ = env._to_device(action)
    if a.numel() != n:
        raise AssertionError(f"{action!r} ({type(action)}) invalid: expected {n} actions, got shape {tuple(a.shape)}")
    return action_rule(env, a.reshape(n), continuous).contiguous()


class StepOutputs:
    """Ping-pong reward / done buffers of the zero-copy mode (``copy_outputs=False``): what step t returns stays valid
    until step t+2 overwrites it (the charged ball's observation is the live ``free`` array: valid until step t+1).
    The default ``copy_outputs=True`` returns fresh tensors instead, like the reference's ``state.copy()``."""

    def __init__(self, n, dtype, device):
        self.reward = [torch.empty((n, 1), dtype=dtype, device=device) for _ in range(2)]
        self.done = [torch.empty((n, 1), dtype=torch.uint8, device=device) for _ in range(2)]


class Engine:
    """Base of the engines: episode bookkeeping buffers, the call of a fused T-step rollout entry point and the
    freeze snapshots of the live state arrays (``_state_arrays``).

    float32 without state noise: the packed kernels (emei_cartpole_rollout_f32 / emei_charged_ball_rollout_f32).
    float64 (reference-exact), the inverted double pendulum and obs_noise_params: the reference-arithmetic kernels
    (emei_cartpole_rollout_ref_* / emei_i2p_rollout_* / emei_charged_ball_rollout_ref_f64), one env per thread, the
    step entry points' own device functions.  Records, rewards and episode returns have the engine dtype."""

    ep_step = ep_return = ep_index = None
    t_global = 0
    obs_dim = 4

    def _alloc_episode(self):
        if self.ep_step is None:
            dev = self.env.device
            self.ep_step = torch.zeros(self.n, dtype=torch.int32, device=dev)
            self.ep_return = torch.zeros(self.n, dtype=self.env.dtype, device=dev)
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

    def _rollout(self, entry: str, state_ptrs, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, extra=()):
        """entry: C-ABI symbol (with the precision suffix); extra: its trailing arguments before the stream (noise / init tables)."""
        env = self.env
        self._alloc_episode()
        T, n, dev, D, rdt = int(rp.horizon), self.n, env.device, self.obs_dim, env.dtype
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

    # ---- sampling-based planning (emei_*_plan_eval_* / emei_plan_update_*): the env's own state is never touched
    def _plan_eval(self, entry: str, state_ptrs, mean: torch.Tensor, std, candidates: int, q: _lib.PlanParams, want_actions: bool):
        """-> (returns [B, K] float64, actions [H, B, K] in the plan's action type or None) of the candidates drawn around
        (mean, std) [H, B] from the start states behind ``state_ptrs``."""
        env = self.env
        H, B = mean.shape
        returns = (torch.zeros if H == 0 else torch.empty)((B, candidates), dtype=torch.float64, device=env.device)
        actions = torch.empty((H, B, candidates), dtype=_KIND_DTYPE[q.action_kind], device=env.device) if want_actions else None
        self.params.action_kind = q.action_kind
        env._call(entry, *state_ptrs, mean.data_ptr(), std.data_ptr() if std is not None else None, returns.data_ptr(),
                  actions.data_ptr() if actions is not None else None, B, candidates, H, ctypes.byref(q), ctypes.byref(self.params),
                  env._stream())
        return returns, actions

    def plan_update(self, returns: torch.Tensor, mean: torch.Tensor, std, q: _lib.PlanParams, want_best: bool):
        """Refit ``mean`` / ``std`` [H, B] in place from ``returns`` [B, K] of the candidates drawn with ``q``
        (emei_plan_update_*) -> (best_actions [H, B], best_return [B]) when ``want_best``, else (None, None)."""
        env = self.env
        H, B = mean.shape
        best_a = torch.empty((H, B), dtype=_KIND_DTYPE[q.action_kind], device=env.device) if want_best else None
        best_r = torch.empty((B,), dtype=torch.float64, device=env.device) if want_best else None
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        env._call("emei_plan_update", returns.data_ptr(), mean.data_ptr(), ptr(std), ptr(best_a), ptr(best_r), B, returns.shape[1], H,
                  ctypes.byref(q), env._stream())
        return best_a, best_r

    # ---- policy search (emei_*_policy_eval_* / emei_policy_perturb / emei_policy_update): the env's own state is never touched
    def _policy_eval(self, entry: str, state_ptrs, E: int, params: torch.Tensor, H: int, q: _lib.PolicyParams, want_actions: bool):
        """-> (returns [C, E] float64, actions [H, C, E] in the policy's action type or None) of the linear policies
        ``params`` [C, P] (float64, contiguous) run closed loop for H steps from the E start states behind ``state_ptrs``."""
        env = self.env
        C = params.shape[0]
        returns = (torch.zeros if H == 0 else torch.empty)((C, E), dtype=torch.float64, device=env.device)
        actions = torch.empty((H, C, E), dtype=_KIND_DTYPE[q.action_kind], device=env.device) if want_actions else None
        self.params.action_kind = q.action_kind
        env._call(entry, *state_ptrs, params.data_ptr(), returns.data_ptr(), actions.data_ptr() if actions is not None else None, C, E,
                  H, ctypes.byref(q), ctypes.byref(self.params), env._stream())
        return returns, actions

    def policy_perturb(self, theta: torch.Tensor, directions: int, q: _lib.PolicyParams) -> torch.Tensor:
        """-> params [2N, P] float64: theta +- noise delta_k of the directions keyed by ``q.seed`` (emei_policy_perturb)."""
        env = self.env
        params = torch.empty((2 * directions, theta.numel()), dtype=torch.float64, device=env.device)
        with torch.cuda.device(env.device):
            _lib.call("emei_policy_perturb", theta.data_ptr(), params.data_ptr(), directions, theta.numel(), ctypes.byref(q), env._stream())
        return params

    def policy_update(self, returns: torch.Tensor, theta: torch.Tensor, q: _lib.PolicyParams, stats=None):
        """Step ``theta`` [P] (float64) in place along the ``q.top`` best of the directions behind ``returns`` [2N, E]
        (emei_policy_update); ``stats``: a device double[4] to write, or None."""
        env = self.env
        with torch.cuda.device(env.device):
            _lib.call("emei_policy_update", returns.data_ptr(), theta.data_ptr(), stats.data_ptr() if stats is not None else None,
                      returns.shape[0] // 2, returns.shape[1], theta.numel(), ctypes.byref(q), env._stream())

    # freeze/unfreeze: device-side copies of the live state arrays (base_control.py:32-36)
    def snapshot(self) -> tuple:
        snaps = tuple(torch.empty_like(t) for t in self._state_arrays())
        self._copy(snaps, self._state_arrays())
        return snaps

    def restore(self, snaps: tuple):
        self._alloc()
        self._copy(self._state_arrays(), snaps)
        self.has_state = True

    def _copy(self, dsts, srcs):
        with torch.cuda.device(self.env.device):
            for dst, src in zip(dsts, srcs):
                _lib.call("emei_snapshot_copy", dst.data_ptr(), src.data_ptr(), src.numel() * src.element_size(), self.env._stream())


class RowStateEngine(Engine):
    """State [B, width], one row per env, in a ping-pong pair of buffers; ``separate_obs``: the observation goes to a
    buffer pair of its own (the pendulums, whose observation wraps the angles), else it is the next state row."""

    def __init__(self, env, params, width: int, separate_obs: bool, step_entry: str, noisy_entry: str):
        self.env = env
        self.params = params
        self.n = env.num_envs
        self.obs_dim = width
        self.separate_obs = separate_obs
        self._step_entry, self._noisy_entry = step_entry, noisy_entry
        self._jacobian_entry, self._vjp_entry = step_entry + "_jacobian", step_entry + "_vjp"
        self._trajectory_entry = step_entry[: -len("_step")] + "_trajectory"
        self._trajectory_vjp_entry = self._trajectory_entry + "_vjp"
        self._plan_eval_entry = step_entry[: -len("_step")] + "_plan_eval"
        self._policy_eval_entry = step_entry[: -len("_step")] + "_policy_eval"
        self._bufs = self._obs = self._out = None
        self._cur = 0
        self.has_state = False

    def _alloc(self):
        if self._bufs is None:
            dev, dt = self.env.device, self.env.dtype
            self._bufs = [torch.empty((self.n, self.obs_dim), dtype=dt, device=dev) for _ in range(2)]
            if self.separate_obs:
                self._obs = [torch.empty((self.n, self.obs_dim), dtype=dt, device=dev) for _ in range(2)]
            self._out = StepOutputs(self.n, dt, dev)

    def _state_arrays(self):
        return [self._bufs[self._cur]]

    @property
    def state(self) -> Optional[torch.Tensor]:
        return self._bufs[self._cur] if self.has_state else None

    def set_state(self, state):
        self._alloc()
        s, _ = self.env._to_device(state, self.env.dtype)
        if tuple(s.shape) != (self.n, self.obs_dim):
            raise ValueError(f"state must have shape {(self.n, self.obs_dim)}, got {tuple(s.shape)}")
        self._bufs[self._cur].copy_(s)
        self.has_state = True
        self.new_episodes(reseed=False)

    def _launch(self, lo: int, hi: int, src, dst, obs, action, reward, done, stats, noise):
        """One step launch over rows [lo, hi) of the given arrays.  ``noise``: the step's NoiseParams
        (obs_noise_params); a range draws the streams of its own global env ids."""
        env = self.env
        self.params.action_kind = _ACTION_KIND[action.dtype]
        # byte strides of the arrays, needed for a range only (a whole-batch step is on the host's per-call path)
        es, ea, er = (src.element_size() * self.obs_dim, action.element_size(), reward.element_size()) if lo else (0, 0, 0)
        args = (src.data_ptr() + lo * es, dst.data_ptr() + lo * es, (obs.data_ptr() + lo * es) if obs is not None else None,
                action.data_ptr() + lo * ea, reward.data_ptr() + lo * er, done.data_ptr() + lo, stats, hi - lo,
                ctypes.byref(self.params))
        if noise is None:
            env._call(self._step_entry, *args, env._stream())
            return
        if lo:
            z = _lib.NoiseParams()
            ctypes.memmove(ctypes.byref(z), ctypes.byref(noise), ctypes.sizeof(z))
            z.env_offset = noise.env_offset + lo
            noise = z
        env._call(self._noisy_entry, *args, ctypes.byref(noise), env._stream())

    def step(self, action: torch.Tensor, copy_obs: bool, noise: Optional[_lib.NoiseParams] = None):
        """``step_range(0, n)`` + ``flip()``, with the outputs of ``copy_obs`` (fresh tensors) or the ping-pong buffers."""
        self._alloc()
        nxt = 1 - self._cur
        src, dst = self._bufs[self._cur], self._bufs[nxt]
        obs = self._obs[nxt] if self.separate_obs else None
        reward, done = self._out.reward[nxt], self._out.done[nxt]
        if copy_obs:
            obs, reward, done = torch.empty_like(src), torch.empty_like(reward), torch.empty_like(done)
        self._launch(0, self.n, src, dst, obs, action, reward, done, self.env.stats.data_ptr(), noise)
        self._cur = nxt
        return (obs if obs is not None else dst), reward, done.view(torch.bool)

    def step_range(self, lo: int, hi: int, action: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, obs_out,
                   noise: Optional[_lib.NoiseParams] = None):
        """Launch the step kernel for envs [lo, hi) only (src -> dst of the CURRENT ping-pong pair, no flip):
        the building block of the chunked host pipeline (``step_host``).  Call ``flip()`` once all ranges are launched."""
        self._alloc()
        dst = self._bufs[1 - self._cur]
        if self.separate_obs and obs_out is None:
            obs_out = self._obs[1 - self._cur]
        self._launch(lo, hi, self._bufs[self._cur], dst, obs_out, action, reward, done, self.env.stats.data_ptr(), noise)
        return obs_out if obs_out is not None else dst

    def flip(self):
        self._cur = 1 - self._cur

    def transition_stateless(self, rows: torch.Tensor, action: torch.Tensor):
        """One step of the step kernel from caller-supplied state rows [b, width] (any batch size, no state noise, no
        statistics); the engine's own state is untouched.  -> (state_out, obs, reward [b,1], done bool [b,1]); obs is
        state_out itself when the family has no separate observation."""
        env = self.env
        b = rows.shape[0]
        out = torch.empty_like(rows)
        obs = torch.empty_like(rows) if self.separate_obs else None
        reward = torch.empty((b, 1), dtype=env.dtype, device=env.device)
        done = torch.empty((b, 1), dtype=torch.uint8, device=env.device)
        self._launch(0, b, rows, out, obs, action, reward, done, None, None)
        return out, (obs if obs is not None else out), reward, done.view(torch.bool)

    def next_obs_stateless(self, rows: torch.Tensor, action: torch.Tensor):
        """get_batch_next_obs: the observation of ``transition_stateless``."""
        return self.transition_stateless(rows, action)[1]

    def jacobian(self, rows: torch.Tensor, action: torch.Tensor):
        """d(state_out, reward) / d(state_in, action) of ``transition_stateless`` (emei_*_step_jacobian_*):
        -> (jac [b, width, width + 1], reward_grad [b, width + 1]); the last column is the action's."""
        env = self.env
        b, d = rows.shape[0], self.obs_dim
        jac = torch.empty((b, d, d + 1), dtype=env.dtype, device=env.device)
        reward_grad = torch.empty((b, d + 1), dtype=env.dtype, device=env.device)
        self.params.action_kind = _ACTION_KIND[action.dtype]
        env._call(self._jacobian_entry, rows.data_ptr(), action.data_ptr(), jac.data_ptr(), reward_grad.data_ptr(), b,
                  ctypes.byref(self.params), env._stream())
        return jac, reward_grad

    def vjp(self, rows: torch.Tensor, action: torch.Tensor, g_state_out, g_obs, g_reward, want_action: bool):
        """Backward of ``transition_stateless`` (emei_*_step_vjp_*): the cotangents ``g_state_out`` / ``g_obs`` [b, width]
        and ``g_reward`` [b] are contiguous tensors or None (zero).  -> (g_state_in [b, width], g_action [b] or None)."""
        env = self.env
        b = rows.shape[0]
        g_in = torch.empty_like(rows)
        g_act = torch.empty((b,), dtype=env.dtype, device=env.device) if want_action else None
        self.params.action_kind = _ACTION_KIND[action.dtype]
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        env._call(self._vjp_entry, rows.data_ptr(), action.data_ptr(), ptr(g_state_out), ptr(g_obs), ptr(g_reward), g_in.data_ptr(),
                  ptr(g_act), b, ctypes.byref(self.params), env._stream())
        return g_in, g_act

    def trajectory(self, rows: torch.Tensor, actions: torch.Tensor):
        """``T`` open-loop steps of ``transition_stateless`` from rows [b, width] under actions [T, b] in one launch
        (emei_*_trajectory_*) -> (states [T+1, b, width], obs [T, b, width] or None when the family has no separate
        observation, rewards [T, b], dones bool [T, b]); states[0] = rows.  The engine's own state is untouched."""
        env = self.env
        T, b, d = actions.shape[0], rows.shape[0], self.obs_dim
        states = torch.empty((T + 1, b, d), dtype=env.dtype, device=env.device)
        obs = torch.empty((T, b, d), dtype=env.dtype, device=env.device) if self.separate_obs else None
        rewards = torch.empty((T, b), dtype=env.dtype, device=env.device)
        dones = torch.empty((T, b), dtype=torch.uint8, device=env.device)
        if T == 0 or b == 0:
            states.copy_(rows.reshape(1, b, d))
        else:
            self.params.action_kind = _ACTION_KIND[actions.dtype]
            env._call(self._trajectory_entry, rows.data_ptr(), actions.data_ptr(), states.data_ptr(),
                      obs.data_ptr() if obs is not None else None, rewards.data_ptr(), dones.data_ptr(), b, T,
                      ctypes.byref(self.params), env._stream())
        return states, obs, rewards, dones.view(torch.bool)

    def trajectory_vjp(self, states: torch.Tensor, actions: torch.Tensor, g_states, g_obs, g_rewards, want_action: bool):
        """Reverse sweep of ``trajectory`` (emei_*_trajectory_vjp_*): the cotangents ``g_states`` [T+1, b, width],
        ``g_obs`` [T, b, width] and ``g_rewards`` [T, b] are contiguous tensors or None (zero).
        -> (g_state0 [b, width], g_actions [T, b] or None)."""
        env = self.env
        T, b = actions.shape[0], states.shape[1]
        g0 = torch.empty_like(states[0])
        g_act = torch.empty((T, b), dtype=env.dtype, device=env.device) if want_action else None
        if T == 0 or b == 0:
            g0.copy_(g_states[0]) if g_states is not None else g0.zero_()
            if g_act is not None:
                g_act.zero_()
            return g0, g_act
        self.params.action_kind = _ACTION_KIND[actions.dtype]
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        env._call(self._trajectory_vjp_entry, states.data_ptr(), actions.data_ptr(), ptr(g_states), ptr(g_obs), ptr(g_rewards),
                  g0.data_ptr(), ptr(g_act), b, T, ctypes.byref(self.params), env._stream())
        return g0, g_act

    def plan_start(self, state):
        """Start states of a plan -> (rows [B, width] on the device, B, came_from_numpy)."""
        rows, was_np = self.env._to_device(state, self.env.dtype)
        if rows.dim() != 2 or rows.shape[1] != self.obs_dim:
            raise ValueError(f"state must be [B, {self.obs_dim}], got {tuple(rows.shape)}")
        return _aligned16(rows), rows.shape[0], was_np

    def plan_eval(self, rows: torch.Tensor, mean: torch.Tensor, std, candidates: int, q: _lib.PlanParams, want_actions: bool):
        """``_plan_eval`` from start rows [B, width] (``plan_start``)."""
        return self._plan_eval(self._plan_eval_entry, [rows.data_ptr()], mean, std, candidates, q, want_actions)

    def policy_eval(self, rows: torch.Tensor, params: torch.Tensor, H: int, q: _lib.PolicyParams, want_actions: bool):
        """``_policy_eval`` from start rows [E, width] (``plan_start``)."""
        return self._policy_eval(self._policy_eval_entry, [rows.data_ptr()], rows.shape[0], params, H, q, want_actions)


class CartPoleEngine(RowStateEngine):
    """cart-pole family (state = observation) + analytic inverted pendulum (emei_cartpole_step_* / emei_ip_step_noisy_*)."""

    def __init__(self, env, params: _lib.CartPoleParams, separate_obs: bool):
        RowStateEngine.__init__(self, env, params, 4, separate_obs, "emei_cartpole_step", "emei_ip_step_noisy")

    def rollout(self, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, noise=None):
        self._alloc()
        state = self._bufs[self._cur]
        if self.env.dtype == torch.float32 and noise is None:
            return self._rollout("emei_cartpole_rollout_f32", [state.data_ptr()], rp, actions, record, rollout_stats)
        # float64 reference-exact mode / obs_noise_params: the step entry points' own arithmetic, one env per thread
        z = ctypes.byref(noise) if noise is not None else None
        return self._rollout("emei_cartpole_rollout_ref" + self.env._suffix, [state.data_ptr()], rp, actions, record, rollout_stats,
                             extra=(z,))


class I2PEngine(RowStateEngine):
    """analytic inverted double pendulum (emei_i2p_step_*): state [B,6] + observation buffers."""

    def __init__(self, env, params: _lib.I2PParams):
        RowStateEngine.__init__(self, env, params, 6, True, "emei_i2p_step", "emei_i2p_step_noisy")

    def rollout(self, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, noise=None):
        """emei_i2p_rollout_*: the four I2P tasks of zoo/conf/task/BI2P*.yaml through the collection loop of
        zoo/util.py:33-93, one launch; in-kernel resets = reset_model (init_qpos || init_qvel + N(0, sigma))."""
        self._alloc()
        state = self._bufs[self._cur]
        mean, sigma = self.env._init_tables()
        Arr = ctypes.c_double * 6
        z = ctypes.byref(noise) if noise is not None else None
        return self._rollout("emei_i2p_rollout" + self.env._suffix, [state.data_ptr()], rp, actions, record, rollout_stats,
                             extra=(Arr(*mean), Arr(*sigma), z))


class ChargedBallEngine(Engine):
    """charged ball (emei_charged_ball_step_*): three state arrays updated in place."""

    # step_host: the observation is the `free` state array itself, so it needs a copy anyway and kernel-side stores of
    # reward / done alone measured slower than the DMA path (16384 envs: 50.8 us against 41.5)
    zero_copy_ok = False

    def rollout(self, rp: _lib.RolloutParams, actions, record: bool, rollout_stats: torch.Tensor, noise=None):
        entry = "emei_charged_ball_rollout_f32" if self.env.dtype == torch.float32 else "emei_charged_ball_rollout_ref_f64"
        return self._rollout(entry, [self.on_circle.data_ptr(), self.circle.data_ptr(), self.free.data_ptr()], rp, actions, record,
                             rollout_stats)

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

    def _state_arrays(self):
        return [self.on_circle, self.circle, self.free]

    def plan_start(self, state):
        """Start states of a plan, a dict like ``env.state`` or a tuple (on_circle, circle, free) ->
        ((on_circle uint8 [B], circle [B, 2], free [B, 4]) on the device, B, came_from_numpy)."""
        env = self.env
        parts = (state["on_circle"], state["circle_state"], state["free_state"]) if isinstance(state, dict) else tuple(state)
        on, was_np = env._to_device(parts[0], torch.uint8)
        b = on.numel()
        circle = _aligned16(env._to_device(parts[1], env.dtype)[0].reshape(b, 2))
        free = _aligned16(env._to_device(parts[2], env.dtype)[0].reshape(b, 4))
        return (on.reshape(b), circle, free), b, was_np

    def plan_eval(self, state: tuple, mean: torch.Tensor, std, candidates: int, q: _lib.PlanParams, want_actions: bool):
        """``_plan_eval`` from start states (on_circle, circle, free) (``plan_start``)."""
        return self._plan_eval("emei_charged_ball_plan_eval", [t.data_ptr() for t in state], mean, std, candidates, q, want_actions)

    def policy_eval(self, state: tuple, params: torch.Tensor, H: int, q: _lib.PolicyParams, want_actions: bool):
        """``_policy_eval`` from start states (on_circle, circle, free) (``plan_start``)."""
        return self._policy_eval("emei_charged_ball_policy_eval", [t.data_ptr() for t in state], state[0].shape[0], params, H, q,
                                 want_actions)


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """The row loaders use 128-bit accesses: a contiguous view that starts at an odd offset (``obs[k:]`` of 12-byte
    action rows or 72-byte observation rows) is copied to a fresh, aligned allocation (the reference accepts any slice)."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _sumsq(env, a: torch.Tensor, group, entry="emei_sumsq"):
    """batch-wide sum of squared actions (hopper.py:98 / half_cheetah.py:61), all-reduced when the batch is sharded.
    ``entry="emei_sum"``: the plain sum (of the reward cotangents, for the control cost's derivative), same exchange."""
    sumsq = torch.empty(1, dtype=torch.float64, device=env.device)
    ws = getattr(env, "_sumsq_ws", None)
    if ws is None:  # zero-filled once; the kernel leaves its ticket counter at zero
        ws = env._sumsq_ws = torch.zeros(_lib.SUMSQ_WORKSPACE_BYTES // 8, dtype=torch.float64, device=env.device)
    env._call(entry, a.data_ptr(), a.numel(), sumsq.data_ptr(), ws.data_ptr(), env._stream())
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


def needs_grad(*tensors) -> bool:
    """Does a scoring call on these tensors need a differentiable reward (grad mode on, an input requires grad)?"""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def score_rows(env, params: _lib.ScoringParams, o: torch.Tensor, p, a, group):
    """The kernels of one ``score`` pass on device rows: pass 1 (Hopper / HalfCheetah: emei_sumsq_*) and the fused row
    kernel -> (reward [B,1], done bool [B,1]).  ``p`` / ``a`` None for Hopper / HalfCheetah: terminal only."""
    b = o.shape[0]
    needs_pre = params.family in (_lib.HOPPER, _lib.HALFCHEETAH)
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
    return reward, done.view(torch.bool)


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
    With grad mode on and ``obs``, ``pre_obs`` or ``action`` requiring grad, the reward is recorded in the autograd graph
    (``autodiff.RewardScore``: same kernels forward, emei_reward_vjp_* backward) and never served from that cache.
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
    if want != "terminal" and needs_grad(o, p, a):  # a differentiable reward: never served from the cache below
        from .autodiff import RewardScore

        reward, done = RewardScore.apply(o, p, a, env, params, group)
        return reward, done, was_np
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
    reward, done = score_rows(env, params, o, p, a, group)
    if key is not None and not getattr(env, "accumulate_scoring_stats", False):
        env._score_cache = (key, key_obs, _lib.launch_count, reward, done, want)
    return reward, done, was_np


def score_seq(env, params: _lib.ScoringParams, obs_seq, action=None, group=None):
    """Trajectory scoring through emei_reward_terminal_seq_*: ``obs_seq`` [T+1, n, D] (an imagined rollout),
    ``action`` [T, n, A] -> reward [T, n, 1], done bool [T, n, 1].  Equal to ``score`` on
    ``obs = obs_seq[1:], pre_obs = obs_seq[:-1]`` flattened; every observation row is read once.  Differentiable like
    ``score`` (``autodiff.RewardScoreSeq``, backward emei_reward_seq_vjp_*)."""
    family = params.family
    s, was_np = env._to_device(obs_seq, env.dtype)
    d = _lib.lib.emei_family_obs_dim(family)
    if s.dim() != 3 or s.shape[2] != d or s.shape[0] < 1:
        raise ValueError(f"obs_seq must be [T+1, n, {d}], got {tuple(s.shape)}")
    T, n = s.shape[0] - 1, s.shape[1]
    needs_pre = family in (_lib.HOPPER, _lib.HALFCHEETAH)
    a = None
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
    if needs_grad(s, a):
        from .autodiff import RewardScoreSeq

        reward, done = RewardScoreSeq.apply(s, a, env, params, group)
        return reward, done, was_np
    reward, done = score_seq_rows(env, params, s, a, group)
    return reward, done, was_np


def score_seq_rows(env, params: _lib.ScoringParams, s: torch.Tensor, a, group):
    """The kernels of one ``score_seq`` pass on a device trajectory s [T+1, n, D] whose rows keep 16-byte alignment:
    pass 1 (Hopper / HalfCheetah: emei_sumsq_* over a) and emei_reward_terminal_seq_* -> (reward [T,n,1], done bool [T,n,1])."""
    T, n = s.shape[0] - 1, s.shape[1]
    sumsq = None
    if params.family in (_lib.HOPPER, _lib.HALFCHEETAH):
        sumsq = _sumsq(env, _aligned16(a), group)
    s = _aligned16(s)
    reward = torch.empty((T, n, 1), dtype=env.dtype, device=env.device)
    done = torch.empty((T, n, 1), dtype=torch.uint8, device=env.device)
    env._call(
        "emei_reward_terminal_seq", s.data_ptr(), reward.data_ptr(), done.data_ptr(),
        env.stats.data_ptr() if getattr(env, "accumulate_scoring_stats", False) else None,
        sumsq.data_ptr() if sumsq is not None else None, n, T, ctypes.byref(params), env._stream(),
    )
    return reward, done.view(torch.bool)


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
        noise = env._next_obs_noise()
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
