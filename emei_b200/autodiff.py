"""Gradients of the analytic dynamics: ``torch.autograd`` through the step kernels.

The cart-pole family, the analytic inverted pendulum and the analytic inverted double pendulum have closed-form dynamics
(freq_rate forward-Euler sub-steps), so their step is differentiable almost everywhere.  Two entry points serve them:

* ``transition(env, state, action)`` -> ``(next_state, obs, reward [B,1], done bool [B,1])``: the step kernel run
  statelessly on caller rows (outputs bit-equal to ``get_batch_next_obs`` / ``step`` from the same rows), recorded in the
  autograd graph when ``state`` or ``action`` requires grad; its backward is the vector-Jacobian-product kernel
  (``emei_*_step_vjp_*``), which never materialises the Jacobian.  Chaining it T times is backpropagation through time.
* ``jacobian(env, state, action)`` -> ``(jac [B,D,D+1], reward_grad [B,D+1])``: the per-sample Jacobian
  ``d(next_state, reward) / d(state, action)`` (``emei_*_step_jacobian_*``); the last column is the action's.
* ``trajectory(env, state, actions)`` -> ``(states [T+1,B,D], obs [T,B,D], rewards [T,B], dones bool [T,B])``: T open-loop
  steps under actions [T,B] (or [T,B,1]) in one launch (``emei_*_trajectory_*``), bit-equal to T chained ``transition``
  calls; its backward is one reverse-sweep launch (``emei_*_trajectory_vjp_*``) that carries the state cotangent in
  registers.  The shooting / open-loop MPC primitive; a closed-loop policy stays on the chained path.

* Scoring: ``get_batch_reward`` / ``get_batch_reward_terminal`` / ``get_batch_reward_terminal_seq`` of every env record
  their reward in the autograd graph when grad mode is on and ``obs``, ``pre_obs`` or ``action`` requires grad
  (``RewardScore`` / ``RewardScoreSeq``: the scoring kernels forward, ``emei_reward_vjp_*`` / ``emei_reward_seq_vjp_*``
  backward).  Hopper / HalfCheetah's control cost is summed over the whole batch, so every action's gradient is
  ``-2 ctrl_w a`` times the sum G of ALL reward cotangents (``emei_sum_*``); with ``ctrl_cost_scope="global"`` and
  torch.distributed initialised the backward all-reduces G, so every rank must backpropagate through its call (a
  collective, as with DDP).  ``done`` is not differentiable.  Otherwise the call takes the plain path: same launches,
  same bits, no ``grad_fn``.

Semantics of the dynamics (include/emei_b200.h, DESIGN.md "Derivatives"): no state noise; the action gradient passes the control clamp
where ``ctrl_low <= ctrl <= ctrl_high`` and is 0 for discrete actions; the I2P observation's angles have slope pi (the
``current_obs`` precedence quirk).  The float64 cart-pole gradient is that of the float64 Euler step (the forward keeps
the reference's float32-rounded increments).  A continuous action is cast to the env dtype inside the graph, so its
gradient comes back in the caller's dtype and shape (``[B]`` or ``[B,1]``).
"""
import ctypes

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _lib
from .engine import _aligned16, _sumsq, normalise_action, score_rows, score_seq_rows


def _rows(t: torch.Tensor) -> torch.Tensor:
    """contiguous rows at a 16-byte aligned address (the kernels' row loads)"""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _inputs(env, state, action, steps=1):
    """-> (engine, state rows [B, D] in the env dtype, action [steps * B] in its kernel encoding, came_from_numpy).  Every
    conversion is an autograd-tracked op, so gradients flow back to the caller's tensors."""
    eng = env._ensure_engine()
    s, was_np = env._to_device(state, env.dtype)
    if s.dim() != 2 or s.shape[1] != eng.obs_dim:
        raise ValueError(f"state must be [B, {eng.obs_dim}], got {tuple(s.shape)}")
    continuous = len(env.action_space.shape) > 0
    a = normalise_action(env, action, continuous, steps * s.shape[0])
    if continuous:
        a = a.to(env.dtype)
    return eng, s, a, was_np


class StepTransition(torch.autograd.Function):
    """forward: ``RowStateEngine.transition_stateless``; backward: ``RowStateEngine.vjp``."""

    @staticmethod
    def forward(ctx, state, action, engine):
        rows, act = _rows(state.detach()), action.detach().contiguous()
        s_out, obs, reward, done = engine.transition_stateless(rows, act)
        if obs is s_out:  # cart-pole: the observation is the next state; two outputs need two tensors
            obs = s_out.clone()
        ctx.engine = engine
        ctx.save_for_backward(rows, act)
        ctx.mark_non_differentiable(done)
        ctx.set_materialize_grads(False)
        return s_out, obs, reward, done

    @staticmethod
    @once_differentiable
    def backward(ctx, g_state, g_obs, g_reward, g_done):
        rows, act = ctx.saved_tensors
        want_state, want_action = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if g_state is None and g_obs is None and g_reward is None:
            return None, None, None
        g_state = _rows(g_state) if g_state is not None else None
        g_obs = _rows(g_obs) if g_obs is not None else None
        g_reward = g_reward.reshape(-1).contiguous() if g_reward is not None else None
        g_in, g_act = ctx.engine.vjp(rows, act, g_state, g_obs, g_reward, want_action)
        return (g_in if want_state else None), g_act, None


def transition(env, state, action):
    """``env.get_batch_transition``: see the module docstring."""
    eng, s, a, was_np = _inputs(env, state, action)
    out = StepTransition.apply(s, a, eng)
    return tuple(env._ret(t, was_np) for t in out) if was_np else out


def jacobian(env, state, action):
    """``env.get_batch_jacobian``: see the module docstring."""
    eng, s, a, was_np = _inputs(env, state, action)
    with torch.no_grad():
        jac, reward_grad = eng.jacobian(_rows(s.detach()), a.detach().contiguous())
    return env._ret(jac, was_np), env._ret(reward_grad, was_np)


class StepTrajectory(torch.autograd.Function):
    """forward: ``RowStateEngine.trajectory``; backward: ``RowStateEngine.trajectory_vjp``.  ``obs`` is None for the
    cart-pole envs, whose observation is the next state (``trajectory`` returns ``states[1:]`` for it)."""

    @staticmethod
    def forward(ctx, state, actions, engine):
        rows, act = _rows(state.detach()), actions.detach().contiguous()
        states, obs, rewards, dones = engine.trajectory(rows, act)
        ctx.engine = engine
        ctx.save_for_backward(states, act)
        ctx.mark_non_differentiable(dones)
        ctx.set_materialize_grads(False)
        return states, obs, rewards, dones

    @staticmethod
    @once_differentiable
    def backward(ctx, g_states, g_obs, g_rewards, g_dones):
        states, act = ctx.saved_tensors
        want_state, want_action = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if g_states is None and g_obs is None and g_rewards is None:
            return None, None, None
        g_states = _rows(g_states) if g_states is not None else None
        g_obs = _rows(g_obs) if g_obs is not None else None
        g_rewards = g_rewards.contiguous() if g_rewards is not None else None
        g0, g_act = ctx.engine.trajectory_vjp(states, act, g_states, g_obs, g_rewards, want_action)
        return (g0 if want_state else None), g_act, None


def trajectory(env, state, actions):
    """``env.get_batch_trajectory``: see the module docstring."""
    shape = tuple(actions.shape) if isinstance(actions, torch.Tensor) else np.shape(actions)
    B = len(state)
    if len(shape) not in (2, 3) or shape[1:] not in ((B,), (B, 1)):
        raise ValueError(f"actions must be [T, B={B}] or [T, B, 1], got shape {shape}")
    eng, s, a, was_np = _inputs(env, state, actions, steps=shape[0])
    states, obs, rewards, dones = StepTrajectory.apply(s, a.reshape(shape[0], B), eng)
    if obs is None:  # cart-pole: the observation is the next state; autograd routes its gradient into states
        obs = states[1:]
    out = (states, obs, rewards, dones)
    return tuple(env._ret(t, was_np) for t in out) if was_np else out


# ---------------------------------------------------------------------------------------------------------------------
# scoring
# ---------------------------------------------------------------------------------------------------------------------
_MUJOCO = (_lib.HOPPER, _lib.HALFCHEETAH)


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _grad_inputs(env, params, obs, action, want_action, rows, group):
    """-> (obs pointer source or None, action rows or None, G or None): the obs rows only where the family's derivative
    reads them (not Hopper / HalfCheetah's), and G = the all-reduced sum of the reward cotangents ``rows`` when the
    action gradient is wanted (one 8-byte all-reduce with ``ctrl_cost_scope="global"``, as the forward's sum of squares)."""
    mj = params.family in _MUJOCO
    g_sum = _sumsq(env, rows, group, entry="emei_sum") if want_action else None
    return (None if mj else _aligned16(obs)), (_aligned16(action) if want_action else None), g_sum


def _check_action_width(params, a, rows: int):
    if params.family in _MUJOCO and a is not None:
        width = _lib.lib.emei_family_action_dim(params.family)
        if a.numel() != rows * width:
            raise ValueError(f"a differentiable reward needs actions of width {width}, got shape {tuple(a.shape)}")


class RewardScore(torch.autograd.Function):
    """forward: ``engine.score_rows`` (the scoring kernels of ``engine.score``); backward: ``emei_reward_vjp_*``."""

    @staticmethod
    def forward(ctx, obs, pre_obs, action, env, params, group):
        _check_action_width(params, action, obs.shape[0])
        reward, done = score_rows(env, params, obs, pre_obs, action, group)
        ctx.env, ctx.params, ctx.group = env, params, group
        ctx.save_for_backward(obs, action)
        ctx.mark_non_differentiable(done)
        ctx.set_materialize_grads(False)
        return reward, done

    @staticmethod
    @once_differentiable
    def backward(ctx, g_reward, g_done):
        if g_reward is None:
            return None, None, None, None, None, None
        env, params = ctx.env, ctx.params
        obs, action = ctx.saved_tensors
        want_o, want_p, want_a = ctx.needs_input_grad[:3]
        b = obs.shape[0]
        g = _aligned16(g_reward.reshape(b).contiguous())
        o, a, g_sum = _grad_inputs(env, params, obs, action, want_a, g, ctx.group)
        g_obs = torch.empty_like(obs) if want_o else None
        g_pre = torch.empty_like(obs) if want_p else None
        g_act = torch.empty_like(action) if want_a else None
        launches = int(want_o or want_p) + int(want_a)
        env._call("emei_reward_vjp", _ptr(o), _ptr(a), g.data_ptr(), _ptr(g_sum), _ptr(g_obs), _ptr(g_pre), _ptr(g_act), b,
                  ctypes.byref(params), env._stream(), launches=launches)
        return g_obs, g_pre, g_act, None, None, None


class RewardScoreSeq(torch.autograd.Function):
    """forward: ``engine.score_seq_rows`` (emei_reward_terminal_seq_*); backward: ``emei_reward_seq_vjp_*``, which writes
    every row of d/d obs_seq once (row t: transition t-1's obs term + transition t's pre_obs term)."""

    @staticmethod
    def forward(ctx, obs_seq, action, env, params, group):
        T, n = obs_seq.shape[0] - 1, obs_seq.shape[1]
        _check_action_width(params, action, T * n)
        reward, done = score_seq_rows(env, params, obs_seq, action, group)
        ctx.env, ctx.params, ctx.group = env, params, group
        ctx.save_for_backward(obs_seq, action)
        ctx.mark_non_differentiable(done)
        ctx.set_materialize_grads(False)
        return reward, done

    @staticmethod
    @once_differentiable
    def backward(ctx, g_reward, g_done):
        if g_reward is None:
            return None, None, None, None, None
        env, params = ctx.env, ctx.params
        obs_seq, action = ctx.saved_tensors
        want_s, want_a = ctx.needs_input_grad[:2]
        T, n = obs_seq.shape[0] - 1, obs_seq.shape[1]
        g = _aligned16(g_reward.reshape(T, n).contiguous())
        s, a, g_sum = _grad_inputs(env, params, obs_seq, action, want_a, g, ctx.group)
        # every row is written by the kernel; an empty trajectory launches nothing, so its one row is zero-filled here
        g_seq = (torch.empty_like if T and n else torch.zeros_like)(obs_seq)
        g_act = torch.empty_like(action) if want_a else None
        env._call("emei_reward_seq_vjp", _ptr(s), _ptr(a), g.data_ptr(), _ptr(g_sum), g_seq.data_ptr(), _ptr(g_act), n, T,
                  ctypes.byref(params), env._stream(), launches=1 + int(want_a))
        return (g_seq if want_s else None), g_act, None, None, None
