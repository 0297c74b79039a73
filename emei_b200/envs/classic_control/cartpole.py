"""Batched cart-pole envs: counterpart of ``emei/envs/classic_control/cartpole.py``.

Classes and constants follow the reference (BaseCartPoleEnv :16-46, CartPoleBalancingEnv :115-132,
CartPoleSwingUpEnv :135-156).  The two Continuous* classes are REGISTERED by the reference
(register_env.py:24-33) but never defined there; they are built here from the discrete class and the
continuous-action rule of ContinuousChargedBallCenteringEnv (charged_ball.py:163-170):
``Box(-1, 1, (1,), float32)`` and ``force = force_mag * action[0]`` (SURVEY.md 8(a8)).

dtype=float32 : all-float32 arithmetic (1e-5 rel + 1e-6 abs per step vs the reference).
dtype=float64 : the reference's exact mixed arithmetic (float64 derivative -> float32 -> times
                float32(dt) -> float64 accumulate; cartpole.py:60, base_control.py:164).
"""
import ctypes
import math

import numpy as np
import torch

from ... import _lib, autodiff, spaces
from ...engine import CartPoleEngine, normalise_action, score
from .base_control import BaseControlEnv


class BaseCartPoleEnv(BaseControlEnv):
    _variant = None

    def __init__(self, freq_rate: int = 1, real_time_scale: float = 0.02, integrator: str = "euler", **kwargs):
        super().__init__(freq_rate=freq_rate, real_time_scale=real_time_scale, integrator=integrator, **kwargs)
        # cartpole.py:22-31
        self.gravity = 9.8
        self.mass_cart = 1.0
        self.mass_pole = 0.1
        self.total_mass = self.mass_pole + self.mass_cart
        self.length = 0.5  # half the pole's length
        self.force_mag = 10.0
        self.theta_threshold_radians = 12 * 2 * math.pi / 360
        self.x_threshold = 2.4
        high = np.array(
            [self.x_threshold * 2, np.finfo(np.float32).max, self.theta_threshold_radians * 2, np.finfo(np.float32).max],
            dtype=np.float32,
        )
        if self._continuous:
            one = np.ones(1, dtype=np.float32)
            self.action_space = spaces.Box(-one, one, dtype=np.float32)
        else:
            self.action_space = spaces.Discrete(2)
        self.observation_space = spaces.Box(-high, high, dtype=np.float32)

    # built lazily so subclasses can change constants (x_threshold) in their constructors
    def _params(self) -> _lib.CartPoleParams:
        p = _lib.CartPoleParams()
        p.gravity, p.mass_pole, p.total_mass, p.length = self.gravity, self.mass_pole, self.total_mass, self.length
        p.pole_mass_length = self.mass_pole * self.length  # cartpole.py:51
        p.force_mag = self.force_mag
        p.x_threshold, p.theta_threshold = float(self.x_threshold), self.theta_threshold_radians
        p.dt, p.freq_rate = self.real_time_scale, self.freq_rate  # base_control.py:73
        p.variant = self._variant
        return p

    def _scoring_params(self) -> _lib.ScoringParams:
        p = _lib.ScoringParams()
        p.family = self._variant
        p.x_threshold, p.theta_threshold = float(self.x_threshold), self.theta_threshold_radians
        return p

    def _ensure_engine(self):
        if self._variant is None:
            raise NotImplementedError  # abstract base: reset() raises (test/test_envs/.../test_cartpole.py:4-11)
        if self._engine is None:
            self._engine = CartPoleEngine(self, self._params(), separate_obs=False)
        return self._engine

    def get_batch_init_state(self, batch_size):
        raise NotImplementedError

    _init_pi_column = -1

    def _rollout_params(self) -> _lib.RolloutParams:
        rp = _lib.RolloutParams()
        rp.init_kind, rp.init_pi_column = 0, self._init_pi_column  # cartpole.py:131-132,153-156
        rp.init_low, rp.init_high = -0.05, 0.05
        rp.action_low, rp.action_high = -1.0, 1.0
        return rp

    def _sample_uniform(self, batch_size, pi_column):
        out = torch.empty((batch_size, 4), dtype=self.dtype, device=self.device)
        self._call(
            "emei_init_uniform", out.data_ptr(), batch_size, 4, -0.05, 0.05, pi_column,
            ctypes.c_uint64(self._next_sample_seed()), ctypes.c_uint64(self.env_offset), self._stream(),
        )
        return out

    def get_batch_reward_terminal(self, obs, pre_obs=None, action=None):
        """Additive: both outputs from ONE fused launch."""
        r, d, was_np = score(self, self._scoring_params(), obs)
        return self._ret(r, was_np), self._ret(d, was_np)

    def get_batch_next_obs(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        """core.py:190-193: requires a frozen env; one dynamics step from the given observations."""
        assert self.frozen
        eng = self._ensure_engine()
        o, was_np = self._to_device(obs, self.dtype)
        a = normalise_action(self, action, self._continuous, o.shape[0])
        return self._ret(eng.next_obs_stateless(o, a), was_np)

    def get_batch_transition(self, state, action):
        """One differentiable step from caller rows ``state`` [B,4] (any B; no freeze needed, the env's state, stats and
        buffers are untouched) -> ``(next_state, obs, reward [B,1], done bool [B,1])``, bit-equal to
        ``get_batch_next_obs`` / ``step``.  Records the autograd graph when ``state`` or a continuous ``action`` requires
        grad (backward: emei_cartpole_step_vjp_*).  float64: the gradient is that of the float64 Euler step; the forward
        keeps the reference's float32-rounded increments (DESIGN.md "Derivatives")."""
        return autodiff.transition(self, state, action)

    def get_batch_jacobian(self, state, action):
        """``(jac [B,4,5], reward_grad [B,5])`` = d(next_state, reward) / d(state, action) of the same step; the action
        column is 0 for discrete actions."""
        return autodiff.jacobian(self, state, action)

    def get_batch_trajectory(self, state, actions):
        """T open-loop steps from caller rows ``state`` [B,4] under ``actions`` [T,B] (or [T,B,1]) in one launch ->
        ``(states [T+1,B,4], obs [T,B,4], rewards [T,B], dones bool [T,B])``; states[0] = state, obs = states[1:], and
        step t equals the t-th of T chained ``get_batch_transition`` calls bit for bit.  No resets, noise or statistics: an
        env whose done flag is set keeps being integrated, so mask with ``dones``.  Differentiable w.r.t. ``state`` and a
        continuous ``actions``; the backward is one reverse-sweep launch (emei_cartpole_trajectory_vjp_*)."""
        return autodiff.trajectory(self, state, actions)


class CartPoleBalancingEnv(BaseCartPoleEnv):
    _variant = _lib.CARTPOLE_BALANCING

    def get_batch_init_state(self, batch_size):
        return self._sample_uniform(batch_size, -1)  # cartpole.py:131-132


class CartPoleSwingUpEnv(BaseCartPoleEnv):
    _variant = _lib.CARTPOLE_SWINGUP

    def __init__(self, freq_rate: int = 1, real_time_scale: float = 0.02, integrator: str = "euler", **kwargs):
        super().__init__(freq_rate=freq_rate, real_time_scale=real_time_scale, integrator=integrator, **kwargs)
        self.x_threshold = 5  # cartpole.py:140

    _init_pi_column = 2

    def get_batch_init_state(self, batch_size):
        return self._sample_uniform(batch_size, 2)  # cartpole.py:153-156 (theta += pi)


class ContinuousCartPoleBalancingEnv(CartPoleBalancingEnv):
    _continuous = True


class ContinuousCartPoleSwingUpEnv(CartPoleSwingUpEnv):
    _continuous = True
