"""Batched inverted-pendulum envs: counterpart of ``emei/envs/mujoco/inverted_pendulum.py``.

Observation ``[x, theta, v, omega]`` (qpos || qvel), theta wrapped to [-pi, pi) in the observation
only (:45-49); reward / terminal :73-79,103-111,139-146,174-183; transition graph :39-41.

DYNAMICS: the reference steps MuJoCo (``mj_step``), which is not available; the step here is the
reference's own closed-form cart-pole acceleration (classic_control/cartpole.py:48-60 ==
auxiliary/lagrange_eqs.py:12-69) with the constants of assets/inverted_pendulum.xml and the
forward-Euler rule of mujoco_env.py:91-97 -- analytic, NOT MuJoCo-parity (thin-rod inertia, no
joint-limit constraint forces).  Boundary* variants terminate at the rail so the missing
constraint is never active; for Rebound* variants the rail rebound is NOT modelled (the cart passes
|x| = 2): their ``step`` is provided for the scoring path but documented as unconstrained.
"""
import math

import numpy as np
import torch

from ... import _lib
from ...engine import CartPoleEngine
from .mujoco_env import AnalyticPendulumEnv, EmeiMujocoEnv

# capsule volume = pi r^2 L + 4/3 pi r^3 at MuJoCo's default density 1000 kg/m^3
# (inverted_pendulum.xml:15 cart r=0.1 half-length 0.1; :18 pole r=0.049 length 0.6)
_MASS_CART = 1000.0 * (math.pi * 0.1**2 * 0.2 + 4.0 / 3.0 * math.pi * 0.1**3)
_MASS_POLE = 1000.0 * (math.pi * 0.049**2 * 0.6 + 4.0 / 3.0 * math.pi * 0.049**3)


class BaseInvertedPendulumEnv(AnalyticPendulumEnv):
    _model = (2, 1, (-3.0, 3.0), [0.0, 0.0])  # nq, nu, ctrlrange (:23), init_qpos

    def __init__(self, freq_rate: int = 1, real_time_scale: float = 0.02, integrator="euler",
                 init_noise_params=5e-3, obs_noise_params=0.0, **kwargs):
        EmeiMujocoEnv.__init__(
            self, observation_dim=4, freq_rate=freq_rate, real_time_scale=real_time_scale, integrator=integrator,
            init_noise_params=init_noise_params, obs_noise_params=obs_noise_params, **kwargs,
        )
        self.gravity = 9.81  # inverted_pendulum.xml:8
        self.gear = 100.0  # :23
        self.mass_cart, self.mass_pole = _MASS_CART, _MASS_POLE
        self.total_mass = self.mass_pole + self.mass_cart
        self.length = 0.3  # half the pole length
        self.jnt_range = np.array([[-2.0, 2.0], [-math.pi / 2, math.pi / 2]])  # :14,17
        self._update_model()
        self._transition_graph = np.array(
            [[0, 0, 0, 0], [0, 0, 1, 1], [1, 0, 0, 0], [0, 1, 1, 1], [0, 0, 1, 1]]  # x, theta, v, omega, action
        )  # inverted_pendulum.py:39-41

    def _update_model(self):
        pass

    def _params(self) -> _lib.CartPoleParams:
        p = _lib.CartPoleParams()
        p.gravity, p.mass_pole, p.total_mass, p.length = self.gravity, self.mass_pole, self.total_mass, self.length
        p.pole_mass_length = self.mass_pole * self.length
        p.force_mag = self.gear
        p.x_left, p.x_right = float(self.jnt_range[0][0]), float(self.jnt_range[0][1])
        p.ctrl_low, p.ctrl_high = float(self.action_space.low[0]), float(self.action_space.high[0])
        p.dt, p.freq_rate = self.real_time_scale, self.freq_rate
        p.variant = self._family
        return p

    def _rollout_params(self) -> _lib.RolloutParams:
        rp = _lib.RolloutParams()
        rp.init_kind, rp.init_pi_column = 1, -1  # reset_model: init_qpos/qvel + N(0, sigma) (mujoco_env.py:130-140)
        mean, sigma = self._init_tables()
        for j in range(4):
            rp.init_mean[j], rp.init_sigma[j] = float(mean[j]), float(sigma[j])
        rp.action_low, rp.action_high = float(self.action_space.low[0]), float(self.action_space.high[0])
        return rp

    def _new_engine(self):
        return CartPoleEngine(self, self._params(), separate_obs=True)

    @property
    def current_obs(self):
        """inverted_pendulum.py:45-49."""
        s = self.state.clone()
        s[:, 1] = torch.remainder(s[:, 1] + math.pi, 2 * math.pi) - math.pi
        return s


class ReboundInvertedPendulumBalancingEnv(BaseInvertedPendulumEnv):
    _family = _lib.IP_REBOUND_BALANCING


class BoundaryInvertedPendulumBalancingEnv(BaseInvertedPendulumEnv):
    _family = _lib.IP_BOUNDARY_BALANCING


class ReboundInvertedPendulumSwingUpEnv(BaseInvertedPendulumEnv):
    _family = _lib.IP_REBOUND_SWINGUP

    def _update_model(self):
        self.jnt_range[1] = [-np.inf, np.inf]  # inverted_pendulum.py:135-137 (pole body flipped: theta=0 hangs down)


class BoundaryInvertedPendulumSwingUpEnv(BaseInvertedPendulumEnv):
    _family = _lib.IP_BOUNDARY_SWINGUP

    def _update_model(self):
        self.jnt_range[1] = [-np.inf, np.inf]  # inverted_pendulum.py:170-172
