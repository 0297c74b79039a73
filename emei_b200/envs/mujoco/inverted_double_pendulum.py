"""Inverted double pendulum: reward / terminal of ``emei/envs/mujoco/inverted_double_pendulum.py``
(:84-90,114-122,150-157,185-196) on 6-d observations ``[x, th1, th2, v, w1, w2]``.

Dynamics: the reference gets its accelerations from MuJoCo's ``mj_step`` (third-party); ``step`` here runs the
reference's own Lagrangian model, ``classic_control/auxiliary/lagrange_eqs.py:12-60`` ``cartpole(2)`` -- cart plus two
thin rods with relative hinge angles -- with the complete potential energy (the script omits the height of pole 1's
hinge for n >= 2, lagrange_eqs.py:45; ``oracle/gen_golden_i2p.py``), the constants of
``assets/inverted_double_pendulum.xml`` and the forward-Euler rule of mujoco_env.py:91-97
(``emei_i2p_step_*``).  Parity against MuJoCo itself is unpinned (thin-rod vs capsule inertia), as for the single
pendulum.  The observation replicates ``current_obs`` (:56-60) including its precedence quirk
``(theta + pi) % 2 * pi - pi``.
Reference quirk kept visible: the 7x6 causal matrix is stored as ``_causal_graph`` (:42), so the
reference's ``get_transition_graph()`` raises; here the matrix is exposed under both names.
"""
import math

import numpy as np
import torch

from ... import _lib
from ...engine import I2PEngine
from .mujoco_env import AnalyticPendulumEnv, EmeiMujocoEnv


class BaseInvertedDoublePendulumEnv(AnalyticPendulumEnv):
    _model = (3, 1, (-1.0, 1.0), [0.0, 0.0, 0.0])  # inverted_double_pendulum.xml:45

    def __init__(self, freq_rate: int = 1, real_time_scale: float = 0.02, integrator="euler",
                 init_noise_params=5e-3, obs_noise_params=0.0, **kwargs):
        EmeiMujocoEnv.__init__(
            self, observation_dim=6, freq_rate=freq_rate, real_time_scale=real_time_scale, integrator=integrator,
            init_noise_params=init_noise_params, obs_noise_params=obs_noise_params, **kwargs,
        )
        self.jnt_range = np.array([[-3.0, 3.0], [-np.inf, np.inf], [-np.inf, np.inf]])  # xml:31
        self._causal_graph = np.array(
            [
                [0, 0, 0, 0, 0, 0],
                [0, 0, 0, 1, 1, 1],
                [0, 0, 0, 1, 1, 1],
                [1, 0, 0, 0, 0, 0],
                [0, 1, 0, 1, 1, 1],
                [0, 0, 1, 1, 1, 1],
                [0, 0, 0, 1, 1, 1],
            ]
        )  # inverted_double_pendulum.py:42-52
        self._transition_graph = self._causal_graph

        # inverted_double_pendulum.xml: gravity (:25), gear (:45), capsule geoms (:32 cart r=0.1 half-len 0.1; :35,:38
        # poles r=0.045, fromto length 0.6) at MuJoCo's default density 1000 kg/m^3
        self.gravity = 9.81
        self.gear = 500.0
        self.mass_cart = 1000.0 * (math.pi * 0.1**2 * 0.2 + 4.0 / 3.0 * math.pi * 0.1**3)
        self.mass_pole = 1000.0 * (math.pi * 0.045**2 * 0.6 + 4.0 / 3.0 * math.pi * 0.045**3)
        self.pole_half_length = 0.3

    def _params(self) -> _lib.I2PParams:
        p = _lib.I2PParams()
        p.gravity, p.mass_cart, p.mass_pole0, p.mass_pole1 = self.gravity, self.mass_cart, self.mass_pole, self.mass_pole
        p.length0 = p.length1 = self.pole_half_length
        p.gear = self.gear
        p.ctrl_low, p.ctrl_high = float(self.action_space.low[0]), float(self.action_space.high[0])
        p.x_left, p.x_right = float(self.jnt_range[0][0]), float(self.jnt_range[0][1])
        p.dt, p.freq_rate, p.variant = self.real_time_scale, self.freq_rate, self._family
        return p

    def _rollout_params(self) -> _lib.RolloutParams:
        rp = _lib.RolloutParams()
        rp.init_kind, rp.init_pi_column = 1, -1  # reset_model: init_qpos/qvel + N(0, sigma) (mujoco_env.py:130-140); 6-d tables travel separately
        rp.action_low, rp.action_high = float(self.action_space.low[0]), float(self.action_space.high[0])
        return rp

    def _new_engine(self):
        return I2PEngine(self, self._params())

    @property
    def current_obs(self):
        """inverted_double_pendulum.py:56-60 (precedence quirk replicated)."""
        s = self.state.clone()
        s[:, 1:3] = torch.remainder(s[:, 1:3] + math.pi, 2) * math.pi - math.pi
        return s

    def _next_obs_rows(self, obs, state):
        """The dynamics need the STATE (qpos||qvel): ``state=`` when given, else ``obs`` holding unwrapped states
        (``current_obs`` is not invertible, :56-60)."""
        return state if state is not None else obs


class ReboundInvertedDoublePendulumBalancingEnv(BaseInvertedDoublePendulumEnv):
    _family = _lib.I2P_REBOUND_BALANCING


class BoundaryInvertedDoublePendulumBalancingEnv(BaseInvertedDoublePendulumEnv):
    _family = _lib.I2P_BOUNDARY_BALANCING


class ReboundInvertedDoublePendulumSwingUpEnv(BaseInvertedDoublePendulumEnv):
    _family = _lib.I2P_REBOUND_SWINGUP


class BoundaryInvertedDoublePendulumSwingUpEnv(BaseInvertedDoublePendulumEnv):
    _family = _lib.I2P_BOUNDARY_SWINGUP
