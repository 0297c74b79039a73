"""Batched charged-ball envs: counterpart of ``emei/envs/classic_control/charged_ball.py``.

The reference classes cannot be constructed (charged_ball.py:11-12 passes ``time_step=`` to a
constructor without that parameter) and their reward/terminal are scalar (:110-111,158-160); what
is implemented is the semantics of the physics helpers (:25-82), batched, with the state carrying the
``on_circle`` flag explicitly: ``state = (on_circle uint8[B], circle [B,2], free [B,4])`` and the
observation is ``free`` (:96-97).  Constructor keywords follow the reference: ``freq_rate``,
``time_step`` (the reference then overwrites time_step with 0.02, :17 -- replicated).
"""
from ... import _lib, spaces
from ...engine import ChargedBallEngine
from .base_control import BaseControlEnv

import numpy as np


class BaseChargedBallEnv(BaseControlEnv):
    _no_derivatives = "the ball's landing / take-off events (charged_ball.py:62-82) make its step discontinuous"

    def __init__(self, freq_rate=1, time_step=0.02, **kwargs):
        BaseControlEnv.__init__(self, freq_rate=freq_rate, **kwargs)
        # the reference intends env_params = (freq_rate, time_step): charged_ball.py:11-12
        self.env_params = dict(freq_rate=freq_rate, time_step=time_step)
        self.gravity_acc = 9.8
        self.mass_ball = 1.0
        self.radius = 1.0
        self.charge = 10.0
        self.time_step = 0.02  # charged_ball.py:17 (constructor argument is ignored by the reference)
        state_high = np.full(4, np.inf, dtype=np.float32)
        self.observation_space = spaces.Box(-state_high, state_high, dtype=np.float32)
        if self._continuous:
            one = np.ones(1, dtype=np.float32)
            self.action_space = spaces.Box(-one, one, dtype=np.float32)  # charged_ball.py:165-166
        else:
            self.action_space = spaces.Discrete(2)  # charged_ball.py:153
        p = _lib.ChargedBallParams()
        p.gravity_acc, p.mass_ball, p.radius, p.charge = self.gravity_acc, self.mass_ball, self.radius, self.charge
        p.time_step, p.freq_rate = self.time_step, self.freq_rate
        self._engine = ChargedBallEngine(self, p)

    def _scoring_params(self):
        p = _lib.ScoringParams()
        p.family, p.radius = _lib.CHARGED_BALL, self.radius
        return p

    @property
    def state(self):
        """dict(on_circle, circle_state, free_state) of device tensors (views), like the reference's dict."""
        e = self._engine
        if not e.has_state:
            return None
        return dict(on_circle=e.on_circle, circle_state=e.circle, free_state=e.free)

    @state.setter
    def state(self, value):
        self._engine.set_state(value["on_circle"], value["circle_state"], value["free_state"])

    def reset(self, *, seed=None, options=None):
        self._reseed(seed)
        self._engine.sample_initial(self._next_sample_seed(), self.env_offset)  # charged_ball.py:84-94
        self._engine.new_episodes(reseed=True)
        return self._engine.free.clone(), {}

    def _rollout_params(self) -> _lib.RolloutParams:
        rp = _lib.RolloutParams()
        rp.init_kind, rp.init_pi_column = 2, -1  # in-kernel reset = charged_ball.py:84-94
        rp.action_low, rp.action_high = -1.0, 1.0
        return rp

    def get_batch_init_state(self, batch_size):
        tmp = type(self)(freq_rate=self.freq_rate, num_envs=batch_size, device=self.device, dtype=self.dtype,
                         env_offset=self.env_offset)
        tmp._engine.sample_initial(self._next_sample_seed(), self.env_offset)
        return dict(on_circle=tmp._engine.on_circle, circle_state=tmp._engine.circle, free_state=tmp._engine.free)

    def transform_state_to_obs(self, batch_state):
        return batch_state["free_state"].clone()

    def transform_obs_to_state(self, batch_obs):
        raise NotImplementedError("the 4-float observation does not determine on_circle (charged_ball.py:99-108)")


class ChargedBallCenteringEnv(BaseChargedBallEnv):
    pass


class ContinuousChargedBallCenteringEnv(BaseChargedBallEnv):
    _continuous = True
