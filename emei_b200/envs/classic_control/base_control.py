"""Batched counterpart of ``emei/envs/classic_control/base_control.py`` (BaseControlEnv, :11-83).

Same constructor keywords (``freq_rate``, ``real_time_scale``, ``integrator``, ``render_mode``) plus
the additive ``num_envs``, ``device``, ``dtype``, ``env_offset``; same ``reset`` / ``step`` /
``freeze`` / ``unfreeze`` contract with ``[num_envs, ...]`` tensors.  The step itself --
``_extract_action`` + ``ODE_approximation`` (forward Euler, :133-164) + ``_dsdt`` + reward/terminal --
is ONE kernel launch (emei_cartpole_step_* / emei_charged_ball_step_*).

Reference quirks handled here (SURVEY.md appendix A):
  * ``integrator`` is accepted and recorded in ``env_params`` but classic control is always forward
    Euler (the reference never forwards it: base_control.py:73 vs :133-135).
  * ``freeze()`` in the reference never sets ``frozen`` (:32-36); here it does (as core.py:23-37 and
    test/test_core.py:17-23 expect), double freeze overwrites the snapshot, and ``unfreeze()``
    without a snapshot raises a clear error instead of AttributeError.
  * rendering (:85-130) is out of scope.
"""
from typing import Optional

import torch

from ...core import EmeiEnv
from ...engine import normalise_action, score


class BaseControlEnv(EmeiEnv):
    metadata = {"render_modes": [], "render_fps": 50}
    _continuous = False

    def __init__(
        self,
        freq_rate: int = 1,
        real_time_scale: float = 0.02,
        integrator: str = "euler",
        render_mode: Optional[str] = None,
        num_envs: int = 1,
        device=None,
        dtype=torch.float32,
        env_offset: int = 0,
        validate_actions: bool = False,
        copy_outputs: bool = True,
    ):
        if render_mode is not None:
            raise NotImplementedError("rendering is outside the emei_b200 hot path")
        self.freq_rate = int(freq_rate)
        self.real_time_scale = float(real_time_scale)
        self.integrator = integrator
        self.render_mode = render_mode
        self.env_offset = int(env_offset)  # global id of env 0 (sharding: keys the Philox streams)
        self.validate_actions = bool(validate_actions)
        # True (default, the reference's contract: base_control.py:47,69,76 return state.copy()): step() returns freshly
        # allocated tensors the caller owns.  False (zero-copy opt-in): step() returns views of the engine's live
        # ping-pong buffers -- valid until the NEXT step() (charged ball: obs is updated in place by it; cart-pole /
        # pendulums: overwritten two steps later), and writing into them corrupts the env state.
        self.copy_outputs = bool(copy_outputs)
        EmeiEnv.__init__(
            self,
            env_params=dict(freq_rate=freq_rate, real_time_scale=real_time_scale, integrator=integrator),
            num_envs=num_envs,
            device=device,
            dtype=dtype,
        )

    # ---- state access -------------------------------------------------------------------------
    @property
    def state(self):
        """[num_envs, 4] device tensor (a view of the live buffer) or None before reset."""
        return self._engine.state if self._engine is not None else None

    @state.setter
    def state(self, value):
        """Host- or device-supplied states (teacher forcing / set_state)."""
        self._ensure_engine().set_state(value)

    # ---- freeze / unfreeze ----------------------------------------------------------------------
    def freeze(self) -> None:
        assert self.state is not None, "Call reset before freezing."
        self.frozen_state = self._engine.snapshot()
        self.frozen = True

    def unfreeze(self) -> None:
        if self.frozen_state is None:
            raise RuntimeError("unfreeze() called before freeze(): there is no snapshot to restore")
        self._engine.restore(self.frozen_state)
        self.frozen = False

    # ---- gym API ----------------------------------------------------------------------------------
    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        self._reseed(seed)
        self.state = self.get_batch_init_state(self.num_envs)
        self._engine.new_episodes(reseed=True)
        return self.state.clone(), {}

    def step(self, action):
        assert self.state is not None, "Call reset before using step method."
        a = normalise_action(self, action, self._continuous, self.num_envs)
        obs, reward, terminal = self._engine.step(a, self.copy_outputs)
        return obs, reward, terminal, False, {}

    # ---- scoring (the reward and terminal of both families depend on obs only) ------------------------
    def get_batch_reward(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        r, _, was_np = score(self, self._scoring_params(), obs)
        return self._ret(r, was_np)

    def get_batch_terminal(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        _, d, was_np = score(self, self._scoring_params(), obs)
        return self._ret(d, was_np)
