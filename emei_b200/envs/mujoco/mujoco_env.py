"""Batched counterpart of the numpy SHELL of ``emei/envs/mujoco/mujoco_env.py`` (EmeiMujocoEnv).

In scope (SURVEY.md section 2 row 7): constructor keywords, ``dt``, batched Gaussian initial-state
sampling (:137-140,197-249), ``transform_state_to_obs`` / ``transform_obs_to_state`` (:142-151),
freeze semantics (:114-120) and the scoring interface.  Out of scope: ``mujoco.mj_step`` rigid-body
dynamics (third-party C library, un-vendored) -- ``step`` exists only for the inverted pendulums
(``AnalyticPendulumEnv``), whose accelerations have a closed form (classic_control/cartpole.py:48-60).

Reference quirks (SURVEY.md appendix A + DESIGN.md):
  * ``additive_gaussian_noise`` slices ROWS where it means columns (:243-244), so the reference
    raises for batch_size > 1 and adds ONE shared sample to every coordinate for batch_size = 1.
    Implemented here: the evident intent -- an independent N(0, sigma) per coordinate per row.
  * ``transform_obs_to_state`` compares an int with a tuple and always raises (:146-151); here it
    returns ``(obs[:, :nq], obs[:, nq:])``.
  * the noise uses the process-global ``np.random`` (ignores the env seed); here it is a Philox
    stream keyed by ``reset(seed=)``.
  * ``obs_noise_params`` is, despite its name, STATE noise: after every sub-step the simulator state is
    overwritten with ``additive_gaussian_noise(qpos, qvel)`` (:98-104).  Implemented for the analytic
    pendulums (``emei_ip_step_noisy_*`` / ``emei_i2p_step_noisy_*``), same per-coordinate intent as above.
"""
import ctypes
from typing import Dict, Optional, Tuple, Union

import numpy as np
import torch

from ... import _lib, autodiff, spaces
from ...core import EmeiEnv
from ...engine import normalise_action, score, score_seq


class EmeiMujocoEnv(EmeiEnv):
    metadata = {"render_modes": [], "render_fps": 25}

    # subclasses set: (nq, nu, ctrlrange, init_qpos)
    _model = None
    _family = None
    _no_derivatives = "its dynamics are MuJoCo's mj_step, which is outside the emei_b200 hot path"

    def __init__(
        self,
        observation_dim: int,
        freq_rate: int = 1,
        real_time_scale: float = 0.02,
        integrator: str = "euler",
        init_noise_params: Union[float, Tuple[float, float], Dict[int, Tuple[float, float]]] = 5e-3,
        obs_noise_params: Union[float, Tuple[float, float], Dict[int, Tuple[float, float]]] = 0.0,
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
        if integrator not in ("euler", "semi_implicit_euler", "rk4"):
            raise NotImplementedError  # mujoco_env.py:69-78
        self.freq_rate = int(freq_rate)
        self.real_time_scale = float(real_time_scale)
        self.integrator = integrator
        self.init_noise_params = init_noise_params
        self.obs_noise_params = obs_noise_params
        self.env_offset = int(env_offset)
        self.validate_actions = bool(validate_actions)
        self.copy_outputs = bool(copy_outputs)
        EmeiEnv.__init__(
            self,
            env_params=dict(freq_rate=freq_rate, real_time_scale=real_time_scale, integrator=integrator),
            num_envs=num_envs,
            device=device,
            dtype=dtype,
        )
        nq, nu, ctrl, qpos0 = self._model
        self.nq = self.nv = nq
        self.init_qpos = np.array(qpos0, dtype=np.float64)
        self.init_qvel = np.zeros(nq, dtype=np.float64)
        self._noise_step = 0
        self.observation_space = spaces.Box(-np.inf, np.inf, shape=(observation_dim,), dtype=np.float64)
        self.action_space = spaces.Box(ctrl[0], ctrl[1], shape=(nu,), dtype=np.float32)

    @property
    def dt(self):
        """gym MujocoEnv.dt = model.opt.timestep * frame_skip."""
        return self.real_time_scale * self.freq_rate

    # ---- initial states ------------------------------------------------------------------------------
    def _noise_sigmas(self, noise_params):
        """per-coordinate (sigma_pos[nq], sigma_vel[nv]) from scalar / (pos, vel) / {jnt_id: (pos, vel)}
        (mujoco_env.py:217-227; every in-scope model has one coordinate per joint)."""
        sp, sv = np.zeros(self.nq), np.zeros(self.nv)
        if isinstance(noise_params, dict):
            for j, (a, b) in noise_params.items():
                sp[j], sv[j] = a, b
        elif isinstance(noise_params, tuple):
            sp[:], sv[:] = noise_params[0], noise_params[1]
        else:
            sp[:], sv[:] = noise_params, noise_params
        return sp, sv

    # ---- per-sub-step state noise (obs_noise_params, mujoco_env.py:98-104) -------------------------
    def _obs_noise_on(self) -> bool:
        sp, sv = self._noise_sigmas(self.obs_noise_params)
        return bool(np.any(sp != 0) or np.any(sv != 0))

    def _init_tables(self):
        """(mean[nq+nv], sigma[nq+nv]) of reset_model: init_qpos || init_qvel and the per-coordinate init noise."""
        sp, sv = self._noise_sigmas(self.init_noise_params)
        return np.concatenate([self.init_qpos, self.init_qvel]), np.concatenate([sp, sv])

    def _next_obs_noise(self, advance: int = 1) -> Optional[_lib.NoiseParams]:
        """NoiseParams of the NEXT step call (None when obs_noise_params is zero): per-coordinate sigmas
        (scalar / (pos, vel) / {jnt_id: (pos, vel)} forms of mujoco_env.py:217-227), a Philox key derived from
        ``reset(seed=)`` and the env-step counter, which ``reset`` zeroes."""
        if not self._obs_noise_on():
            return None
        sp, sv = self._noise_sigmas(self.obs_noise_params)
        z = _lib.NoiseParams()
        for j, v in enumerate(np.concatenate([sp, sv])):
            z.sigma[j] = float(v)
        z.seed = (self._seed * 0xA24BAED4963EE407 + 0x9FB21C651E98DF25 + max(self._rollout_epoch, 0) * 0x8EBC6AF09C88C6E3) & 0xFFFFFFFFFFFFFFFF
        z.env_offset = self.env_offset
        z.step = self._noise_step
        self._noise_step += int(advance)  # a fused rollout consumes one step index per env step
        return z

    def get_batch_init_state(self, batch_size):
        """-> (pos [B,nq], vel [B,nv]) like mujoco_env.py:137-140."""
        obs = self._sample_init_obs(batch_size)
        return obs[:, : self.nq], obs[:, self.nq :]

    def _sample_init_obs(self, batch_size):
        mean, sigma = self._init_tables()
        d = mean.shape[0]
        out = torch.empty((batch_size, d), dtype=self.dtype, device=self.device)
        Arr = ctypes.c_double * d
        self._call(
            "emei_init_gaussian", out.data_ptr(), batch_size, d, Arr(*mean), Arr(*sigma),
            ctypes.c_uint64(self._next_sample_seed()), ctypes.c_uint64(self.env_offset), self._stream(),
        )
        return out

    def get_batch_init_obs(self, batch_size):
        return self._sample_init_obs(batch_size)  # = concat(pos, vel) (mujoco_env.py:142-144), one launch

    def transform_state_to_obs(self, batch_state):
        pos, vel = batch_state
        if isinstance(pos, torch.Tensor):
            return torch.cat([pos, vel], dim=1)
        return np.concatenate([pos, vel], axis=1)

    def transform_obs_to_state(self, batch_obs):
        assert len(batch_obs.shape) == 2
        if batch_obs.shape[1] == self.nq + self.nv:
            return batch_obs[:, : self.nq], batch_obs[:, self.nq :]
        raise NotImplementedError

    # ---- scoring ---------------------------------------------------------------------------------------
    def _scoring_params(self) -> _lib.ScoringParams:
        p = _lib.ScoringParams()
        p.family = self._family
        p.dt = self.dt
        return p

    def get_batch_reward(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        r, _, was_np = score(self, self._scoring_params(), obs, pre_obs, action, want="reward")
        return self._ret(r, was_np)

    def get_batch_terminal(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        _, d, was_np = score(self, self._scoring_params(), obs, pre_obs, action, want="terminal")
        return self._ret(d, was_np)

    def get_batch_reward_terminal(self, obs, pre_obs=None, action=None):
        """Additive: both outputs from ONE fused row pass (what an MBRL scorer wants)."""
        r, d, was_np = score(self, self._scoring_params(), obs, pre_obs, action, want="both")
        return self._ret(r, was_np), self._ret(d, was_np)

    def get_batch_reward_terminal_seq(self, obs_seq, action=None):
        """Additive: score a whole imagined rollout ``obs_seq`` [T+1, n, D] with ``action`` [T, n, A] ->
        (reward [T, n, 1], terminal bool [T, n, 1]).  Same numbers as ``get_batch_reward`` / ``get_batch_terminal``
        on ``obs = obs_seq[1:]``, ``pre_obs = obs_seq[:-1]`` (hopper.py:95-106, half_cheetah.py:59-67), with every
        observation row read once (emei_reward_terminal_seq_*)."""
        r, d, was_np = score_seq(self, self._scoring_params(), obs_seq, action)
        return self._ret(r, was_np), self._ret(d, was_np)

    # ---- dynamics: only where the reference has a closed form -------------------------------------
    def reset(self, *, seed=None, options=None):
        raise NotImplementedError(
            f"{type(self).__name__}: MuJoCo rigid-body dynamics (mujoco.mj_step) are outside the emei_b200 hot path; "
            "use get_batch_init_obs / get_batch_reward / get_batch_terminal"
        )

    def step(self, action):
        raise NotImplementedError(
            f"{type(self).__name__}: MuJoCo rigid-body dynamics (mujoco.mj_step) are outside the emei_b200 hot path"
        )

    def freeze(self):
        # mujoco_env.py:114-116 (sets the flag, no assert)
        self.frozen = True

    def unfreeze(self):
        self.frozen = False


class AnalyticPendulumEnv(EmeiMujocoEnv):
    """The inverted pendulums, whose accelerations have a closed form: ``reset`` / ``step`` / ``get_batch_next_obs`` /
    ``freeze`` run on the device through the engine that the subclass's ``_new_engine`` builds (forward Euler,
    mujoco_env.py:91-97).  State = qpos || qvel, angles unwrapped."""

    def _ensure_engine(self):
        if self._family is None:
            raise NotImplementedError(f"{type(self).__name__} is abstract")
        if self._engine is None:
            self._engine = self._new_engine()
        return self._engine

    def _scoring_params(self) -> _lib.ScoringParams:
        p = EmeiMujocoEnv._scoring_params(self)
        p.x_left, p.x_right = float(self.jnt_range[0][0]), float(self.jnt_range[0][1])
        return p

    @property
    def state(self):
        return self._engine.state if self._engine is not None else None

    @state.setter
    def state(self, value):
        self._ensure_engine().set_state(value)

    def reset(self, *, seed=None, options=None):
        if self.integrator != "euler":
            raise NotImplementedError(f"{type(self).__name__}: the analytic dynamics implement integrator='euler' (mujoco_env.py:94-97)")
        self._reseed(seed)
        self._noise_step = 0
        self.state = self._sample_init_obs(self.num_envs)  # reset_model: mujoco_env.py:130-135 (returns qpos||qvel)
        self._engine.new_episodes(reseed=True)
        return self.state.clone(), {}

    def step(self, action):
        assert self.state is not None, "Call reset before using step method."
        a = normalise_action(self, action, True, self.num_envs)
        obs, reward, terminal = self._engine.step(a, self.copy_outputs, noise=self._next_obs_noise())
        return obs, reward, terminal, False, {}

    def get_batch_transition(self, state, action):
        """One differentiable step from caller rows ``state`` = qpos || qvel, angles unwrapped (as ``state=`` of
        ``get_batch_next_obs``; any B, no freeze needed, the env's state, stats and buffers are untouched) ->
        ``(next_state, obs, reward [B,1], done bool [B,1])``, bit-equal to ``get_batch_next_obs`` / ``step``.  Records the
        autograd graph when ``state`` or ``action`` requires grad (backward: emei_cartpole_step_vjp_* / emei_i2p_step_vjp_*);
        the action gradient passes the control clamp on [ctrl_low, ctrl_high] only."""
        return autodiff.transition(self, state, action)

    def get_batch_jacobian(self, state, action):
        """``(jac [B,D,D+1], reward_grad [B,D+1])`` = d(next_state, reward) / d(state, action) of the same step."""
        return autodiff.jacobian(self, state, action)

    def get_batch_trajectory(self, state, actions):
        """T open-loop steps from rows ``state`` = qpos || qvel (angles unwrapped) under ``actions`` [T,B] (or [T,B,1]) in
        one launch -> ``(states [T+1,B,D], obs [T,B,D], rewards [T,B], dones bool [T,B])``; states[0] = state, and step t
        equals the t-th of T chained ``get_batch_transition`` calls bit for bit.  No resets, noise or statistics: an env
        whose done flag is set keeps being integrated, so mask with ``dones``.  Differentiable w.r.t. ``state`` and
        ``actions``; the backward is one reverse-sweep launch (emei_cartpole_trajectory_vjp_* / emei_i2p_trajectory_vjp_*)."""
        return autodiff.trajectory(self, state, actions)

    def _next_obs_rows(self, obs, state):
        """The rows get_batch_next_obs steps: ``obs`` (``state=`` is not read)."""
        return obs

    def get_batch_next_obs(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        """core.py:190-193: requires a frozen env; one dynamics step from the given rows, the env does not move."""
        assert self.frozen
        o, was_np = self._to_device(self._next_obs_rows(obs, state), self.dtype)
        a = normalise_action(self, action, True, o.shape[0])
        return self._ret(self._ensure_engine().next_obs_stateless(o, a), was_np)

    def freeze(self):
        self.frozen = True  # mujoco_env.py:114-116: snapshot (qpos, qvel)
        if self.state is not None:
            self.frozen_state = self._engine.snapshot()

    def unfreeze(self):
        self.frozen = False  # mujoco_env.py:118-120
        if self.frozen_state is not None:
            self._engine.restore(self.frozen_state)
