"""Batched, device-resident counterpart of the reference's API contract ``emei/core.py``.

Mirrors ``Freezable`` (core.py:18-37) and ``EmeiEnv`` (core.py:131-193): same method names,
argument meaning and error behaviour, with arrays generalised to ``[num_envs, dim]`` CUDA tensors.
numpy inputs are accepted everywhere (copied to the device; results come back as numpy), so code
written against the reference's ``get_batch_*`` keeps working unchanged.

``OfflineEnv`` (core.py:40-128): datasets are read from the reference's local cache layout
(``emei_b200.offline``); the download step (``urllib``, core.py:94-107) is out of scope -- there is no network --
so ``dataset_names`` lists what is on disk and ``get_dataset`` raises for anything that is not.
"""
from collections import namedtuple
from typing import Dict, Union

import numpy as np
import torch

from . import _lib
from .engine import HostStaging, action_rule


class Freezable:
    """core.py:18-37."""

    def __init__(self):
        self.frozen_state = None
        self.frozen = False

    def freeze(self):
        assert not self.frozen, "env has frozen"
        self.frozen = True

    def unfreeze(self):
        assert self.frozen, "env has unfrozen"
        self.frozen = False

PlanResult = namedtuple("PlanResult", "mean std best_actions best_return returns")
PlanResult.__doc__ = """Result of ``EmeiEnv.plan``: the refitted plan distribution ``mean`` / ``std`` [H, B] (``std`` None for discrete
actions, whose ``mean`` is the probability of action 1), the best candidate of the last iteration (``best_actions`` [H, B],
``best_return`` [B] float64) and that iteration's ``returns`` [B, K] (float64)."""

_M64 = 0xFFFFFFFFFFFFFFFF


def plan_iteration_seed(seed: int, i: int) -> int:
    """The Philox key of iteration ``i`` of a plan keyed by ``seed``."""
    return (seed * 0xD1B54A32D192ED03 + (i + 1) * 0x9E3779B97F4A7C15) & _M64

PolicySearchResult = namedtuple("PolicySearchResult", "theta returns stats")
PolicySearchResult.__doc__ = """Result of ``EmeiEnv.policy_search``: the linear policy ``theta`` [P] (float64, P = observation dimension + 1:
the weights, then the bias), the last iteration's ``returns`` [2N, E] (float64; rows 2k / 2k + 1: theta +- noise delta_k) and
per iteration ``stats`` [iterations, 4] (float64): the number of directions stepped along, the std of their returns, the best
direction's max(r+, r-) and the mean of every finite direction return (NaN where there is none)."""


def policy_starts_seed(seed: int) -> int:
    """The Philox key of the start states an iteration keyed by ``seed`` draws (``policy_search``, and
    ``get_batch_policy_returns`` with ``starts=None``)."""
    return (seed * 0x9E3779B97F4A7C15 + 0xBF58476D1CE4E5B9) & _M64


def _torch_dtype(dtype) -> torch.dtype:
    if isinstance(dtype, torch.dtype):
        out = dtype
    else:
        out = {"float32": torch.float32, "float64": torch.float64}[np.dtype(dtype).name]
    if out not in (torch.float32, torch.float64):
        raise ValueError("emei_b200 computes in float32 or float64")
    return out


class EmeiEnv(Freezable):
    """core.py:131-193, batched.  ``num_envs`` environments live in one set of device buffers."""

    def __init__(
        self,
        env_params: Dict[str, Union[str, int, float]],
        num_envs: int = 1,
        device: Union[str, torch.device, None] = None,
        dtype=torch.float32,
    ):
        Freezable.__init__(self)
        self.env_name = self.__class__.__name__[:-3]  # core.py:42
        self.env_params = env_params
        self.num_envs = int(num_envs)
        if self.num_envs < 1:
            raise ValueError("num_envs must be >= 1")
        self._device_arg = device
        self._device = None
        self.dtype = _torch_dtype(dtype)
        self._suffix = "_f32" if self.dtype == torch.float32 else "_f64"
        self._transition_graph = None
        self._reward_mech_graph = None
        self._termination_mech_graph = None
        self._stats = None
        self._seed = 0
        self._reset_count = 0
        self._plan_count = 0  # planner calls since the last explicit seed: keys plan() / get_batch_plan_returns with seed=None
        self._policy_count = 0  # unseeded policy-search calls since the last explicit seed (policy_search / get_batch_policy_returns)
        self._sample_key = None  # set: the Philox key of the next initial-state draw instead of the reset stream's (_policy_starts)
        self._rollout_epoch = -1  # resets since the last explicit seed (0 = the seeded one): keys the rollout / noise streams

    # ------------------------------------------------------------------ engine protocol (engine.py)
    _engine = None  # the device-buffer owner of an env with a step kernel

    def _ensure_engine(self):
        """The env's engine, built on first use where the subclass builds it lazily; None: no dynamics kernel."""
        return self._engine

    def _next_obs_noise(self, advance: int = 1):
        """NoiseParams of the next step call (obs_noise_params), or None: no state noise."""
        return None

    # ------------------------------------------------------------------ device plumbing
    @property
    def device(self) -> torch.device:
        if self._device is None:
            if not torch.cuda.is_available():
                raise _lib.EmeiB200Error("emei_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
            d = torch.device("cuda", torch.cuda.current_device()) if self._device_arg is None else torch.device(self._device_arg)
            if d.type != "cuda":
                raise _lib.EmeiB200Error(f"emei_b200 runs on CUDA devices only, got {d}")
            if d.index is None:
                d = torch.device("cuda", torch.cuda.current_device())
            self._device = d
        return self._device

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _to_device(self, x, dtype=None, non_blocking=True):
        """-> (contiguous device tensor, came_from_host_numpy)."""
        if x is None:
            return None, False
        was_np = not isinstance(x, torch.Tensor)
        t = torch.as_tensor(x) if was_np else x
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        if t.device != self.device:
            t = t.to(self.device, non_blocking=non_blocking)
        return t.contiguous(), was_np

    @staticmethod
    def _ret(t: torch.Tensor, as_numpy: bool):
        return t.cpu().numpy() if as_numpy else t

    def _call(self, base: str, *args, launches=1):
        with torch.cuda.device(self.device):
            _lib.call(base + self._suffix, *args, launches=launches)

    # ------------------------------------------------------------------ statistics (rollout returns)
    @property
    def stats(self) -> torch.Tensor:
        """device double[2] = [sum of rewards, number of done flags] accumulated by every kernel call."""
        if self._stats is None:
            self._stats = torch.zeros(2, dtype=torch.float64, device=self.device)
        return self._stats

    def reset_stats(self):
        with torch.cuda.device(self.device):
            _lib.call("emei_stats_reset", self.stats.data_ptr(), self._stream(), launches=0)

    def read_stats(self, group=None):
        """(return_sum, done_count) over ALL ranks of ``group`` when torch.distributed is initialised
        (one NCCL all-reduce of 2 doubles), else over this process."""
        from .dist import all_reduce_sum_

        s = all_reduce_sum_(self.stats.clone(), group)
        r, d = s.tolist()
        return r, int(round(d))

    # ------------------------------------------------------------------ core.py contract
    @property
    def dataset_names(self) -> list:
        """core.py:52-54: the names known for this env / parameter set -- here, the files present in the
        reference's cache directory (core.py:83-92)."""
        from . import offline

        d = offline.dataset_path(self, "")
        return sorted(p.name for p in d.iterdir() if p.suffix in (".h5", ".hdf5", ".npz")) if d.is_dir() else []

    def get_dataset(self, dataset_name: str):
        """core.py:109-128 without the download (no network): loads ``DATASET_PATH/<env_name>/<env_params_name>/
        <dataset_name>`` (.h5 needs h5py; .npz always works) and runs the reference's key checks."""
        from . import offline

        path = offline.dataset_path(self, dataset_name)
        if not path.exists():
            raise FileNotFoundError(f"{path} does not exist and emei_b200 does not download datasets (core.py:94-107)")
        return offline.load_dataset(path)

    @property
    def env_params_name(self):
        # core.py:56-58
        return "&".join("{}={}".format(key, self.env_params[key]) for key in sorted(self.env_params.keys()))

    def get_transition_graph(self, repeat_times=1):
        """core.py:142-161.  Envs without a graph raise AttributeError in the reference
        (``None.copy()``); here the error says why."""
        if self._transition_graph is None:
            raise AttributeError(f"{type(self).__name__} defines no transition graph (the reference has none for it)")
        g = self._transition_graph.copy()
        num_obs, num_action = self.observation_space.shape[0], self.action_space.shape[0]
        assert g.shape == (num_obs + num_action, num_obs)
        if repeat_times == 1:
            return g
        n = num_obs + num_action
        aug_g = np.zeros([n, n])
        aug_g[:, :num_obs] = g
        prod_g, sum_g = aug_g.copy(), np.zeros([n, n])
        for _ in range(repeat_times):
            sum_g += prod_g
            prod_g = np.matmul(prod_g, aug_g)
        return (sum_g > 0).astype(int)[:, :num_obs]

    def get_reward_mech_graph(self):
        return self._reward_mech_graph

    def get_termination_mech_graph(self):
        return self._termination_mech_graph

    def transform_state_to_obs(self, batch_state):
        return batch_state.clone() if isinstance(batch_state, torch.Tensor) else np.array(batch_state, copy=True)

    def transform_obs_to_state(self, batch_obs):
        return batch_obs.clone() if isinstance(batch_obs, torch.Tensor) else np.array(batch_obs, copy=True)

    def get_batch_init_state(self, batch_size):
        raise NotImplementedError

    def get_batch_init_obs(self, batch_size):
        return self.transform_state_to_obs(self.get_batch_init_state(batch_size=batch_size))

    def get_batch_reward(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        raise NotImplementedError

    def get_batch_terminal(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        raise NotImplementedError

    def get_batch_next_obs(self, obs, pre_obs=None, action=None, state=None, pre_state=None):
        assert self.frozen
        raise NotImplementedError

    # ------------------------------------------------------------------ derivatives (autodiff.py)
    _no_derivatives = "it has no differentiable dynamics kernel"  # why get_batch_transition / get_batch_jacobian raise

    def get_batch_transition(self, state, action):
        """Differentiable stateless step ``(next_state, obs, reward [B,1], done bool [B,1])``: the analytic families only."""
        raise NotImplementedError(f"{type(self).__name__}: no gradients, {self._no_derivatives}")

    def get_batch_jacobian(self, state, action):
        """``(jac [B,D,D+1], reward_grad [B,D+1])`` of the step: the analytic families only."""
        raise NotImplementedError(f"{type(self).__name__}: no Jacobian, {self._no_derivatives}")

    def get_batch_trajectory(self, state, actions):
        """Differentiable open-loop trajectory ``(states [T+1,B,D], obs [T,B,D], rewards [T,B], dones bool [T,B])`` of
        actions [T,B]: the analytic families only."""
        raise NotImplementedError(f"{type(self).__name__}: no gradients, {self._no_derivatives}")

    # ------------------------------------------------------------------ sampling-based planning (CEM / MPPI)
    def _plan_setup(self, state):
        """-> (engine, device start states, B, came_from_numpy, PlanParams with the action kind, box and env_offset)."""
        eng = self._ensure_engine()
        if eng is None or not hasattr(eng, "plan_eval"):
            raise NotImplementedError(f"{type(self).__name__}: no planning, it has no dynamics kernel")
        if state is None:
            assert self.state is not None, "Call reset before planning from the env's state."
            state = self.state
        start, b, was_np = eng.plan_start(state)
        q = _lib.PlanParams()
        q.env_offset = int(getattr(self, "env_offset", 0))
        q.method, q.elites, q.temperature = _lib.PLAN_CEM, 1, 1.0
        if len(self.action_space.shape) == 0:
            q.action_kind = _lib.ACTION_DISCRETE_U8
        else:
            q.action_kind = _lib.ACTION_CONTINUOUS_F32 if self.dtype == torch.float32 else _lib.ACTION_CONTINUOUS_F64
            q.action_low, q.action_high = float(self.action_space.low.min()), float(self.action_space.high.max())
        return eng, start, b, was_np, q

    def _plan_table(self, x, b: int, what: str, horizon=None) -> torch.Tensor:
        """mean / std as a fresh contiguous device tensor [H, B] in the env dtype ([H] is broadcast over the starts)."""
        t, _ = self._to_device(x, self.dtype)
        if t.dim() == 1:
            t = t.reshape(-1, 1).expand(t.shape[0], b)
        if t.dim() != 2 or t.shape[1] != b or (horizon is not None and t.shape[0] != horizon):
            raise ValueError(f"{what} must be [H, B={b}] or [H], got {tuple(t.shape)}")
        return t.clone(memory_format=torch.contiguous_format)

    def get_batch_plan_returns(self, state, mean, std, candidates: int, seed=None, gamma: float = 1.0, return_actions: bool = False):
        """Score ``candidates`` action sequences per start state in one launch: candidate k of start b draws its actions
        around ``mean`` / ``std`` [H, B] (discrete actions: ``mean`` is the probability of action 1, ``std`` is unused) from
        the counter-based stream of (``seed``, start, k) and is rolled out open-loop for H steps with the step arithmetic of
        ``rollout()``.  -> ``returns`` [B, K] float64, the discounted sum of rewards up to and including the step that
        terminates; with ``return_actions`` also the actions [H, B, K] (``actions.view(H, B*K)`` teacher-forces a rollout of
        the candidates).  ``state``: start rows [B, D] (qpos || qvel, angles unwrapped, for the pendulums) or the charged
        ball's state dict; ``seed=None`` draws a fresh key from the env's seed and a planner call counter of its own.  The
        env's state, statistics and initial-state stream are not touched."""
        eng, start, b, was_np, q = self._plan_setup(state)
        discrete = q.action_kind == _lib.ACTION_DISCRETE_U8
        m = self._plan_table(mean, b, "mean")
        s = None if discrete else self._plan_table(std, b, "std", m.shape[0])
        q.seed = self._next_plan_seed() if seed is None else int(seed) & _M64
        q.gamma = float(gamma)
        returns, actions = eng.plan_eval(start, m, s, int(candidates), q, bool(return_actions))
        if return_actions:
            return self._ret(returns, was_np), self._ret(actions, was_np)
        return self._ret(returns, was_np)

    def plan(self, horizon: int, candidates: int = 512, iterations: int = 5, method: str = "cem", elites: int = 64,
             temperature: float = 1.0, momentum: float = 0.1, gamma: float = 1.0, mean=None, std=None, min_std: float = 0.0,
             state=None, seed=None) -> PlanResult:
        """Sampling-based MPC over the env's own dynamics (the loop of PETS / PlaNet / TD-MPC with the true model):
        ``iterations`` x (score ``candidates`` sequences of ``horizon`` steps per start state, refit the plan distribution),
        two launches per iteration.  ``method``: "cem" (refit to the ``elites`` best) or "mppi" (exponential weights with
        ``temperature``); then ``mean <- momentum mean + (1 - momentum) fit`` and ``std <- max(momentum std + (1 - momentum)
        fit_std, min_std)``.  ``mean`` / ``std`` [H, B] warm-start the plan (default: the centre of the action box and a
        quarter of its width; discrete actions: probability 0.5); they are not modified.  ``state=None`` plans from the env's
        live state (after ``reset()``); ``seed=None`` draws a fresh key from the env's seed and a planner call counter of its own
        (a later unseeded ``reset()`` draws the same start states with or without planning), iteration i uses
        ``plan_iteration_seed(seed, i)``.  numpy start states give numpy results.  -> ``PlanResult``."""
        eng, start, b, was_np, q = self._plan_setup(state)
        H, iters = int(horizon), int(iterations)
        if H < 1 or iters < 1:
            raise ValueError("horizon and iterations must be >= 1")
        discrete = q.action_kind == _lib.ACTION_DISCRETE_U8
        lo, hi = (0.0, 1.0) if discrete else (q.action_low, q.action_high)
        m = self._plan_table(mean, b, "mean", H) if mean is not None else torch.full((H, b), 0.5 * (lo + hi), dtype=self.dtype,
                                                                                       device=self.device)
        s = None
        if not discrete:
            s = self._plan_table(std, b, "std", H) if std is not None else torch.full((H, b), 0.25 * (hi - lo), dtype=self.dtype,
                                                                                      device=self.device)
        methods = {"cem": _lib.PLAN_CEM, "mppi": _lib.PLAN_MPPI}
        if method not in methods:
            raise ValueError(f"method must be 'cem' or 'mppi', got {method!r}")
        q.method, q.elites, q.temperature = methods[method], int(elites), float(temperature)
        q.momentum, q.min_std, q.gamma = float(momentum), float(min_std), float(gamma)
        base = self._next_plan_seed() if seed is None else int(seed) & _M64
        for i in range(iters):
            q.seed = plan_iteration_seed(base, i)
            returns, _ = eng.plan_eval(start, m, s, int(candidates), q, False)
            best_a, best_r = eng.plan_update(returns, m, s, q, want_best=i == iters - 1)
        r = lambda t: self._ret(t, was_np) if t is not None else None  # noqa: E731
        return PlanResult(r(m), r(s), r(best_a), r(best_r), r(returns))

    # ------------------------------------------------------------------ policy search (linear feedback policies, ARS)
    def _policy_setup(self):
        """-> (engine, P, PolicyParams with the action kind and box)."""
        eng = self._ensure_engine()
        if eng is None or not hasattr(eng, "policy_eval"):
            raise NotImplementedError(f"{type(self).__name__}: no policy search, it has no dynamics kernel")
        q = _lib.PolicyParams()
        if len(self.action_space.shape) == 0:
            q.action_kind = _lib.ACTION_DISCRETE_U8
        else:
            q.action_kind = _lib.ACTION_CONTINUOUS_F32 if self.dtype == torch.float32 else _lib.ACTION_CONTINUOUS_F64
            q.action_low, q.action_high = float(self.action_space.low.min()), float(self.action_space.high.max())
        return eng, int(self.observation_space.shape[0]) + 1, q

    def _policy_starts(self, n: int, key: int):
        """``n`` start states from the env's initial-state distribution under Philox key ``key``, in the layout ``plan_start``
        takes; the reset stream's counter does not move."""
        self._sample_key = key
        try:
            return self._sample_init_obs(n) if hasattr(self, "_sample_init_obs") else self.get_batch_init_state(n)
        finally:
            self._sample_key = None

    def _policy_horizon(self, horizon) -> int:
        H = getattr(self, "max_episode_steps", None) if horizon is None else horizon
        if H is None or int(H) < 1:
            raise ValueError("horizon must be >= 1 (None: the env's max_episode_steps)")
        return int(H)

    def get_batch_policy_returns(self, params, starts=None, horizon=None, gamma: float = 1.0, seed=None, return_actions: bool = False):
        """Closed-loop returns of linear feedback policies in one launch: policy c, ``params[c] = (w_0 .. w_{D-1}, b)`` (float64
        [C, P] or [P], P = observation dimension + 1), acts ``u = b + sum_j w_j obs_j`` on the observation ``step()`` would
        return (continuous actions: u clamped to the action box; discrete: ``u > 0``) from each of E start states for
        ``horizon`` steps (None: ``max_episode_steps``) with the step arithmetic of ``rollout()``.  -> ``returns`` [C, E]
        float64, the discounted sum of rewards up to and including the step that terminates; with ``return_actions`` also
        the actions [H, C, E] (``actions.view(H, C*E)`` teacher-forces a rollout of the pairs, candidate-major).
        ``starts``: start rows [E, D] (qpos || qvel with unwrapped angles, for the pendulums) or the charged ball's state dict;
        None draws ``num_envs`` starts from the initial-state distribution, keyed by ``seed`` (None: a counter of the policy
        search's own, so a later unseeded ``reset()`` draws the same states).  The env's state, statistics and initial-state
        stream are not touched.  numpy in, numpy out."""
        eng, P, q = self._policy_setup()
        th, was_np = self._to_device(params, torch.float64)
        th = th.reshape(1, -1) if th.dim() == 1 else th
        if th.dim() != 2 or th.shape[1] != P:
            raise ValueError(f"params must be [C, {P}] or [{P}], got {tuple(th.shape)}")
        H = self._policy_horizon(horizon)
        if starts is None:
            key = self._next_policy_seed() if seed is None else int(seed) & _M64
            starts = self._policy_starts(self.num_envs, policy_starts_seed(key))
        start, _, st_np = eng.plan_start(starts)
        q.gamma = float(gamma)
        returns, actions = eng.policy_eval(start, th, H, q, bool(return_actions))
        as_np = was_np or st_np
        if return_actions:
            return self._ret(returns, as_np), self._ret(actions, as_np)
        return self._ret(returns, as_np)

    def policy_search(self, horizon=None, iterations: int = 20, directions: int = 32, top=None, step_size: float = 0.02,
                      noise: float = 0.03, episodes: int = 16, gamma: float = 1.0, theta=None, seed=None) -> PolicySearchResult:
        """Random search over linear feedback policies (ARS V1-t, Mania, Guy & Recht 2018) on the env's own dynamics.  Each
        of ``iterations`` draws ``episodes`` fresh start states from the initial-state distribution, perturbs ``theta``
        along ``directions`` Gaussian directions (theta +- ``noise`` delta_k), scores the 2N policies closed loop for
        ``horizon`` steps (None: ``max_episode_steps``) from those starts (the mean discounted return over the episodes),
        and steps ``theta += step_size / (b sigma_R) sum (r_k+ - r_k-) delta_k`` along the ``top`` (None: all) best
        directions, sigma_R being the std of their returns.  Four launches per iteration, no host synchronisation.
        ``theta`` [P] warm-starts the search (default 0) and is not modified; ``seed=None`` draws a fresh key from the env's
        seed and a counter of the search's own (a later unseeded ``reset()`` draws the same start states with or without a
        search); iteration i is keyed by ``plan_iteration_seed(seed, i)``.  -> ``PolicySearchResult``; numpy ``theta`` in,
        numpy out."""
        eng, P, q = self._policy_setup()
        H, iters, N = self._policy_horizon(horizon), int(iterations), int(directions)
        E = int(episodes)
        if iters < 1 or E < 1:
            raise ValueError("iterations and episodes must be >= 1")
        if not 1 <= N <= _lib.POLICY_MAX_DIRECTIONS:
            raise ValueError(f"directions must be in [1, {_lib.POLICY_MAX_DIRECTIONS}], got {N}")
        was_np = theta is not None and not isinstance(theta, torch.Tensor)
        th = torch.zeros(P, dtype=torch.float64, device=self.device) if theta is None else self._to_device(theta, torch.float64)[0]
        th = th.reshape(-1).clone()
        if th.numel() != P:
            raise ValueError(f"theta must have {P} elements, got {th.numel()}")
        q.top, q.step_size, q.noise, q.gamma = N if top is None else int(top), float(step_size), float(noise), float(gamma)
        base = self._next_policy_seed() if seed is None else int(seed) & _M64
        stats = torch.empty((iters, 4), dtype=torch.float64, device=self.device)
        returns = None
        for i in range(iters):
            q.seed = plan_iteration_seed(base, i)
            start, _, _ = eng.plan_start(self._policy_starts(E, policy_starts_seed(q.seed)))
            params = eng.policy_perturb(th, N, q)
            returns, _ = eng.policy_eval(start, params, H, q, False)
            eng.policy_update(returns, th, q, stats[i])
        return PolicySearchResult(self._ret(th, was_np), self._ret(returns, was_np), self._ret(stats, was_np))

    # ------------------------------------------------------------------ fused rollouts
    def rollout(self, horizon: int, actions=None, record: bool = False, auto_reset: bool = True, max_episode_steps=None):
        """``horizon`` steps of every env in ONE kernel launch: the batched counterpart of the reference's
        collection loop (zoo/util.py:33-93) with gym's TimeLimit (``max_episode_steps`` of the registry,
        register_env.py) and the per-episode ``reset()`` done on the device.

        actions: ``[horizon, num_envs]`` tensor / numpy (teacher-forced policy) or None for the uniform
        random policy (``env.action_space.sample()``, zoo/util.py:57).
        record:  also return the transitions in the reference's dataset layout (zoo/util.py:62-67):
        ``observations, next_observations [T,B,4]; actions, rewards [T,B]; dones, timeouts bool[T,B]``.
        Returns a dict with those records (if any) and ``stats``: device double[6] = [sum of rewards,
        #terminated, #truncated, #episodes finished, sum of finished returns, sum of finished lengths];
        ``rollout_info(stats)`` turns it into the reference's avg_reward / avg_length / total_episode_num."""
        eng = self._ensure_engine()
        if eng is None:
            raise NotImplementedError(f"{type(self).__name__} has no fused rollout kernel")
        assert self.state is not None, "Call reset before using rollout."
        if actions is not None and not record:
            piped = self._rollout_host_actions(int(horizon), actions, auto_reset, max_episode_steps)
            if piped is not None:
                return piped
        rp = self._rollout_params()
        rp.horizon = int(horizon)
        mes = getattr(self, "max_episode_steps", 0) if max_episode_steps is None else max_episode_steps
        rp.max_episode_steps = int(mes or 0)
        rp.auto_reset = int(bool(auto_reset))
        rp.random_policy = int(actions is None)
        rp.env_offset = int(getattr(self, "env_offset", 0))
        # reset() zeroes the episode / step counters of the streams, so the streams themselves must change with every
        # un-seeded reset: `env.reset(); env.rollout(T)` in a loop (offline.collect_dataset) would otherwise replay the
        # same random actions and in-kernel reset samples each cycle.  reset(seed=s) restarts at epoch 0 (reproducible).
        epoch = max(self._rollout_epoch, 0)
        rp.seed_reset = (self._seed * 0x9E3779B97F4A7C15 + 0x5851F42D4C957F2D + epoch * 0xA0761D6478BD642F) & 0xFFFFFFFFFFFFFFFF
        rp.seed_action = (self._seed * 0xD1B54A32D192ED03 + 0x14057B7EF767814F + epoch * 0xE7037ED1A0B428DB) & 0xFFFFFFFFFFFFFFFF
        a = None
        if actions is not None:
            a = action_rule(self, self._to_device(actions)[0], len(self.action_space.shape) > 0)
        stats = torch.zeros(6, dtype=torch.float64, device=self.device)
        # obs_noise_params (mujoco_env.py:98-104): the step counter of the noise stream continues through the rollout
        noise = self._next_obs_noise(advance=int(horizon))
        out = eng.rollout(rp, a, bool(record), stats, noise=noise)
        out["stats"] = stats
        return out

    # a teacher-forced rollout whose actions live on the HOST: uploading [horizon, n] first and launching afterwards leaves
    # the GPU idle during the upload and PCIe idle during the kernel (a charged-ball env-step costs 18 ps of upload and
    # 4 ps of kernel).  A rollout of T steps equals consecutive rollouts of its pieces bit for bit (state, counters, the
    # streams' step counter and the noise counter all continue: tested), so the horizon is cut into pieces whose uploads
    # run on a side stream one piece ahead of the kernels.
    _ROLLOUT_PIECE_BYTES = 32 << 20
    _ROLLOUT_PIECE_MIN_STEPS = 8

    @staticmethod
    def plan_rollout_pieces(horizon: int, row_bytes: int, piece_bytes: int, min_steps: int):
        """[(lo, hi), ...] tiling [0, horizon) in pieces of equal length (the last may be shorter), or None when the rollout is
        too small to be worth cutting.  A piece holds >= ``piece_bytes`` of actions and >= ``min_steps`` steps: a launch reads
        and writes every env's state and counters once (74 bytes per charged-ball env), which one-step pieces of a 2^26-env
        batch turn into HBM-bound launches that starve the concurrent upload (measured: 34 G env-steps/s end to end
        against 40 G unpipelined, 47 G with 8-step pieces)."""
        steps = max(int(min_steps), int(piece_bytes) // max(int(row_bytes), 1), 1)
        if horizon < 2 * steps or horizon * row_bytes < 2 * piece_bytes:
            return None
        return [(lo, min(horizon, lo + steps)) for lo in range(0, horizon, steps)]

    def _rollout_host_actions(self, horizon, actions, auto_reset, max_episode_steps):
        a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(actions)
        if a.is_cuda or a.dim() < 2 or a.shape[0] != horizon or a.shape[1] != self.num_envs or not a.is_contiguous():
            return None
        pieces = self.plan_rollout_pieces(horizon, a[0].numel() * a.element_size(), self._ROLLOUT_PIECE_BYTES, self._ROLLOUT_PIECE_MIN_STEPS)
        if pieces is None:
            return None  # small: one upload, one launch
        steps = pieces[0][1]
        cur = torch.cuda.current_stream(self.device)
        side = getattr(self, "_upload_stream", None)
        if side is None:
            side = self._upload_stream = torch.cuda.Stream(self.device)
        bufs = [torch.empty((steps,) + tuple(a.shape[1:]), dtype=a.dtype, device=self.device) for _ in range(2)]
        free = [None, None]  # event: the kernel that read this buffer has finished
        stats = None
        for k, (lo, hi) in enumerate(pieces):
            buf = bufs[k & 1]
            with torch.cuda.stream(side):
                if free[k & 1] is not None:
                    side.wait_event(free[k & 1])
                elif k == 0:
                    side.wait_stream(cur)  # the buffers' allocation and everything queued before this call
                buf[: hi - lo].copy_(a[lo:hi], non_blocking=True)
                up = torch.cuda.Event()
                up.record(side)
            cur.wait_event(up)
            out = self.rollout(hi - lo, actions=buf[: hi - lo], record=False, auto_reset=auto_reset, max_episode_steps=max_episode_steps)
            ev = torch.cuda.Event()
            ev.record(cur)
            free[k & 1] = ev
            stats = out["stats"] if stats is None else stats + out["stats"]
        return {"stats": stats}

    @staticmethod
    def rollout_info(stats) -> dict:
        """zoo/util.py:87-91 (one device->host read)."""
        r_sum, n_term, n_trunc, n_fin, fin_ret, fin_len = [float(v) for v in stats.tolist()]
        n = max(n_fin, 1.0)
        return dict(avg_reward=fin_ret / n, avg_length=fin_len / n, total_episode_num=int(n_fin), reward_sum=r_sum,
                    terminated=int(n_term), truncated=int(n_trunc))

    def _rollout_params(self):
        raise NotImplementedError(f"{type(self).__name__} has no fused rollout kernel")

    # ------------------------------------------------------------------ host-side callers
    def step_host(self, action, outputs=None):
        """``step`` for callers that live on the host (the reference's numpy world): ``action`` is a
        numpy array / CPU tensor; returns numpy ``(obs, reward, terminated, False, {})``.

        Per call: pinned H2D copy of the actions, the step kernel, D2H copies of obs / reward / done
        into pinned staging buffers, one stream synchronise.  The returned arrays are views of those
        staging buffers (valid until the next ``step_host``).  ``outputs``: subset of ("obs", "reward", "done") to
        download (default all, the reference's contract); the rest stays on the device and comes back as None."""
        if getattr(self, "_staging", None) is None:
            self._staging = HostStaging(self)
        return self._staging.step(action, outputs)

    # ------------------------------------------------------------------ seeding (gym.Env.reset(seed=))
    def _reseed(self, seed):
        if seed is not None:
            self._seed = int(seed) & 0xFFFFFFFFFFFFFFFF
            self._reset_count = 0
            self._plan_count = 0
            self._policy_count = 0
            self._rollout_epoch = 0
        else:
            self._rollout_epoch += 1

    def _next_plan_seed(self):
        """A fresh Philox key per unseeded planner call: (seed, planner call counter).  A counter of its own, so planning does
        not shift the initial-state draws of a later unseeded reset() (``_next_sample_seed``)."""
        s = (self._seed * 0xC2B2AE3D27D4EB4F + self._plan_count * 0x165667B19E3779F9 + 0x27D4EB2F165667C5) & 0xFFFFFFFFFFFFFFFF
        self._plan_count += 1
        return s

    def _next_policy_seed(self):
        """A fresh Philox key per unseeded policy-search call: (seed, a counter of its own), so searching does not shift the
        initial-state draws of a later unseeded reset()."""
        s = (self._seed * 0x94D049BB133111EB + self._policy_count * 0xBF58476D1CE4E5B9 + 0x2545F4914F6CDD1D) & _M64
        self._policy_count += 1
        return s

    def _next_sample_seed(self):
        """A fresh Philox key per sampling call: (seed, call counter) so repeated resets differ but a
        given (seed, call index) is reproducible and independent of sharding.  While ``_sample_key`` is set, that key, with
        the counter left alone (the policy search's start states)."""
        if self._sample_key is not None:
            return self._sample_key
        s = (self._seed * 0x9E3779B97F4A7C15 + self._reset_count * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF
        self._reset_count += 1
        return s
