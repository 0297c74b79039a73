"""Batched, device-resident counterpart of the reference's API contract ``emei/core.py``.

Mirrors ``Freezable`` (core.py:18-37) and ``EmeiEnv`` (core.py:131-193): same method names,
argument meaning and error behaviour, with arrays generalised to ``[num_envs, dim]`` CUDA tensors.
numpy inputs are accepted everywhere (copied to the device; results come back as numpy), so code
written against the reference's ``get_batch_*`` keeps working unchanged.

``OfflineEnv`` (core.py:40-128): datasets are read from the reference's local cache layout
(``emei_b200.offline``); the download step (``urllib``, core.py:94-107) is out of scope -- there is no network --
so ``dataset_names`` lists what is on disk and ``get_dataset`` raises for anything that is not.
"""
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
            self._rollout_epoch = 0
        else:
            self._rollout_epoch += 1

    def _next_sample_seed(self):
        """A fresh Philox key per sampling call: (seed, call counter) so repeated resets differ but a
        given (seed, call index) is reproducible and independent of sharding."""
        s = (self._seed * 0x9E3779B97F4A7C15 + self._reset_count * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF
        self._reset_count += 1
        return s
