"""Offline datasets in the reference's on-disk format, produced from and loaded onto the device layout.

Reference anchors: the collection loop and its record keys ``zoo/util.py:33-93`` (``observations,
next_observations, actions, rewards, dones, timeouts``; ``dones = float(terminated or truncated)``,
``timeouts = float(truncated)``), the flat h5 writer ``zoo/util.py:108-111``, the loader and its sanity checks
``emei/core.py:61-81,109-128``, the local cache path ``emei/core.py:15,83-92``
(``~/.emei/offline_data/<env_name>/<env_params_name>/<file>``; ``$EMEI_DATASET_PATH`` overrides the root, additive).

The fused rollout kernels record time-major ``[T, num_envs, ...]`` arrays; the reference's files are written
episode after episode.  ``records_to_dataset`` transposes each record to env-major on the device
(``emei_records_transpose``: every env's trajectory, hence each of its episodes, becomes contiguous) and
flattens it to the reference's ``[N, ...]`` shape.  h5 needs ``h5py`` (not a dependency of this package):
``.npz`` is always available and holds the same keys.
"""
import os
import pathlib
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib

KEYS = ("observations", "next_observations", "actions", "rewards", "dones", "timeouts")
# emei/core.py:15
DATASET_PATH = pathlib.Path(os.environ.get("EMEI_DATASET_PATH", "~/.emei/offline_data")).expanduser()


def _transpose(t: torch.Tensor, stream) -> torch.Tensor:
    """[T, n, ...] -> [n, T, ...] through the C ABI (element = everything after the first two dims)."""
    T, n = int(t.shape[0]), int(t.shape[1])
    src = t.view(torch.uint8) if t.dtype == torch.bool else t
    src = src.contiguous()
    elem = src.element_size()
    for d in src.shape[2:]:
        elem *= int(d)
    if elem not in (1, 4, 8, 16, 24, 32, 48):
        raise ValueError(f"record element of {elem} bytes is not a dataset record (1, 4, 8, 16, 24, 32 or 48 bytes)")
    out = torch.empty((n, T) + tuple(src.shape[2:]), dtype=src.dtype, device=src.device)
    with torch.cuda.device(src.device):
        _lib.call("emei_records_transpose", src.data_ptr(), out.data_ptr(), T, n, elem, stream)
    return out.view(torch.bool) if t.dtype == torch.bool else out


def records_to_dataset(records: Dict[str, torch.Tensor], order: str = "env") -> Dict[str, torch.Tensor]:
    """``env.rollout(..., record=True)`` output -> flat device tensors with the reference's keys and shapes:
    observations / next_observations ``[N, obs_dim]``, actions ``[N]`` (Discrete) or ``[N, 1]`` (Box),
    rewards ``[N]``, dones / timeouts ``[N]`` float32 (zoo/util.py:62-67 stores ``float(done)``).
    order="env": env-major (each env's trajectory contiguous, the reference's episode-after-episode order);
    order="time": time-major, no transposition."""
    if order not in ("env", "time"):
        raise ValueError("order must be 'env' or 'time'")
    out = {}
    for k in KEYS:
        t = records[k]
        if order == "env":
            t = _transpose(t, torch.cuda.current_stream(t.device).cuda_stream)
        t = t.reshape((t.shape[0] * t.shape[1],) + tuple(t.shape[2:]))
        if k in ("dones", "timeouts"):
            t = t.to(torch.float32)
        if k == "actions" and t.dtype.is_floating_point:
            t = t.reshape(-1, 1)  # Box(-1, 1, (1,)) actions are 1-vectors in the reference's files
        out[k] = t
    return out


def collect_dataset(env, total_sample_num: int, actions=None, order: str = "env") -> Tuple[Dict[str, np.ndarray], dict]:
    """Batched counterpart of ``zoo/util.py:33-93`` ``rollout(env, total_sample_num, agent)``: resets, then advances
    every env ``ceil(total_sample_num / num_envs)`` steps in ONE fused launch (TimeLimit and per-episode resets
    in-kernel), with the uniform random policy (``agent is None``, zoo/util.py:57) or teacher-forced
    ``actions [T, num_envs]``.  Returns ``(samples, rollout_info)`` like the reference: numpy arrays under the
    six dataset keys and ``avg_reward / avg_length / total_episode_num`` over the episodes that finished.
    The reference stops at the end of the episode that crosses ``total_sample_num``; here every env stops after the
    same number of steps, so the last episode of each env may be cut short (its final ``dones`` is then 0)."""
    n = env.num_envs
    T = (int(total_sample_num) + n - 1) // n
    env.reset()
    rec = env.rollout(T, actions=actions, record=True)
    ds = records_to_dataset(rec, order)
    info = env.rollout_info(rec["stats"])
    samples = {k: v.cpu().numpy() for k, v in ds.items()}
    return samples, dict(avg_reward=info["avg_reward"], avg_length=info["avg_length"], total_episode_num=info["total_episode_num"])


def save_dataset(dataset: Dict, path) -> pathlib.Path:
    """zoo/util.py:108-111 ``save_as_h5`` (flat, one array per key) for ``.h5`` / ``.hdf5`` paths when ``h5py`` is
    importable; ``.npz`` otherwise / for ``.npz`` paths."""
    path = pathlib.Path(path)
    arrays = {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in dataset.items()}
    path.parent.mkdir(parents=True, exist_ok=True)
    if path.suffix in (".h5", ".hdf5"):
        try:
            import h5py
        except ImportError as e:
            raise ImportError("writing .h5 needs h5py; use a .npz path (same keys) instead") from e
        with h5py.File(path, "w") as f:
            for k, v in arrays.items():
                f[k] = v
    else:
        if path.suffix != ".npz":
            path = path.with_suffix(path.suffix + ".npz")
        np.savez(path, **arrays)
    return path


def check_dataset(data: Dict[str, np.ndarray]) -> None:
    """the sanity checks of ``OfflineEnv.get_dataset`` (core.py:117-126), plus consistent lengths."""
    for key in ("observations", "actions", "rewards", "dones", "timeouts"):
        assert key in data, "Dataset is missing key %s" % key
    n = data["observations"].shape[0]
    for key in KEYS:
        if key in data:
            assert data[key].shape[0] == n, f"Dataset key {key} has {data[key].shape[0]} rows, observations has {n}"


def load_dataset(path, device: Optional[torch.device] = None) -> Dict:
    """core.py:61-81 ``load_h5_data`` for ``.h5`` / ``.hdf5`` (needs h5py) and the same for ``.npz``; runs
    ``check_dataset``.  With ``device`` the arrays are returned as tensors on that device."""
    path = pathlib.Path(path)
    if path.suffix in (".h5", ".hdf5"):
        try:
            import h5py
        except ImportError as e:
            raise ImportError("reading .h5 needs h5py") from e
        data = {}
        with h5py.File(path, "r") as f:
            def visitor(name, item):
                if isinstance(item, h5py.Dataset):
                    data[name] = item[()]
            f.visititems(visitor)
    else:
        with np.load(path) as z:
            data = {k: z[k] for k in z.files}
    check_dataset(data)
    if device is not None:
        return {k: torch.as_tensor(v).to(device) for k, v in data.items()}
    return data


def dataset_path(env, dataset_name: str) -> pathlib.Path:
    """core.py:83-92 ``get_path_from_url`` without the url: ``DATASET_PATH/<env_name>/<env_params_name>/<file>``."""
    return DATASET_PATH / env.env_name / env.env_params_name / dataset_name
