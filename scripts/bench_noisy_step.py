"""Time of the noisy float32 inverted-pendulum step (emei_ip_step_noisy_f32: the step of every float32 inverted pendulum
built with obs_noise_params) at one size, with CUDA events around back-to-back launches on one stream.  The state ping-pongs
between two buffers of 2^20 x 16 B, so the working set (~45 MB with the observations, rewards and flags) stays in the 126 MB
L2 after the first launch: this is the step's compute time, not its HBM time.

usage: python scripts/bench_noisy_step.py [--n 1048576] [--fr 4] [--iters 200]  -> one JSON line"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--fr", type=int, default=4)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    n = a.n
    env = E.make("BoundaryInvertedPendulumSwingUp-v0", num_envs=1, freq_rate=a.fr, dtype=torch.float32)
    src = env._ensure_engine().params
    p = _lib.CartPoleParams()
    ctypes.memmove(ctypes.byref(p), ctypes.byref(src), ctypes.sizeof(p))
    p.action_kind = _lib.ACTION_CONTINUOUS_F32
    z = _lib.NoiseParams()
    for j, s in enumerate((0.01, 0.01, 0.03, 0.03)):
        z.sigma[j] = s
    z.seed = 12345
    rng = np.random.default_rng(0)
    st = torch.as_tensor((rng.uniform(-1, 1, size=(n, 4)) * np.array([1.9, np.pi, 5.0, 8.0])).astype(np.float32)).cuda()
    bufs = [st, torch.empty_like(st)]
    obs = torch.empty_like(st)
    act = torch.as_tensor(rng.uniform(-3, 3, size=n).astype(np.float32)).cuda()
    rew = torch.empty(n, dtype=torch.float32, device="cuda")
    done = torch.empty(n, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    f = _lib.lib.emei_ip_step_noisy_f32

    def step(k):
        z.step = k
        rc = f(bufs[k & 1].data_ptr(), bufs[1 - (k & 1)].data_ptr(), obs.data_ptr(), act.data_ptr(), rew.data_ptr(), done.data_ptr(),
               None, n, ctypes.byref(p), ctypes.byref(z), stream)
        assert rc == 0

    for k in range(a.warmup):
        step(k)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for k in range(a.iters):
        step(a.warmup + k)
    t1.record()
    torch.cuda.synchronize()
    us = t0.elapsed_time(t1) * 1e3 / a.iters
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"entry": "emei_ip_step_noisy_f32", "n": n, "freq_rate": a.fr, "iters": a.iters, "us_per_step": round(us, 2),
                      "gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}))


if __name__ == "__main__":
    main()
