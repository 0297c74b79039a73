"""Times differentiable scoring: get_batch_reward / get_batch_reward_terminal_seq forward, their backward(), and a plain-torch
restatement of the same reward under torch.autograd.

Workloads, float32 and float64, 2^24 transitions each:
  hopper / halfcheetah  one-shot (obs, pre_obs [2^24, D] separate allocations, action [2^24, A]) and trajectory layout
                        (obs_seq [T+1, n, D], action [T, n, A], T = 64, n = 2^18)
  ip_swingup / i2p_swingup  one-shot obs [2^24, D] (BoundaryInvertedPendulumSwingUp, BoundaryInvertedDoublePendulumSwingUp)
Records per workload:
  fwd         the scoring call alone (grad-requiring inputs: the kernels of the differentiable path's forward)
  bwd         r.backward(w) alone on a retained graph (the leaves' .grad reset to None, so nothing is accumulated)
  fwd_bwd     fwd + bwd
  bwd_kernels the backward's launches through the C ABI into preallocated buffers (emei_sum_* when the action gradient is
              wanted, then emei_reward_vjp_* / emei_reward_seq_vjp_*): no autograd
  split_*     each of those launches alone (rows: the row / trajectory VJP kernel; sum: emei_sum_*; action: the flat
              action-gradient kernel), with its own bytes over its own time
  torch_fwd_bwd  the plain-torch restatement, forward + backward under torch.autograd
The backward's algorithmic bytes per transition (es = element size, D / A = obs / action width; every array read or written
once, except g_reward, which the sum and the VJP both read):
  mujoco one-shot : g_reward 2 es + g_obs D es + g_pre_obs D es + action A es + g_action A es
  mujoco seq      : g_reward 2 es + g_obs_seq D es (T+1 rows per T transitions) + action A es + g_action A es
                    (e.g. Hopper float32: 8 + 48 + 12 + 12 = 80 B)
  pendulum        : obs D es + g_reward es + g_obs D es (no action gradient, no sum)
Share of the copy peak = bytes / time / 6549.1 GB/s (the measured copy peak bench.py uses).  Card name and power limit are
read in the same run.  Output lines are appended to --out.

    python scripts/bench_scoring_grad.py [--out profiles/r05_bench_scoring_grad.jsonl]
"""
import argparse
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib  # noqa: E402
from bench_autodiff import card, time_ms  # noqa: E402

COPY_PEAK_BPS = 6549.1e9
N = 1 << 24
T_SEQ = 64
ENV = {"hopper": ("HopperRunning-v0", 12, 3, 1e-3), "halfcheetah": ("HalfCheetahRunning-v0", 18, 6, 0.1),
       "ip_swingup": ("BoundaryInvertedPendulumSwingUp-v0", 4, 0, 0.0),
       "i2p_swingup": ("BoundaryInvertedDoublePendulumSwingUp-v0", 6, 0, 0.0)}


def torch_reward(kind, o, p, a, dt):
    """the plain-torch restatement of the reward (Hopper with terminate_when_unhealthy=True: healthy term 1)"""
    if kind == "hopper":
        return (1.0 + (o[:, 0] - p[:, 0]) / dt - 1e-3 * (a * a).sum()).reshape(-1, 1)
    if kind == "halfcheetah":
        return ((o[:, 0] - p[:, 0]) / dt - 0.1 * (a * a).sum()).reshape(-1, 1)
    if kind == "ip_swingup":
        return ((1 - torch.cos(o[:, 1])) / 2).reshape(-1, 1)
    y = torch.cos(o[:, 1]) + torch.cos(o[:, 1] + o[:, 2])
    return ((2 - y) / 4 - (5e-3 * o[:, 4] ** 2 + 1e-4 * o[:, 5] ** 2)).reshape(-1, 1)


def bwd_bytes(kind, layout, es, D, A, T):
    if A == 0:
        return (2 * D + 1) * es
    if layout == "seq":
        return (2 + D * (T + 1) / T + 2 * A) * es
    return (2 + 2 * D + 2 * A) * es


def run(kind, layout, dtype, iters):
    env_id, D, A, _ = ENV[kind]
    dev = "cuda:0"
    env = E.make(env_id, dtype=dtype, device=dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    mj = A > 0
    es = torch.empty(0, dtype=dtype).element_size()
    T, n = (T_SEQ, N // T_SEQ) if layout == "seq" else (1, N)
    if layout == "seq":
        x = torch.randn(T + 1, n, D, device=dev, dtype=dtype, generator=gen)
        act = torch.rand(T, n, A, device=dev, dtype=dtype, generator=gen) * 2 - 1
        w = torch.randn(T, n, 1, device=dev, dtype=dtype, generator=gen)
    else:
        x = torch.randn(N, D, device=dev, dtype=dtype, generator=gen)
        pre = torch.randn(N, D, device=dev, dtype=dtype, generator=gen) if mj else None
        act = (torch.rand(N, A, device=dev, dtype=dtype, generator=gen) * 2 - 1) if mj else None
        w = torch.randn(N, 1, device=dev, dtype=dtype, generator=gen)
    leaves = [t.requires_grad_(True) for t in ((x, act) if layout == "seq" else (x, pre, act)) if t is not None]

    def fwd():
        if layout == "seq":
            return env.get_batch_reward_terminal_seq(x, act)[0]
        return env.get_batch_reward(x, pre, act) if mj else env.get_batch_reward(x)

    r = fwd()

    def bwd():
        for t in leaves:
            t.grad = None
        r.backward(w, retain_graph=True)

    def fwd_bwd():
        for t in leaves:
            t.grad = None
        fwd().backward(w)

    rec = dict(kind=kind, layout=layout, dtype=str(dtype).replace("torch.", ""), transitions=N, T=T if layout == "seq" else None,
               n=n)
    rec["fwd_ms"] = time_ms(lambda: fwd(), iters)
    rec["bwd_ms"] = time_ms(bwd, iters)
    rec["fwd_bwd_ms"] = time_ms(fwd_bwd, iters)

    # the backward's launches alone, preallocated buffers
    prm, stream = ctypes.byref(env._scoring_params()), torch.cuda.current_stream().cuda_stream
    sfx = env._suffix
    g_sum = torch.empty(1, dtype=torch.float64, device=dev)
    ws = torch.zeros(_lib.SUMSQ_WORKSPACE_BYTES // 8, dtype=torch.float64, device=dev)
    gx = torch.empty_like(x)
    gp = torch.empty_like(x) if (mj and layout != "seq") else None
    ga = torch.empty_like(act) if mj else None
    wv = w.reshape(-1)
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    lib = _lib.lib

    def kernels():
        if mj:
            getattr(lib, "emei_sum" + sfx)(wv.data_ptr(), wv.numel(), g_sum.data_ptr(), ws.data_ptr(), stream)
        if layout == "seq":
            getattr(lib, "emei_reward_seq_vjp" + sfx)(None, ptr(act), wv.data_ptr(), g_sum.data_ptr(), gx.data_ptr(), ptr(ga), n, T, prm, stream)
        else:
            getattr(lib, "emei_reward_vjp" + sfx)(None if mj else x.data_ptr(), ptr(act), wv.data_ptr(), ptr(g_sum) if mj else None,
                                         gx.data_ptr(), ptr(gp), ptr(ga), N, prm, stream)

    rec["bwd_kernels_ms"] = time_ms(kernels, iters)
    # where the backward's kernel time goes: each launch alone, with its own bytes and share of the copy peak
    split = {}
    if layout == "seq":
        split["rows"] = (lambda: getattr(lib, "emei_reward_seq_vjp" + sfx)(None, None, wv.data_ptr(), None, gx.data_ptr(), None, n, T,
                                                                           prm, stream), (1 + D * (T + 1) / T) * es)
    else:
        split["rows"] = (lambda: getattr(lib, "emei_reward_vjp" + sfx)(None if mj else x.data_ptr(), None, wv.data_ptr(), None,
                                                                       gx.data_ptr(), ptr(gp), None, N, prm, stream),
                         (1 + 2 * D) * es)  # g_reward + g_obs + g_pre_obs (mujoco) / obs + g_reward + g_obs (pendulums)
    if mj:
        split["sum"] = (lambda: getattr(lib, "emei_sum" + sfx)(wv.data_ptr(), wv.numel(), g_sum.data_ptr(), ws.data_ptr(), stream), es)
        split["action"] = (lambda: getattr(lib, "emei_reward_vjp" + sfx)(None, ptr(act), wv.data_ptr(), g_sum.data_ptr(), None, None,
                                                                         ptr(ga), N, prm, stream), 2 * A * es)
    for part, (fn, part_bytes) in split.items():
        ms = time_ms(fn, iters)
        rec[f"split_{part}_ms"] = ms
        rec[f"split_{part}_share_of_copy_peak"] = round(part_bytes * N / (ms * 1e-3) / COPY_PEAK_BPS, 3)
    b = bwd_bytes(kind, layout, es, D, A, T)
    rec["bwd_bytes_per_transition"] = b
    for key in ("bwd_ms", "bwd_kernels_ms"):
        rec[key.replace("_ms", "") + "_share_of_copy_peak"] = round(b * N / (rec[key] * 1e-3) / COPY_PEAK_BPS, 3)

    # plain torch under autograd (the same shapes; the seq layout through its two shifted views)
    dt = env.dt if mj else 0.0

    def torch_fwd_bwd():
        for t in leaves:
            t.grad = None
        if layout == "seq":
            rt = torch_reward(kind, x[1:].reshape(N, D), x[:-1].reshape(N, D), act.reshape(N, A), dt)
        else:
            rt = torch_reward(kind, x, pre, act, dt)
        rt.backward(w.reshape(-1, 1))

    rec["torch_fwd_bwd_ms"] = time_ms(torch_fwd_bwd, iters)
    del r, gx, gp, ga
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_scoring_grad.jsonl"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scoring_grad.py measures on a CUDA device; there is none")
    name, power = card()
    lines = [json.dumps(dict(card=name, power_limit_and_max_sm_clock=power, copy_peak_Bps=COPY_PEAK_BPS, transitions=N))]
    print(lines[0], flush=True)
    for kind, layouts in (("hopper", ("one_shot", "seq")), ("halfcheetah", ("one_shot", "seq")), ("ip_swingup", ("one_shot",)),
                          ("i2p_swingup", ("one_shot",))):
        for layout in layouts:
            for dtype in (torch.float32, torch.float64):
                lines.append(json.dumps(run(kind, layout, dtype, args.iters)))
                print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
