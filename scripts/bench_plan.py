"""Planner iteration timings: the fused CEM / MPPI kernels (emei_*_plan_eval_* + emei_plan_update_*) against the same CEM
written in torch on the existing API, and the eval kernel beside the random-policy rollout kernel at the same n H.

    python scripts/bench_plan.py --out profiles/r06_bench_plan.jsonl

Every number is CUDA-event time over warmed shapes (each shape runs once before its timed window); one JSON line per
(task, precision, B, K).  The card's name and power limit are read in the same run.  H = 50 throughout.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib  # noqa: E402

H = 50
SHAPES = [(1, 1024), (64, 512), (1024, 256)]
TASKS = [("ContinuousCartPoleSwingUp-v0", torch.float32), ("BoundaryInvertedDoublePendulumSwingUp-v0", torch.float32),
         ("BoundaryInvertedDoublePendulumSwingUp-v0", torch.float64), ("ContinuousChargedBallCentering-v0", torch.float32)]


def timed(fn, reps):
    fn()  # warm the shape
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps  # ms


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def torch_cem(env, twin, start, mean, std, K, elites):
    """One CEM iteration as a user writes it today: torch.randn candidates, the trajectory kernel (or a recorded rollout for the
    charged ball), the masked return, topk, gather, mean and std."""
    B = mean.shape[1]
    lo, hi = float(env.action_space.low[0]), float(env.action_space.high[0])
    a = (mean[:, :, None] + std[:, :, None] * torch.randn((H, B, K), device=mean.device, dtype=mean.dtype)).clamp(lo, hi)
    flat = a.reshape(H, B * K)
    if twin is None:
        rows = start.repeat_interleave(K, 0)
        _, _, rew, done = env.get_batch_trajectory(rows, flat)
    else:
        twin.state = start
        rec = twin.rollout(H, actions=flat, record=True, auto_reset=False, max_episode_steps=0)
        rew, done = rec["rewards"], rec["dones"]
    alive = torch.cat([torch.ones_like(done[:1]), ~done[:-1]]).cumprod(0)
    ret = (rew.double() * alive).sum(0).view(B, K)
    idx = ret.topk(elites, dim=1).indices
    el = torch.gather(a, 2, idx[None].expand(H, B, elites))
    return el.mean(-1), el.std(-1, unbiased=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_plan needs a CUDA device"
    torch.cuda.set_device(0)
    gpu, power = card()
    lines = []
    for eid, dtype in TASKS:
        for B, K in SHAPES:
            env = E.make(eid, num_envs=B, dtype=dtype, device="cuda:0")
            env.reset(seed=0)
            eng, start, _, _, q = env._plan_setup(None)
            q.method, q.elites, q.seed = _lib.PLAN_CEM, min(64, K), 1
            mean = torch.zeros((H, B), dtype=dtype, device="cuda:0")
            std = torch.full((H, B), 0.5, dtype=dtype, device="cuda:0")
            returns, _ = eng.plan_eval(start, mean, std, K, q, False)
            t_eval = timed(lambda: eng.plan_eval(start, mean, std, K, q, False), args.reps)
            m2, s2 = mean.clone(), std.clone()
            t_update = timed(lambda: eng.plan_update(returns, m2, s2, q, False), args.reps)
            t_plan = timed(lambda: env.plan(H, candidates=K, iterations=5, elites=min(64, K), seed=3), max(1, args.reps // 5)) / 5
            # the same CEM in torch on the existing API
            cb = "ChargedBall" in eid
            twin = E.make(eid, num_envs=B * K, dtype=dtype, device="cuda:0") if cb else None
            if cb:
                twin.reset(seed=0)
                start_rep = {k: v.repeat_interleave(K, 0) for k, v in env.state.items()}
            else:
                start_rep = env.state.clone()
            t_torch = timed(lambda: torch_cem(env, twin, start_rep, mean, std, K, min(64, K)), max(1, args.reps // 5))
            # the closest existing kernel: the random-policy rollout at the same n H (its own env, no records)
            roll = E.make(eid, num_envs=B * K, dtype=dtype, device="cuda:0")
            roll.reset(seed=0)
            t_roll = timed(lambda: roll.rollout(H), args.reps)
            n = B * K
            rec = dict(task=eid, dtype=str(dtype).replace("torch.", ""), B=B, K=K, H=H, eval_ms=t_eval, update_ms=t_update,
                       plan_iter_ms=t_plan, torch_cem_iter_ms=t_torch, rollout_random_ms=t_roll,
                       eval_cand_steps_per_s=n * H / (t_eval * 1e-3), plan_cand_steps_per_s=n * H / (t_plan * 1e-3),
                       torch_cand_steps_per_s=n * H / (t_torch * 1e-3), rollout_env_steps_per_s=n * H / (t_roll * 1e-3),
                       speedup_vs_torch=t_torch / t_plan, gpu=gpu, power_limit=power)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            del env, twin, roll
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
