"""Policy-search iteration timings: the fused kernels (emei_*_policy_eval_* + emei_policy_perturb + emei_policy_update)
against the same ARS iteration written in torch on the existing API, and the eval beside the random-policy rollout kernel at the
same C E H.

    python scripts/bench_policy_search.py --out profiles/r07_bench_policy_search.jsonl

Every number is CUDA-event time over warmed shapes (each shape runs once before its timed window); one JSON line per
(task, precision, 2N, E).  The card's name and power limit are read in the same run.  H = 200 throughout; the policies are
theta = 0 perturbed with noise 0.5, so balancing episodes end at different steps (the mean episode length is reported: the
eval stops a pair at its terminating step, the torch loop and the rollout run all H steps).
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

H = 200
SHAPES = [(16, 16), (64, 64), (256, 256), (512, 512)]  # (2N, E): one CTA of pairs up to 2^18 pairs
TASKS = [("CartPoleBalancing-v0", torch.float32), ("BoundaryInvertedPendulumBalancing-v0", torch.float32),
         ("BoundaryInvertedPendulumBalancing-v0", torch.float64), ("ReboundInvertedDoublePendulumBalancing-v0", torch.float32),
         ("ChargedBallCentering-v0", torch.float32)]


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


def torch_ars(env, twin, start_rep, params, theta, N, En, top, alpha, directions):
    """One ARS iteration as a user writes it today over a C E batch: H x (torch linear policy, one stateless step, mask), then
    the mean over episodes, top-k and the weighted sum of the directions.  The analytic families step with
    get_batch_transition; the charged ball, which has none, with step() on a C E env."""
    discrete = len(env.action_space.shape) == 0
    D = params.shape[1] - 1
    w = params.repeat_interleave(En, 0)  # [C E, P], candidate-major
    lo, hi = (0.0, 1.0) if discrete else (float(env.action_space.low[0]), float(env.action_space.high[0]))
    ret = torch.zeros(w.shape[0], dtype=torch.float64, device=w.device)
    alive = torch.ones(w.shape[0], dtype=torch.bool, device=w.device)
    if twin is None:
        state = obs = start_rep
    else:
        twin.state = start_rep
        state, obs = None, twin.state["free_state"]
    for _ in range(H):
        u = w[:, D] + (w[:, :D] * obs.double()).sum(1)
        a = (u > 0).to(torch.uint8) if discrete else u.to(env.dtype).clamp(lo, hi)
        if twin is None:
            state, obs, r, d = env.get_batch_transition(state, a)
        else:
            obs, r, d, _, _ = twin.step(a)
        ret += torch.where(alive, r.reshape(-1).double(), torch.zeros_like(ret))
        alive &= ~d.reshape(-1).bool()
    m = ret.view(2 * N, En).mean(1)
    rp, rm = m[0::2], m[1::2]
    idx = torch.maximum(rp, rm).topk(top).indices
    both = torch.cat([rp[idx], rm[idx]])
    step = ((rp[idx] - rm[idx])[:, None] * directions[idx]).sum(0)
    return theta + alpha / (top * both.std(unbiased=False)) * step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_policy_search needs a CUDA device"
    torch.cuda.set_device(0)
    gpu, power = card()
    lines = []
    for eid, dtype in TASKS:
        for N2, En in SHAPES:
            N, top = N2 // 2, max(1, N2 // 4)
            env = E.make(eid, num_envs=En, dtype=dtype, device="cuda:0")
            env.reset(seed=0)
            eng, P, q = env._policy_setup()
            q.seed, q.noise, q.top, q.step_size, q.gamma = 1, 0.5, top, 0.02, 1.0
            theta = torch.zeros(P, dtype=torch.float64, device="cuda:0")
            start, _, _ = eng.plan_start(env._policy_starts(En, 7))
            params = eng.policy_perturb(theta, N, q)
            returns, _ = eng.policy_eval(start, params, H, q, False)
            t_eval = timed(lambda: eng.policy_eval(start, params, H, q, False), args.reps)
            th = theta.clone()
            t_pu = timed(lambda: (eng.policy_perturb(th, N, q), eng.policy_update(returns, th, q)), args.reps)
            iters = 5
            t_iter = timed(lambda: env.policy_search(H, iterations=iters, directions=N, top=top, noise=0.5, episodes=En, seed=3),
                           max(1, args.reps // 5)) / iters
            # episode length under these policies (the eval's reward is 1 per step on the balancing tasks)
            ret_len = float(returns.mean()) if "Balancing" in eid else None
            # the same iteration in torch on the existing API
            cb = "ChargedBall" in eid
            C = 2 * N
            twin = E.make(eid, num_envs=C * En, dtype=dtype, device="cuda:0") if cb else None
            if cb:
                twin.reset(seed=0)
                start_rep = {k: v.repeat((C,) + (1,) * (v.dim() - 1)) for k, v in zip(("on_circle", "circle_state", "free_state"), start)}
            else:
                start_rep = start.repeat(C, 1)
            dirs = (params[0::2] - theta) / 0.5
            with torch.no_grad():
                t_torch = timed(lambda: torch_ars(env, twin, start_rep, params, theta, N, En, top, 0.02, dirs), max(1, args.reps // 5))
            # the eval's ceiling: the random-policy rollout over C E envs for H steps (its own env, no records)
            roll = E.make(eid, num_envs=C * En, dtype=dtype, device="cuda:0")
            roll.reset(seed=0)
            t_roll = timed(lambda: roll.rollout(H), args.reps)
            n = C * En
            rec = dict(task=eid, dtype=str(dtype).replace("torch.", ""), two_N=C, E=En, top=top, H=H, mean_return=ret_len,
                       eval_ms=t_eval, perturb_update_ms=t_pu, search_iter_ms=t_iter, torch_iter_ms=t_torch, rollout_random_ms=t_roll,
                       eval_pair_steps_per_s=n * H / (t_eval * 1e-3), torch_pair_steps_per_s=n * H / (t_torch * 1e-3),
                       rollout_env_steps_per_s=n * H / (t_roll * 1e-3), speedup_vs_torch=t_torch / t_iter, gpu=gpu,
                       power_limit=power)
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
