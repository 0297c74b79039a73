"""Times the fused open-loop trajectory (emei_*_trajectory_* + emei_*_trajectory_vjp_*) against the chained path it replaces.

For ContinuousCartPoleSwingUp (cart-pole kernels) and BoundaryInvertedDoublePendulumSwingUp (I2P kernels), freq_rate 4,
float32 and float64, at (B, T) in {(1024, 50), (4096, 50), (2^20, 50)}:
  fwd            emei_*_trajectory_*: one launch, T steps, into preallocated buffers
  bwd_all        emei_*_trajectory_vjp_* with every cotangent (g_states, g_obs for I2P, g_rewards) and g_actions
  bwd_rewards    the same with g_rewards only
  floor_fwd      T step launches through the C ABI into the same buffers: the forward half of the floor below
  floor_kernels  T step launches + T VJP launches through the C ABI, no autograd, preallocated buffers: the kernel-only floor
                 of the chained path (its VJPs read the carried cotangent as g_state_out; the g_states term is left out)
  fused_api      env.get_batch_trajectory + backward() of loss = <w_s, states> + <w_o, obs> + <w_r, rewards>
  chained_api    T x env.get_batch_transition + backward() of the same loss (DESIGN.md 4.7's BPTT path)
Kernel lines carry their algorithmic bytes (every array read or written once), an ESTIMATED operation count (OPS_TALLY of
bench_autodiff.py, per env-step) and the roofline bound of the two: max(bytes / HBM peak, ops / math peak) over the measured
time.  A batch smaller than one resident grid (148 SMs x 2048 threads) is latency-bound instead: one env per thread walks a
T-long dependent chain, so neither roofline bound applies there.  Speed-ups are measured ratios.  Card name and power
limit are read in the same run.  Output lines are appended to --out.

    python scripts/bench_trajectory.py [--out profiles/r04_bench_trajectory.jsonl]
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
from emei_b200 import autodiff  # noqa: E402
from bench_autodiff import HBM_BPS, OPS_TALLY, PEAK, card, time_ms  # noqa: E402

FR = 4
FAMILY = {"cp": ("ContinuousCartPoleSwingUp-v0", 4), "i2p": ("BoundaryInvertedDoublePendulumSwingUp-v0", 6)}
SIZES = [(1024, 50), (4096, 50), (1 << 20, 50)]
RESIDENT = 148 * 2048


def run(fam, dtype, n, T):
    env_id, D = FAMILY[fam]
    dev = "cuda:0"
    env = E.make(env_id, freq_rate=FR, dtype=dtype, device=dev)
    gen = torch.Generator(device=dev).manual_seed(n + T)
    y = (torch.rand(n, D, device=dev, dtype=dtype, generator=gen) * 2 - 1) * 0.5
    acts = torch.rand(T, n, device=dev, dtype=dtype, generator=gen) * 2 - 1
    eng, s, a, _ = autodiff._inputs(env, y, acts, steps=T)
    a = a.reshape(T, n)
    ws = torch.randn(T + 1, n, D, device=dev, dtype=dtype, generator=gen)
    wo = torch.randn(T, n, D, device=dev, dtype=dtype, generator=gen)
    wr = torch.randn(T, n, device=dev, dtype=dtype, generator=gen)
    esz, row, sep = s.element_size(), D * s.element_size(), fam == "i2p"
    prm, stream, sfx = ctypes.byref(eng.params), torch.cuda.current_stream().cuda_stream, env._suffix
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    # preallocated buffers: every timed kernel call is exactly one launch
    states = torch.empty(T + 1, n, D, device=dev, dtype=dtype)
    obs = torch.empty(T, n, D, device=dev, dtype=dtype) if sep else None
    rew, done = torch.empty(T, n, device=dev, dtype=dtype), torch.empty(T, n, device=dev, dtype=torch.uint8)
    g0, g_act = torch.empty(n, D, device=dev, dtype=dtype), torch.empty(T, n, device=dev, dtype=dtype)
    wo_k = wo if sep else None  # the cart-pole envs' observation is states[1:]: its cotangent arrives in g_states
    carry = torch.empty(T + 1, n, D, device=dev, dtype=dtype)
    eng.params.action_kind = E._lib.ACTION_CONTINUOUS_F32 if dtype == torch.float32 else E._lib.ACTION_CONTINUOUS_F64
    traj, traj_vjp, step, vjp = eng._trajectory_entry + sfx, eng._trajectory_vjp_entry + sfx, eng._step_entry + sfx, eng._vjp_entry + sfx
    call = E._lib.call

    def fwd():
        call(traj, s.data_ptr(), a.data_ptr(), states.data_ptr(), ptr(obs), rew.data_ptr(), done.data_ptr(), n, T, prm, stream)

    def bwd_all():
        call(traj_vjp, states.data_ptr(), a.data_ptr(), ws.data_ptr(), ptr(wo_k), wr.data_ptr(), g0.data_ptr(), g_act.data_ptr(), n, T,
             prm, stream)

    def bwd_rewards():
        call(traj_vjp, states.data_ptr(), a.data_ptr(), None, None, wr.data_ptr(), g0.data_ptr(), g_act.data_ptr(), n, T, prm, stream)

    def floor_fwd():
        for t in range(T):
            call(step, states[t].data_ptr(), states[t + 1].data_ptr(), ptr(obs[t] if sep else None), a[t].data_ptr(), rew[t].data_ptr(),
                 done[t].data_ptr(), None, n, prm, stream)

    def floor_kernels():
        for t in range(T):
            call(step, states[t].data_ptr(), states[t + 1].data_ptr(), ptr(obs[t] if sep else None), a[t].data_ptr(), rew[t].data_ptr(),
                 done[t].data_ptr(), None, n, prm, stream)
        carry[T].zero_()
        for t in range(T - 1, -1, -1):
            call(vjp, states[t].data_ptr(), a[t].data_ptr(), carry[t + 1].data_ptr(), ptr(wo_k[t] if sep else None), wr[t].data_ptr(),
                 carry[t].data_ptr(), g_act[t].data_ptr(), n, prm, stream)

    def loss_of(st, ob, rw):
        return (st * ws).sum() + (ob * wo).sum() + (rw * wr).sum()

    def fused_api():
        sq, aq = s.clone().requires_grad_(True), a.clone().requires_grad_(True)
        st, ob, rw, _ = env.get_batch_trajectory(sq, aq)
        loss_of(st, ob, rw).backward()
        return sq.grad, aq.grad

    def chained_api():
        sq, aq = s.clone().requires_grad_(True), a.clone().requires_grad_(True)
        cur, S, O, R = sq, [sq], [], []
        for t in range(T):
            cur, o, r, _ = env.get_batch_transition(cur, aq[t])
            S.append(cur), O.append(o), R.append(r[:, 0])
        loss_of(torch.stack(S), torch.stack(O), torch.stack(R)).backward()
        return sq.grad, aq.grad

    big = n >= RESIDENT
    iters = 20 if big else 50
    api_iters = 5 if big else 20
    fwd_sub, fwd_once = OPS_TALLY[(fam, "fwd")]
    vjp_sub, vjp_once = OPS_TALLY[(fam, "vjp")]
    steps = n * T
    nbytes = {  # per call: arrays read and written once
        "fwd": 2 * n * row + steps * (row + esz + esz + 1 + (row if sep else 0)),  # state0 -> states[0]; per step states[t+1], action, reward, done, obs
        "bwd_all": n * (row + row) + steps * (row + esz + row + (row if sep else 0) + esz + esz),  # + g_states[0], g_state0
        "bwd_rewards": n * row + steps * (row + esz + esz + esz),
    }
    ops = {"fwd": steps * (fwd_sub * FR + fwd_once), "bwd_all": steps * (vjp_sub * FR + vjp_once), "bwd_rewards": steps * (vjp_sub * FR + vjp_once)}
    base = dict(family=fam, env=env_id, dtype=str(dtype).split(".")[-1], n=n, T=T, freq_rate=FR)
    out = []
    for what, fn in (("fwd", fwd), ("bwd_all", bwd_all), ("bwd_rewards", bwd_rewards)):
        ms = time_ms(fn, iters)
        t_bytes, t_ops = nbytes[what] / HBM_BPS, ops[what] / PEAK[dtype]
        bound = ("HBM" if t_bytes >= t_ops else "math (est.)") if big else "latency (batch < one resident grid)"
        out.append(dict(base, what=what, ms=round(ms, 4), bytes=nbytes[what], bytes_per_env_step=round(nbytes[what] / steps, 1), ops_est=ops[what],
                        GBps=round(nbytes[what] / ms / 1e6, 1), Gops_est=round(ops[what] / ms / 1e6, 1), bound=bound,
                        share_of_roofline=round(max(t_bytes, t_ops) * 1e3 / ms, 3), G_env_steps_per_s=round(steps / ms / 1e6, 2)))
    fused_kernels = out[0]["ms"] + out[1]["ms"]
    ms = time_ms(floor_fwd, max(3, iters // 5), warmup=2)
    out.append(dict(base, what="floor_fwd", ms=round(ms, 4), launches=T, fused_fwd_ms=out[0]["ms"], speedup_fused_fwd=round(ms / out[0]["ms"], 2)))
    ms = time_ms(floor_kernels, max(3, iters // 5), warmup=2)
    out.append(dict(base, what="floor_kernels", ms=round(ms, 4), launches=2 * T, fused_fwd_plus_bwd_all_ms=round(fused_kernels, 4),
                    speedup_fused_kernels=round(ms / fused_kernels, 2)))
    t_fused = time_ms(fused_api, api_iters, warmup=2)
    t_chain = time_ms(chained_api, api_iters, warmup=2)
    gf, gc = fused_api(), chained_api()
    diff = max(float(((x.double() - y.double()).abs() / (1 + y.double().abs())).max()) for x, y in zip(gf, gc))
    out.append(dict(base, what="fused_api", ms=round(t_fused, 4)))
    out.append(dict(base, what="chained_api", ms=round(t_chain, 4), speedup_fused_api=round(t_chain / t_fused, 2),
                    max_scaled_grad_diff_fused_vs_chained=diff))
    del states, obs, carry, ws, wo
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_bench_trajectory.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_trajectory.py measures on a CUDA device; there is none")
    name, power = card()
    lines = [json.dumps(dict(card=name, power_limit_and_max_sm_clock=power, freq_rate=FR, hbm_peak_Bps=HBM_BPS,
                             math_peak_flops={"float32": PEAK[torch.float32], "float64": PEAK[torch.float64]}))]
    print(lines[0], flush=True)
    for n, T in SIZES:
        for fam in ("cp", "i2p"):
            for dtype in (torch.float32, torch.float64):
                for rec in run(fam, dtype, n, T):
                    lines.append(json.dumps(rec))
                    print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
