"""Times the derivative kernels of the analytic steps against the forward step and against torch autograd through a
plain-torch restatement of the same step (what a user without these kernels would run).

For each family (cart-pole kernel: ContinuousCartPoleSwingUp; I2P kernel: BoundaryInvertedDoublePendulumSwingUp),
precision and batch size (freq_rate 4):
  fwd     the stateless step kernel (get_batch_transition's forward)
  vjp     emei_*_step_vjp_* with every cotangent present (get_batch_transition's backward)
  jac     emei_*_step_jacobian_* with reward_grad
  torch   forward + backward of the plain-torch restatement on the GPU (torch.autograd.grad, the same cotangents)
Every kernel line is one C-ABI launch into preallocated buffers (no allocation inside the timed loop) and carries its
algorithmic bytes (arrays read + written once), an ESTIMATED operation count and the roofline bound that limits it:
max(bytes / HBM peak, ops / math peak) against the measured time.  The operation counts are a per-term tally of the
arithmetic written in the source (OPS_TALLY below: every +, -, *, / and a sincos counted as one operation each, an FMA as
two); they are not instruction counts, and the float32 forward step takes the TMA kernel's lean arithmetic, which the
tally of the generic expressions overstates, so the "bound" column is an estimate.  Peaks: the measured 6.55 TB/s copy rate
(DESIGN.md section 4.1) and profiles/math_peaks.json (FP32 63.7, FP64 35.87 TFLOP/s).  A 2^20-env working set fits in
the 126 MB L2; 2^24 envs do not, so those lines are HBM-resident.  Card name and power limit are read in the same run.

    python scripts/bench_autodiff.py [--out FILE] [--sizes 20,24]
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib, autodiff  # noqa: E402

HBM_BPS = 6.55e12
PEAK = {torch.float32: 63.7e12, torch.float64: 35.87e12}
FR = 4
# ESTIMATED operations per env: (per sub-step, once per env), a per-term tally of the expressions in the source.
OPS_TALLY = {
    # kernels.cuh cartpole_env_step: sincos 2, temp 5, den 5, th_acc 4, x_acc 4, Euler 8 | reward + done ~8
    ("cp", "fwd"): (28, 8),
    # derivs.cuh cartpole_tangent: sincos 2, sign 2, primal accel 18, partial coefficients 33 (inv_den, t_th, t_w, den_th,
    # B_th, B_w, B_F, A_th, A_w, A_F), 5 tangent columns x (dxa 5 + dta 5 + 4 updates x 2) = 90, Euler 8 -> 153 |
    # epilogue: force + slope 4, reward slope 3, w 12, 5 columns x 7 = 35 -> vjp 54; jac: 4 + 3 + 35 -> 42
    ("cp", "vjp"): (153, 54),
    ("cp", "jac"): (153, 42),
    # i2p.cuh i2p_env_step: sincos 6, sign 4, A 8, b 29, LDL^T 13, one solve with divisions 15, Euler 12 -> 87 |
    # observation 10, reward 8, finite 6 -> 24
    ("i2p", "fwd"): (87, 24),
    # derivs.cuh i2p_tangent: sincos 6, sign 4, A 8, b 29, LDL^T 13, 6 solves x 15 = 90, right-hand sides 63
    # (dA z and db for th0, th1, w0, w1), 7 tangent columns x 3 x (dz 9 + 2 updates x 2) = 273, Euler 12 -> 498 |
    # epilogue: clamp 4, reward slope 16, w 6 x 4 = 24, 7 columns x 11 = 77 -> vjp 121; jac: 4 + 16 + 77 -> 97
    ("i2p", "vjp"): (498, 121),
    ("i2p", "jac"): (498, 97),
}
FAMILY = {"cp": ("ContinuousCartPoleSwingUp-v0", 4), "i2p": ("BoundaryInvertedDoublePendulumSwingUp-v0", 6)}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        power = f"unavailable ({e})"
    return name, power


def time_ms(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


# ---- plain-torch restatements of the two steps (forward Euler, freq_rate sub-steps, observation, reward) ----------
def cp_torch(env, y, a):
    force = env.force_mag * a
    pml, tm = env.mass_pole * env.length, env.total_mass
    for _ in range(env.freq_rate):
        x, xd, th, thd = y.unbind(1)
        s, c = torch.sin(th), torch.cos(th)
        temp = (force + pml * thd * thd * s) / tm
        tha = (env.gravity * s - c * temp) / (env.length * (4.0 / 3.0 - env.mass_pole * c * c / tm))
        xa = temp - pml * tha * c / tm
        y = y + env.real_time_scale * torch.stack([xd, xa, thd, tha], 1)
    return y, y, (torch.cos(y[:, 2]) + 1) / 2


def i2p_torch(env, y, a):
    M, m0, m1, l0, l1, g = env.mass_cart, env.mass_pole, env.mass_pole, env.pole_half_length, env.pole_half_length, env.gravity
    k_a, k_b, k_c, k_d = (m0 + 2 * m1) * l0, m1 * l1, 2 * m1 * l0 * l1, 4.0 / 3.0 * m1 * l1 * l1
    k_e, k_g1, a00 = 4.0 / 3.0 * m0 * l0 * l0 + 4 * m1 * l0 * l0 + k_d, g * l0 * (m0 + 2 * m1), M + m0 + m1
    F = env.gear * a.clamp(-1.0, 1.0)
    h, sign = env.real_time_scale, -1.0
    for _ in range(env.freq_rate):
        th0, th1, w0, w1 = y[:, 1], y[:, 2], y[:, 4], y[:, 5]
        s0, c0, s1, c1 = sign * torch.sin(th0), sign * torch.cos(th0), torch.sin(th1), torch.cos(th1)
        s01, c01 = sign * torch.sin(th0 + th1), sign * torch.cos(th0 + th1)
        a01, a02, a11, a12, a22 = k_a * c0 + k_b * c01, k_b * c01, k_e + 2 * k_c * c1, k_c * c1 + k_d, k_d
        ws = w0 + w1
        b0 = F + k_a * s0 * w0 * w0 + k_b * s01 * ws * ws
        b1 = k_g1 * s0 + g * k_b * s01 + k_c * s1 * w1 * (2 * w0 + w1)
        b2 = k_b * (g * s01 - 2 * l0 * s1 * w0 * w0)
        l10, l20 = a01 / a00, a02 / a00
        d1, t12 = a11 - l10 * a01, a12 - l10 * a02
        l21 = t12 / d1
        d2 = a22 - l20 * a02 - l21 * t12
        y1 = b1 - l10 * b0
        y2 = b2 - l20 * b0 - l21 * y1
        z2 = y2 / d2
        z1 = y1 / d1 - l21 * z2
        z0 = b0 / a00 - l10 * z1 - l20 * z2
        y = torch.cat([y[:, :3] + y[:, 3:] * h, y[:, 3:] + torch.stack([z0, z1, z2], 1) * h], 1)
    o1 = torch.remainder(y[:, 1] + math.pi, 2) * math.pi - math.pi
    o2 = torch.remainder(y[:, 2] + math.pi, 2) * math.pi - math.pi
    obs = torch.stack([y[:, 0], o1, o2, y[:, 3], y[:, 4], y[:, 5]], 1)
    r = (2 - (torch.cos(o1) + torch.cos(o1 + o2))) / 4 - (5e-3 * y[:, 4] ** 2 + 1e-4 * y[:, 5] ** 2)
    return y, obs, r


def run(fam, dtype, log2n):
    env_id, D = FAMILY[fam]
    n = 1 << log2n
    env = E.make(env_id, freq_rate=FR, dtype=dtype, device="cuda:0")
    gen = torch.Generator(device="cuda:0").manual_seed(log2n)
    y = (torch.rand(n, D, device="cuda:0", dtype=dtype, generator=gen) * 2 - 1) * 2.0
    a = torch.rand(n, device="cuda:0", dtype=dtype, generator=gen) * 2 - 1
    eng, s, act, _ = autodiff._inputs(env, y, a)
    gs, go = torch.randn_like(s), torch.randn_like(s)
    gr = torch.randn(n, device="cuda:0", dtype=dtype, generator=gen)
    esz = s.element_size()
    row = D * esz
    nbytes = {  # arrays read and written once per call
        "fwd": n * (row + esz + row + (row if fam == "i2p" else 0) + esz + 1),  # state, action -> state, obs (I2P), reward, done
        "vjp": n * (row + esz + row + row + esz + row + esz),  # state, action, g_state_out, g_obs, g_reward -> g_state_in, g_action
        "jac": n * (row + esz + D * (D + 1) * esz + (D + 1) * esz),  # state, action -> jac, reward_grad
    }
    # preallocated outputs: each timed call is exactly one launch
    s_out, obs_out = torch.empty_like(s), (torch.empty_like(s) if fam == "i2p" else None)
    reward, done = torch.empty(n, dtype=dtype, device="cuda:0"), torch.empty(n, dtype=torch.uint8, device="cuda:0")
    g_in, g_act = torch.empty_like(s), torch.empty(n, dtype=dtype, device="cuda:0")
    jac, rg = torch.empty(n, D, D + 1, dtype=dtype, device="cuda:0"), torch.empty(n, D + 1, dtype=dtype, device="cuda:0")
    eng.params.action_kind = _lib.ACTION_CONTINUOUS_F32 if dtype == torch.float32 else _lib.ACTION_CONTINUOUS_F64
    prm, stream, base = ctypes.byref(eng.params), torch.cuda.current_stream().cuda_stream, eng._step_entry
    sfx = env._suffix
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    fns = {
        "fwd": lambda: _lib.call(base + sfx, s.data_ptr(), s_out.data_ptr(), ptr(obs_out), act.data_ptr(), reward.data_ptr(),
                                 done.data_ptr(), None, n, prm, stream),
        "vjp": lambda: _lib.call(base + "_vjp" + sfx, s.data_ptr(), act.data_ptr(), gs.data_ptr(), go.data_ptr(), gr.data_ptr(),
                                 g_in.data_ptr(), g_act.data_ptr(), n, prm, stream),
        "jac": lambda: _lib.call(base + "_jacobian" + sfx, s.data_ptr(), act.data_ptr(), jac.data_ptr(), rg.data_ptr(), n, prm, stream),
    }
    iters = 50 if log2n <= 20 else 10
    out = []
    for k, fn in fns.items():
        ms = time_ms(fn, iters)
        per_sub, once = OPS_TALLY[(fam, k)]
        ops = n * (per_sub * FR + once)
        t_bytes, t_ops = nbytes[k] / HBM_BPS, ops / PEAK[dtype]
        bound = "HBM" if t_bytes >= t_ops else "math (est.)"
        out.append(dict(family=fam, dtype=str(dtype).split(".")[-1], n=n, what=k, ms=round(ms, 4), bytes=nbytes[k], ops_est=ops,
                        GBps=round(nbytes[k] / ms / 1e6, 1), Gops_est=round(ops / ms / 1e6, 1), bound=bound,
                        share_of_bound=round(max(t_bytes, t_ops) * 1e3 / ms, 3), G_envs_per_s=round(n / ms / 1e6, 2)))
    del jac, rg
    # torch autograd through the plain-torch restatement: forward + backward with the same cotangents
    step = cp_torch if fam == "cp" else i2p_torch
    yq, aq = s.clone().requires_grad_(True), act.clone().requires_grad_(True)

    def torch_fb():
        ys, obs, r = step(env, yq, aq)
        loss = (ys * gs).sum() + (obs * go).sum() + (r * gr).sum()
        return torch.autograd.grad(loss, (yq, aq))

    ms = time_ms(torch_fb, max(3, iters // 5), warmup=2)
    g_ref = torch_fb()
    g_ker = eng.vjp(s, act, gs, go, gr, True)
    diff = max(float(((g_ker[0] - g_ref[0]).abs() / (1 + g_ref[0].abs())).max()), float(((g_ker[1] - g_ref[1]).abs() / (1 + g_ref[1].abs())).max()))
    kern = out[0]["ms"] + out[1]["ms"]
    out.append(dict(family=fam, dtype=str(dtype).split(".")[-1], n=n, what="torch_autograd", ms=round(ms, 4),
                    G_envs_per_s=round(n / ms / 1e6, 2), kernel_fwd_plus_vjp_ms=round(kern, 4), speedup=round(ms / kern, 1),
                    max_scaled_diff_vs_vjp=diff))
    del yq, aq, g_ref, g_ker
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="20,24")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_autodiff.py measures on a CUDA device; there is none")
    name, power = card()
    head = dict(card=name, power_limit_and_max_sm_clock=power, freq_rate=FR, hbm_peak_Bps=HBM_BPS,
                math_peak_flops={"float32": PEAK[torch.float32], "float64": PEAK[torch.float64]})
    lines = [json.dumps(head)]
    print(lines[0], flush=True)
    for log2n in (int(v) for v in args.sizes.split(",")):
        for fam in ("cp", "i2p"):
            for dtype in (torch.float32, torch.float64):
                for rec in run(fam, dtype, log2n):
                    lines.append(json.dumps(rec))
                    print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
