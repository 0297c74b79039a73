"""Differentiable scoring: emei_sum_* / emei_reward_vjp_* / emei_reward_seq_vjp_* behind get_batch_reward,
get_batch_reward_terminal and get_batch_reward_terminal_seq.

The yardstick is a plain-torch float64 restatement of the 13 rewards, pinned to the oracle's *_reward functions on CPU; its
torch.autograd gradients are what the kernels are checked against on the GPU.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

import emei_b200 as E
from emei_b200 import _lib
from oracle import emei_oracle as O

IP = {"ip_rebound_balancing": "ReboundInvertedPendulumBalancing-v0", "ip_boundary_balancing": "BoundaryInvertedPendulumBalancing-v0",
      "ip_rebound_swingup": "ReboundInvertedPendulumSwingUp-v0", "ip_boundary_swingup": "BoundaryInvertedPendulumSwingUp-v0"}
I2P = {"i2p_rebound_balancing": "ReboundInvertedDoublePendulumBalancing-v0",
       "i2p_boundary_balancing": "BoundaryInvertedDoublePendulumBalancing-v0",
       "i2p_rebound_swingup": "ReboundInvertedDoublePendulumSwingUp-v0", "i2p_boundary_swingup": "BoundaryInvertedDoublePendulumSwingUp-v0"}
KINDS = {"balancing": "CartPoleBalancing-v0", "swingup": "CartPoleSwingUp-v0", **IP, **I2P, "hopper": "HopperRunning-v0",
         "halfcheetah": "HalfCheetahRunning-v0", "charged_ball": "ChargedBallCentering-v0"}
MUJOCO = ("hopper", "halfcheetah")
SEQ_KINDS = [k for k in KINDS if k.startswith("ip_") or k.startswith("i2p_") or k in MUJOCO]  # envs with get_batch_reward_terminal_seq
DIM = {"hopper": 12, "halfcheetah": 18, **{k: 6 for k in I2P}}
ADIM = {"hopper": 3, "halfcheetah": 6}
HOPPER = dict(fw=1.0, ctrl_w=1e-3, healthy=1.0, state=(-100.0, 100.0), z=(0.7, float("inf")))
CHEETAH = dict(fw=1.0, ctrl_w=0.1)
DT = 0.002 * 4


def dim(kind):
    return DIM.get(kind, 4)


# =============================================================================================
# the yardstick: plain torch, any dtype / device, differentiable by torch.autograd
# =============================================================================================
def torch_reward(kind, o, p=None, a=None, dt=DT):
    """reward [B, 1] of the family on rows o (p, a: Hopper / HalfCheetah), the expressions of oracle/emei_oracle.py"""
    if kind in ("balancing",) or kind.endswith("_balancing"):
        return torch.ones_like(o[:, :1])
    if kind == "swingup":
        return ((torch.cos(o[:, 2]) + 1) / 2).reshape(-1, 1)
    if kind.startswith("ip_"):
        return ((1 - torch.cos(o[:, 1])) / 2).reshape(-1, 1)
    if kind.startswith("i2p_"):
        y = torch.cos(o[:, 1]) + torch.cos(o[:, 1] + o[:, 2])
        r = (2 - y) / 4
        if kind == "i2p_boundary_swingup":
            r = r - (5e-3 * o[:, 4] ** 2 + 1e-4 * o[:, 5] ** 2)
        return r.reshape(-1, 1)
    if kind == "hopper":
        h = HOPPER
        with torch.no_grad():
            healthy = ((h["z"][0] < o[:, 1]) & (o[:, 1] < h["z"][1]) &
                       ((h["state"][0] < o[:, 2:]) & (o[:, 2:] < h["state"][1])).all(dim=1))
        return (healthy.to(o.dtype) * h["healthy"] + h["fw"] * (o[:, 0] - p[:, 0]) / dt - h["ctrl_w"] * (a * a).sum()).reshape(-1, 1)
    if kind == "halfcheetah":
        return (CHEETAH["fw"] * (o[:, 0] - p[:, 0]) / dt - CHEETAH["ctrl_w"] * (a * a).sum()).reshape(-1, 1)
    # charged ball (radius 1): 1 - rho; the gradient 0 at rho = 0
    r2 = o[:, 0] * o[:, 0] + o[:, 1] * o[:, 1]
    rho = torch.where(r2 > 0, torch.sqrt(torch.where(r2 > 0, r2, torch.ones_like(r2))), torch.zeros_like(r2))
    return (1 - rho / 1.0).reshape(-1, 1)


def oracle_reward(kind, o, p=None, a=None):
    if kind in ("balancing", "swingup"):
        return O.cartpole_reward(kind, o)
    if kind.startswith("ip_"):
        return O.ip_reward(kind, o)
    if kind.startswith("i2p_"):
        return O.i2p_reward(kind, o)
    if kind == "hopper":
        return O.hopper_reward(o, p, a, O.HopperParams(terminate_when_unhealthy=False, dt=DT))
    if kind == "halfcheetah":
        return O.halfcheetah_reward(o, p, a, O.HalfCheetahParams(dt=DT))
    return O.charged_ball_reward(o, O.ChargedBallParams())


def sample(kind, n, dtype, gen, device="cpu"):
    """finite rows (and for Hopper / HalfCheetah pre rows and actions) with the charged-ball origin and Hopper's health
    boundaries (z = 0.7, a state coordinate at +-100) among them"""
    d = dim(kind)
    scale = {"balancing": [3.0, 2.0, 0.3, 2.0], "swingup": [6.0, 2.0, 4.0, 2.0], "charged_ball": [0.7] * 4,
             "hopper": [1.0, 0.4, 0.15] + [60.0] * 9, "halfcheetah": [1.0] * 18}.get(kind)
    if scale is None:
        scale = [1.5, 2.0, 3.0, 5.0] if kind.startswith("ip") else [2.5, 0.8, 0.8, 3.0, 5.0, 5.0]
    sc = torch.tensor(scale, dtype=dtype, device=device)
    o = torch.randn((n, d), dtype=dtype, device=device, generator=gen) * sc
    p = a = None
    if kind == "hopper":
        o[:, 1] += 1.25
        o[::7, 1] = 0.7
        o[3::11, 2 + 3] = 100.0
        o[5::13, 2 + 5] = -100.0
    if kind == "charged_ball":
        o[::5, :2] = 0.0
    if kind in MUJOCO:
        p = torch.randn((n, d), dtype=dtype, device=device, generator=gen) * sc
        a = torch.rand((n, ADIM[kind]), dtype=dtype, device=device, generator=gen) * 2 - 1
    return o, p, a


def make_env(kind, dtype, **kw):
    if kind == "hopper":
        kw.setdefault("terminate_when_unhealthy", False)
    return E.make(KINDS[kind], dtype=dtype, device="cuda:0", **kw)


# =============================================================================================
# CPU
# =============================================================================================
@pytest.mark.parametrize("kind", list(KINDS))
def test_yardstick_is_the_oracle_reward(kind):
    g = torch.Generator().manual_seed(len(kind))
    o, p, a = sample(kind, 257, torch.float64, g)
    got = torch_reward(kind, o, p, a).numpy()
    want = oracle_reward(kind, o.numpy(), None if p is None else p.numpy(), None if a is None else a.numpy())
    assert got.shape == want.shape == (257, 1)
    np.testing.assert_allclose(got, want, rtol=1e-14, atol=1e-14)


def _scoring_params(family, dt=DT):
    s = _lib.ScoringParams()
    s.family, s.dt, s.radius, s.ctrl_cost_weight, s.forward_reward_weight = family, dt, 1.0, 1e-3, 1.0
    return s


def _validation_cases():
    """(entry, params, pointer args, sizes, {suffix: expected code}, what): every row is rejected (or is a no-op) before
    any launch, so the table runs without a device."""
    buf = (ctypes.c_double * 256)()
    al = (ctypes.addressof(buf) + 15) & ~15
    mis = al + 8
    sw, hop, cb, bal = (_scoring_params(f) for f in (_lib.IP_REBOUND_SWINGUP, _lib.HOPPER, _lib.CHARGED_BALL, _lib.CARTPOLE_BALANCING))
    bad_fam, neg_fam, zero_dt = _scoring_params(13), _scoring_params(-1), _scoring_params(_lib.HOPPER, dt=0.0)
    both = lambda c: {"_f32": c, "_f64": c}  # noqa: E731
    cases = [
        # emei_sum_*: x, n, out, workspace
        ("emei_sum", None, [None, None, None], (-1,), both(-4), "negative n"),
        ("emei_sum", None, [al, None, al], (8,), both(-1), "null out"),
        ("emei_sum", None, [al, al, None], (8,), both(-1), "null workspace"),
        ("emei_sum", None, [None, al, al], (8,), both(-1), "null x"),
        ("emei_sum", None, [mis, al, al], (8,), both(-5), "misaligned x"),
    ]
    # emei_reward_vjp_*: obs, action, g_reward, g_reward_sum, g_obs, g_pre_obs, g_action
    full = [al, None, al, None, al, al, None]
    hop_full = [None, al, al, al, al, al, al]

    def with_(args, **kw):
        out = list(args)
        for j, v in kw.items():
            out[int(j[1:])] = v
        return out

    for entry, sizes in (("emei_reward_vjp", (8,)), ("emei_reward_seq_vjp", (8, 4))):
        seq = entry == "emei_reward_seq_vjp"
        if seq:  # obs_seq, action, g_reward, g_reward_sum, g_obs_seq, g_action
            f, hf = [al, None, al, None, al, None], [None, al, al, al, al, al]
            ga = 5
        else:
            f, hf, ga = full, hop_full, 6
        neg = ((-1, 4), (8, -1)) if seq else ((-1,),)
        for s in neg:
            cases.append((entry, sw, [None] * len(f), s, both(-4), f"negative size {s}"))
            cases.append((entry, None, [None] * len(f), s, both(-4), f"negative size {s} before the params check"))
        cases += [
            (entry, None, f, sizes, both(-1), "null params"),
            (entry, bad_fam, f, sizes, both(-2), "family 13"),
            (entry, neg_fam, f, sizes, both(-2), "family -1"),
            (entry, zero_dt, hf, sizes, both(-6), "Hopper dt 0"),
            (entry, bad_fam, [None] * len(f), (0,) + sizes[1:], both(-2), "bad family before the empty batch"),
            (entry, sw, [None] * len(f), (0,) + sizes[1:], both(0), "empty batch: no-op"),
            (entry, sw, with_(f, a0=None), sizes, both(-1), "null obs of a family whose gradient reads it"),
            (entry, cb, with_(f, a0=None), sizes, both(-1), "null obs of the charged ball"),
            (entry, sw, with_(f, a2=None), sizes, both(-1), "null g_reward"),
            (entry, bal, with_(f, a0=None, a2=None), sizes, both(-1), "null g_reward of a constant reward"),
            (entry, sw, with_(f, **{f"a{ga}": al}), sizes, both(-6), "g_action of a family without control cost"),
            (entry, hop, with_(hf, a1=None), sizes, both(-1), "g_action without action"),
            (entry, hop, with_(hf, a3=None), sizes, both(-1), "g_action without g_reward_sum"),
            (entry, sw, with_(f, a0=mis), sizes, both(-5), "misaligned obs"),
            (entry, hop, with_(hf, a1=mis), sizes, both(-5), "misaligned action"),
            (entry, hop, with_(hf, **{f"a{ga}": mis}), sizes, both(-5), "misaligned g_action"),
            (entry, sw, with_(f, a4=mis), sizes, both(-5), "misaligned g_obs" + ("_seq" if seq else "")),
        ]
        if seq:
            cases += [
                (entry, sw, with_(f, a4=None), sizes, both(-1), "null g_obs_seq"),
                (entry, sw, [None] * len(f), (8, 0), both(0), "zero horizon: no-op"),
                # one HalfCheetah env: rows of 72 bytes in float32 lose 16-byte alignment at t >= 1, 144 in float64 keep it
                (entry, _scoring_params(_lib.HALFCHEETAH), [None, None, al, None, al, None], (1, 4), {"_f32": -5},
                 "odd HalfCheetah column count in float32"),
            ]
        else:
            cases.append((entry, sw, with_(f, a5=mis), sizes, both(-5), "misaligned g_pre_obs"))
    return cases, buf


def test_scoring_vjp_entry_points_validate_arguments_without_a_gpu():
    cases, _buf = _validation_cases()
    seen = set()
    for entry, prm, ptrs, sizes, want, what in cases:
        for sfx, code in want.items():
            f = getattr(_lib.lib, entry + sfx)
            if entry == "emei_sum":
                got = f(ptrs[0], sizes[0], ptrs[1], ptrs[2], None)
            else:
                got = f(*ptrs, *sizes, ctypes.byref(prm) if prm is not None else None, None)
            assert got == code, f"{entry}{sfx} {what}: got {got}, want {code}"
            seen.add(entry + sfx)
    assert seen == {b + s for b in ("emei_sum", "emei_reward_vjp", "emei_reward_seq_vjp") for s in ("_f32", "_f64")}


# =============================================================================================
# GPU
# =============================================================================================
def bar(dtype):
    return 1e-12 if dtype == torch.float64 else 1e-5


def assert_close(got, ref, dtype, what, scale=None):
    """|got - ref| <= bar * (1 + scale), scale = |ref| unless given"""
    got, ref = got.double(), ref.double()
    scale = ref.abs() if scale is None else scale
    err = ((got - ref).abs() / (1 + scale)).max().item() if got.numel() else 0.0
    print(f"scaled error {str(dtype)[6:]} {what}: {err:.3e}")  # with -s: the maxima DESIGN.md 4.9 records
    assert err <= bar(dtype), f"{what}: scaled error {err:.3e} > {bar(dtype):.0e}"
    return err


def one_shot_grads(env, kind, o, p, a, w):
    """kernel gradients of <w, get_batch_reward(o, p, a)>"""
    leaves = [t.detach().clone().requires_grad_(True) if t is not None else None for t in (o, p, a)]
    r = env.get_batch_reward(*leaves)
    assert r.grad_fn is not None
    (r * w).sum().backward()
    return [t.grad if t is not None else None for t in leaves], r


def yardstick_grads(kind, o, p, a, w):
    leaves = [t.detach().double().clone().requires_grad_(True) if t is not None else None for t in (o, p, a)]
    r = torch_reward(kind, *leaves)
    if r.requires_grad:  # a constant reward has no graph: its gradient is zero
        (r * w.double()).sum().backward()
    return [t.grad if t.grad is not None else torch.zeros_like(t) for t in leaves if t is not None]


@pytest.mark.gpu
@pytest.mark.parametrize("n", (37, 9001, 2**20 + 3))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("kind", list(KINDS))
def test_one_shot_gradients_vs_yardstick(kind, dtype, n):
    env = make_env(kind, dtype)
    g = torch.Generator(device="cuda").manual_seed(n + len(kind))
    o, p, a = sample(kind, n, dtype, g, "cuda")
    w = torch.randn((n, 1), dtype=dtype, device="cuda", generator=g)
    got, r = one_shot_grads(env, kind, o, p, a, w)
    ref = yardstick_grads(kind, o, p, a, w)
    assert got[0] is not None  # a constant reward gives a zero gradient, not None
    assert_close(got[0], ref[0], dtype, "d/d obs")
    if kind in MUJOCO:
        assert_close(got[1], ref[1], dtype, "d/d pre_obs")
        assert_close(got[2], ref[2], dtype, "d/d action")
    assert got[0].dtype == dtype and got[0].shape == o.shape


@pytest.mark.gpu
@pytest.mark.parametrize("n", (256, 1001))
@pytest.mark.parametrize("T", (1, 7, 33))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("kind", SEQ_KINDS)
def test_seq_gradients_vs_yardstick(kind, dtype, T, n):
    """obs_seq [T+1, n, D]; float32 HalfCheetah / I2P with n = 1001 take score_seq's flat fallback"""
    env = make_env(kind, dtype)
    g = torch.Generator(device="cuda").manual_seed(T * 1000 + n + len(kind))
    seq, _, _ = sample(kind, (T + 1) * n, dtype, g, "cuda")
    seq = seq.reshape(T + 1, n, -1)
    a = (torch.rand((T, n, ADIM[kind]), dtype=dtype, device="cuda", generator=g) * 2 - 1) if kind in MUJOCO else None
    w = torch.randn((T, n, 1), dtype=dtype, device="cuda", generator=g)
    s_leaf = seq.clone().requires_grad_(True)
    a_leaf = a.clone().requires_grad_(True) if a is not None else None
    r, d = env.get_batch_reward_terminal_seq(s_leaf, a_leaf)
    assert r.grad_fn is not None and d.grad_fn is None and r.shape == (T, n, 1)
    (r * w).sum().backward()
    # the yardstick on separate obs / pre_obs leaves: row t of d/d obs_seq is the sum of transition t-1's obs term and
    # transition t's pre_obs term
    d_ = seq.shape[2]
    o64 = seq[1:].double().reshape(T * n, d_).clone().requires_grad_(True)
    p64 = seq[:-1].double().reshape(T * n, d_).clone().requires_grad_(True)
    a64 = a.double().clone().requires_grad_(True) if a is not None else None
    ref_r = torch_reward(kind, o64, p64, a64.reshape(T * n, -1) if a64 is not None else None)
    if ref_r.requires_grad:  # a constant reward has no graph: its gradient is zero
        (ref_r * w.double().reshape(-1, 1)).sum().backward()
    go = (o64.grad if o64.grad is not None else torch.zeros_like(o64)).reshape(T, n, d_)
    gp = (p64.grad if p64.grad is not None else torch.zeros_like(p64)).reshape(T, n, d_)
    ref, mag = torch.zeros_like(seq, dtype=torch.float64), torch.zeros_like(seq, dtype=torch.float64)
    ref[1:] += go
    ref[:-1] += gp
    mag[1:] += go.abs()
    mag[:-1] += gp.abs()
    # float32: the two terms are rounded before they are added (the bits of the one-shot layout, whose two rows autograd adds),
    # so a row's error scales with the terms' magnitudes (Hopper / HalfCheetah: fw / dt * |g| ~ 125 |g| each), not their sum
    assert_close(s_leaf.grad, ref, dtype, "d/d obs_seq", scale=mag if dtype == torch.float32 else None)
    if a is not None:
        assert_close(a_leaf.grad, a64.grad, dtype, "d/d action")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_gradcheck_float64(kind):
    env = make_env(kind, torch.float64)
    g = torch.Generator(device="cuda").manual_seed(5)
    o, p, a = sample(kind, 6, torch.float64, g, "cuda")
    if kind == "hopper":
        o[:, 1] = 1.25  # away from the health boundaries
        o[:, 2:] = o[:, 2:].clamp(-50, 50)
    if kind == "charged_ball":
        o[:, :2] = o[:, :2] + 0.5  # away from the origin
    inputs = tuple(t.clone().requires_grad_(True) for t in (o, p, a) if t is not None)
    if kind in MUJOCO:
        f = lambda o_, p_, a_: env.get_batch_reward(o_, p_, a_)  # noqa: E731
    else:
        f = lambda o_: env.get_batch_reward(o_)  # noqa: E731
    assert torch.autograd.gradcheck(f, inputs, eps=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("kind", SEQ_KINDS)
def test_seq_layout_bit_equal_to_one_shot(kind, dtype):
    """get_batch_reward_terminal_seq's gradients == get_batch_reward on seq[1:] / seq[:-1], as separate allocations and
    as aliased views of one tensor"""
    env = make_env(kind, dtype)
    T, n = 9, 512
    g = torch.Generator(device="cuda").manual_seed(17 + len(kind))
    seq, _, _ = sample(kind, (T + 1) * n, dtype, g, "cuda")
    seq = seq.reshape(T + 1, n, -1)
    d_ = seq.shape[2]
    a = (torch.rand((T, n, ADIM[kind]), dtype=dtype, device="cuda", generator=g) * 2 - 1) if kind in MUJOCO else None
    w = torch.randn((T, n, 1), dtype=dtype, device="cuda", generator=g)
    mj = kind in MUJOCO

    s0 = seq.clone().requires_grad_(True)
    a0 = a.clone().requires_grad_(True) if mj else None
    r0, _ = env.get_batch_reward_terminal_seq(s0, a0)
    (r0 * w).sum().backward()

    # aliased views
    s1 = seq.clone().requires_grad_(True)
    a1 = a.clone().requires_grad_(True) if mj else None
    args = (s1[1:].reshape(T * n, d_), s1[:-1].reshape(T * n, d_), a1.reshape(T * n, -1)) if mj else (s1[1:].reshape(T * n, d_),)
    r1 = env.get_batch_reward(*args)
    (r1 * w.reshape(-1, 1)).sum().backward()
    assert torch.equal(r0.reshape(-1, 1), r1)
    assert torch.equal(s0.grad, s1.grad)
    if mj:
        assert torch.equal(a0.grad, a1.grad)

    # separate allocations
    o2 = seq[1:].reshape(T * n, d_).clone().requires_grad_(True)
    p2 = seq[:-1].reshape(T * n, d_).clone().requires_grad_(True) if mj else None
    a2 = a.reshape(T * n, -1).clone().requires_grad_(True) if mj else None
    r2 = env.get_batch_reward(o2, p2, a2) if mj else env.get_batch_reward(o2)
    (r2 * w.reshape(-1, 1)).sum().backward()
    want = torch.zeros_like(seq)
    want[1:] += o2.grad.reshape(T, n, d_)
    if mj:
        want[:-1] += p2.grad.reshape(T, n, d_)
        assert torch.equal(a0.grad.reshape(T * n, -1), a2.grad)
    assert torch.equal(s0.grad, want)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("kind", MUJOCO)
def test_control_cost_couples_every_action(kind, dtype):
    """changing one row's cotangent by dg changes every action's gradient by -2 ctrl_w a dg"""
    env = make_env(kind, dtype)
    n = 3001
    g = torch.Generator(device="cuda").manual_seed(3)
    o, p, a = sample(kind, n, dtype, g, "cuda")
    w = torch.randn((n, 1), dtype=dtype, device="cuda", generator=g)
    (_, _, ga0), _ = one_shot_grads(env, kind, o, p, a, w)
    w2 = w.clone()
    w2[1234] += 0.75
    (_, _, ga1), _ = one_shot_grads(env, kind, o, p, a, w2)
    ctrl_w = HOPPER["ctrl_w"] if kind == "hopper" else CHEETAH["ctrl_w"]
    delta = (ga1.double() - ga0.double())
    want = -2 * ctrl_w * a.double() * 0.75
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    assert ((delta - want).abs() <= tol * (1 + ga0.double().abs())).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("hopper", "i2p_boundary_swingup", "charged_ball"))
def test_unchanged_path_without_grad(kind):
    """no requires_grad, or torch.no_grad(): today's launches and bits, no grad_fn; numpy in, numpy out"""
    env = make_env(kind, torch.float64)
    g = torch.Generator(device="cuda").manual_seed(11)
    o, p, a = sample(kind, 4099, torch.float64, g, "cuda")
    args = (o, p, a) if kind in MUJOCO else (o,)

    def run(*xs):
        c0 = _lib.launch_count
        r = env.get_batch_reward(*xs)
        return r, _lib.launch_count - c0

    r0, n0 = run(*args)
    assert r0.grad_fn is None
    leaves = [x.clone().requires_grad_(True) for x in args]
    with torch.no_grad():
        r1, n1 = run(*leaves)
    assert r1.grad_fn is None and torch.equal(r0, r1) and n1 == n0
    r2, n2 = run(*leaves)  # differentiable: the same forward kernels
    assert r2.grad_fn is not None and torch.equal(r0, r2.detach()) and n2 == n0
    rn = env.get_batch_reward(*(x.cpu().numpy() for x in args))
    assert isinstance(rn, np.ndarray) and np.array_equal(rn, r0.cpu().numpy())
    if kind in MUJOCO:
        T, k = 3, 256
        seq = o[: (T + 1) * k].reshape(T + 1, k, -1)
        act = a[: T * k].reshape(T, k, -1)
        c0 = _lib.launch_count
        rs, ds = env.get_batch_reward_terminal_seq(seq, act)
        ns = _lib.launch_count - c0
        with torch.no_grad():
            c0 = _lib.launch_count
            rs1, _ = env.get_batch_reward_terminal_seq(seq.clone().requires_grad_(True), act)
            assert _lib.launch_count - c0 == ns
        assert rs.grad_fn is None and rs1.grad_fn is None and torch.equal(rs, rs1)


@pytest.mark.gpu
def test_reward_after_terminal_on_grad_tensors_has_grad_fn():
    env = make_env("hopper", torch.float64)
    g = torch.Generator(device="cuda").manual_seed(2)
    o, p, a = (t.requires_grad_(True) for t in sample("hopper", 1024, torch.float64, g, "cuda"))
    d = env.get_batch_terminal(o, p, a)
    r = env.get_batch_reward(o, p, a)
    assert d.grad_fn is None and r.grad_fn is not None
    r.sum().backward()
    assert a.grad is not None and o.grad is not None


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("halfcheetah", "i2p_boundary_swingup"))
def test_backward_is_deterministic(kind):
    env = make_env(kind, torch.float32)
    T, n = 16, 4096
    g = torch.Generator(device="cuda").manual_seed(8)
    seq = sample(kind, (T + 1) * n, torch.float32, g, "cuda")[0].reshape(T + 1, n, -1)
    a = torch.rand((T, n, ADIM.get(kind, 1)), device="cuda", generator=g) if kind in MUJOCO else None
    w = torch.randn((T, n, 1), device="cuda", generator=g)
    out = []
    for _ in range(2):
        s = seq.clone().requires_grad_(True)
        al = a.clone().requires_grad_(True) if a is not None else None
        r, _ = env.get_batch_reward_terminal_seq(s, al)
        (r * w).sum().backward()
        out.append((s.grad, al.grad if al is not None else None))
    assert torch.equal(out[0][0], out[1][0])
    if a is not None:
        assert torch.equal(out[0][1], out[1][1])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dist_worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from emei_b200.dist import shard_range

        calls = [0]
        real = dist.all_reduce

        def counting(*args, **kw):
            calls[0] += 1
            return real(*args, **kw)

        dist.all_reduce = counting
        n = 5001
        g = torch.Generator(device="cuda").manual_seed(21)  # the same global batch on every rank
        o, p, a = sample("hopper", n, torch.float64, g, "cuda")
        w = torch.randn((n, 1), dtype=torch.float64, device="cuda", generator=g)
        b, e = shard_range(n)
        res = {}
        for scope in ("global", "local"):
            env = make_env("hopper", torch.float64, ctrl_cost_scope=scope)
            # the unsharded rows (one process's view of the whole batch, no exchange)
            full = make_env("hopper", torch.float64, ctrl_cost_scope="local")
            ref, _ = one_shot_grads(full, "hopper", o, p, a, w)
            sl = slice(b, e)
            before = calls[0]
            got, _ = one_shot_grads(env, "hopper", o[sl], p[sl], a[sl], w[sl])
            issued = calls[0] - before
            if scope == "global":
                ok = all(bool(((x - y[sl]).abs() <= 1e-12 * (1 + y[sl].abs())).all()) for x, y in zip(got, ref))
            else:  # local: the shard's own control cost, i.e. the unsharded rows of the shard alone
                ref_l, _ = one_shot_grads(full, "hopper", o[sl], p[sl], a[sl], w[sl])
                ok = all(torch.equal(x, y) for x, y in zip(got, ref_l))
            res[scope] = (ok, issued)
        q.put((rank, res))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_rank_sharded_backward():
    """two gloo ranks on one GPU: the sharded Hopper backward (G all-reduced) equals the unsharded rows; with
    ctrl_cost_scope="local" no collective is issued"""
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = sorted(q.get(timeout=300) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.kill()
                p.join()
    assert [p.exitcode for p in procs] == [0, 0]
    for rank, r in res:
        ok_g, issued_g = r["global"]
        ok_l, issued_l = r["local"]
        assert ok_g and ok_l, (rank, r)
        assert issued_g == 2  # the forward's sum of squares and the backward's sum of cotangents
        assert issued_l == 0
