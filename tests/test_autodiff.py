"""Derivatives of the analytic steps: emei_*_step_jacobian_* / emei_*_step_vjp_* and the autograd path
(emei_b200.autodiff, env.get_batch_transition / env.get_batch_jacobian).

The yardstick is a complex-step derivative of the oracle's own dynamics (oracle/emei_oracle.py ``cartpole_accel`` /
``i2p_accel`` evaluated in complex128 around an explicit forward-Euler loop): ``Im f(x + i h) / h`` with h = 1e-30 has
no cancellation, so it is exact to float64 rounding.  The model differentiated is the one the step kernels evaluate:
plain Euler sub-steps (the cart-pole float32 increment rounding excluded), the control clamp, the observation (IP wrap
slope 1, I2P current_obs quirk slope pi) and the variant's reward on it.
"""
import ctypes
import itertools
import math

import numpy as np
import pytest
import torch

import emei_b200 as E
from emei_b200 import _lib, autodiff
from oracle import emei_oracle as O

H_CS = 1e-30  # complex-step size
DT = 0.02

CARTPOLE_IDS = ["CartPoleBalancing-v0", "CartPoleSwingUp-v0", "ContinuousCartPoleBalancing-v0", "ContinuousCartPoleSwingUp-v0"]
IP_IDS = ["ReboundInvertedPendulumBalancing-v0", "BoundaryInvertedPendulumBalancing-v0", "ReboundInvertedPendulumSwingUp-v0",
          "BoundaryInvertedPendulumSwingUp-v0"]
I2P_IDS = ["ReboundInvertedDoublePendulumBalancing-v0", "BoundaryInvertedDoublePendulumBalancing-v0",
           "ReboundInvertedDoublePendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"]
ALL_IDS = CARTPOLE_IDS + IP_IDS + I2P_IDS


class Spec:
    """what the complex-step model needs to know about an env id"""

    def __init__(self, env_id):
        self.id = env_id
        self.fam = "i2p" if "Double" in env_id else ("ip" if "Pendulum" in env_id else "cp")
        self.swingup = "SwingUp" in env_id
        self.boundary = env_id.startswith("Boundary")
        self.continuous = self.fam != "cp" or env_id.startswith("Continuous")
        self.D = 6 if self.fam == "i2p" else 4
        self.ctrl = {"cp": (-1.0, 1.0), "ip": (-3.0, 3.0), "i2p": (-1.0, 1.0)}[self.fam]


def _clamp(a, lo, hi):
    """clamp with torch.clamp's gradient: the perturbation passes where lo <= Re a <= hi (inclusive)"""
    inside = (a.real >= lo) & (a.real <= hi)
    return np.where(inside, a, np.clip(a.real, lo, hi) + 0j)


def model_step(spec, y, a, fr, f32_force=True):
    """complex128 rows y [B,D], actions a [B] -> (next state [B,D], obs [B,D], reward [B]); the real-valued model the step
    kernels evaluate.  f32_force=False: the continuous cart-pole force unrounded (for finite differences)."""
    y = np.array(y, dtype=np.complex128)
    a = np.asarray(a, dtype=np.complex128).reshape(-1)
    B = y.shape[0]
    with np.errstate(all="ignore"):
        if spec.fam == "cp":
            p = O.cartpole_params("swingup" if spec.swingup else "balancing")
            if spec.continuous and not f32_force:
                F = p.force_mag * a
            elif spec.continuous:  # the step's force is the float32 product force_mag * a (O.cartpole_force); slope force_mag
                F = O.cartpole_force(a.real.reshape(-1, 1), True, p) + 1j * p.force_mag * a.imag
            else:
                F = np.where(a.real == 1, p.force_mag, -p.force_mag) + 0j
            for _ in range(fr):
                s, c = np.sin(y[:, 2]), np.cos(y[:, 2])
                xa, ta = O.cartpole_accel(y[:, 1], y[:, 2], y[:, 3], F, p, s, c)
                y = y + DT * np.stack([y[:, 1], xa, y[:, 3], ta], axis=1)
            obs = y
            r = (np.cos(y[:, 2]) + 1) / 2 if spec.swingup else np.ones(B, np.complex128)
        elif spec.fam == "ip":
            p = O.InvertedPendulumParams()
            F = p.gear * _clamp(a, p.ctrl_low, p.ctrl_high)
            sign = -1.0 if spec.swingup else 1.0
            for _ in range(fr):
                s, c = sign * np.sin(y[:, 1]), sign * np.cos(y[:, 1])
                xa, ta = O.cartpole_accel(y[:, 2], y[:, 1], y[:, 3], F, p, s, c)
                y = y + DT * np.stack([y[:, 2], y[:, 3], xa, ta], axis=1)
            obs = y.copy()
            obs[:, 1] = y[:, 1] - 2 * np.pi * np.floor((y[:, 1].real + np.pi) / (2 * np.pi))  # (th + pi) mod 2pi - pi
            r = (1 - np.cos(obs[:, 1])) / 2 if spec.swingup else np.ones(B, np.complex128)
        else:
            p = O.I2PParams()
            F = p.gear * _clamp(a, p.ctrl_low, p.ctrl_high)
            for _ in range(fr):
                acc = O.i2p_accel(y[:, :3], y[:, 3:], F, spec.swingup, p, dtype=np.complex128)
                y = np.concatenate([y[:, :3] + y[:, 3:] * DT, y[:, 3:] + acc * DT], axis=1)
            obs = y.copy()
            t = y[:, 1:3] + np.pi
            obs[:, 1:3] = (t - 2 * np.floor(t.real / 2)) * np.pi - np.pi  # ((th + pi) mod 2) * pi - pi  (sic)
            if spec.swingup:
                yy = np.cos(obs[:, 1]) + np.cos(obs[:, 1] + obs[:, 2])
                r = (2 - yy) / 4
                if spec.boundary:
                    r = r - (5e-3 * obs[:, 4] ** 2 + 1e-4 * obs[:, 5] ** 2)
            else:
                r = np.ones(B, np.complex128)
    return y, obs, r


def cs_jacobian(spec, y, a, fr, f32_force=True):
    """complex-step (jac [B,D,D+1], obs_jac [B,D,D+1], reward_grad [B,D+1]) of ``model_step``"""
    y = np.asarray(y, dtype=np.float64)
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    B, D = y.shape
    J, JO, RG = np.zeros((B, D, D + 1)), np.zeros((B, D, D + 1)), np.zeros((B, D + 1))
    for c in range(D + 1):
        yc, ac = y.astype(np.complex128), a.astype(np.complex128)
        if c < D:
            yc[:, c] += 1j * H_CS
        else:
            ac += 1j * H_CS
        yn, o, r = model_step(spec, yc, ac, fr, f32_force)
        J[:, :, c], JO[:, :, c], RG[:, c] = yn.imag / H_CS, o.imag / H_CS, r.imag / H_CS
    return J, JO, RG


def sample_rows(spec, n, rng, swing_omega=20.0):
    """states spread over the reachable set (swing-up ids: |omega| up to ~20) and actions on both sides of the clamp, with
    rows exactly on its boundary"""
    D = spec.D
    if spec.fam == "cp":
        scale = np.array([2.0, 3.0, np.pi, 8.0])
    elif spec.fam == "ip":
        scale = np.array([1.5, np.pi, 3.0, 8.0])
    else:
        scale = np.array([2.0, np.pi, np.pi, 3.0, 8.0, 8.0])
    if spec.swingup:  # the angular velocities
        scale[[4, 5] if spec.fam == "i2p" else [3]] = swing_omega
    y = rng.uniform(-1, 1, size=(n, D)) * scale
    lo, hi = spec.ctrl
    if spec.continuous:
        a = rng.uniform(1.3 * lo, 1.3 * hi, size=n)
        a[1::17], a[2::17] = hi, lo  # on the clamp's boundary: the gradient passes
    else:
        a = rng.integers(0, 2, size=n).astype(np.float64)
    return y, a


def graph_support(J):
    """per-sample local graph in the reference's orientation: rows = (state, action) inputs, columns = next state, J - I"""
    D = J.shape[1]
    G = np.swapaxes(J, 1, 2).copy()  # [B, D+1, D]
    G[:, np.arange(D), np.arange(D)] -= 1.0
    return G != 0


# =============================================================================================
# CPU
# =============================================================================================
@pytest.mark.parametrize("env_id", ALL_IDS)
def test_complex_step_oracle_matches_central_differences(env_id):
    spec = Spec(env_id)
    rng = np.random.default_rng(1)
    y, a = sample_rows(spec, 64, rng, swing_omega=6.0)
    lo, hi = spec.ctrl
    if spec.continuous:
        a = rng.uniform(0.8 * lo, 0.8 * hi, size=64)  # away from the clamp's kinks
    if spec.fam == "ip":
        y[:, 1] = rng.uniform(-2.5, 2.5, 64)  # away from the wrap
    if spec.fam == "i2p":
        y[:, 1:3] = rng.uniform(0.3, 1.7, (64, 2)) - np.pi  # (th + pi) mod 2 away from 0 and 2
    for fr in (1, 3):
        J, JO, RG = cs_jacobian(spec, y, a, fr, f32_force=False)
        d = 1e-6
        for c in range(spec.D + 1):
            yp, ym, ap, am = y.copy(), y.copy(), a.copy(), a.copy()
            if c < spec.D:
                yp[:, c] += d
                ym[:, c] -= d
            else:
                ap += d
                am -= d
            (np_, op, rp), (nm, om, rm) = model_step(spec, yp, ap, fr, False), model_step(spec, ym, am, fr, False)
            for got, fd in ((J[:, :, c], (np_ - nm).real / (2 * d)), (JO[:, :, c], (op - om).real / (2 * d)),
                            (RG[:, c], (rp - rm).real / (2 * d))):
                np.testing.assert_allclose(got, fd, rtol=2e-6, atol=2e-6)
        if spec.fam == "i2p":  # the observation's angle rows carry the slope pi of the current_obs quirk
            np.testing.assert_allclose(JO[:, 1:3], np.pi * J[:, 1:3], rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize("env_id", IP_IDS + I2P_IDS)
@pytest.mark.parametrize("fr", [1, 2, 3, 4])
def test_jacobian_support_is_the_reference_transition_graph(env_id, fr):
    """support(J - I) of the step == get_transition_graph(freq_rate), per sample (inverted_pendulum.py:39-41,
    inverted_double_pendulum.py:42-52, core.py:142-161)."""
    spec = Spec(env_id)
    rng = np.random.default_rng(2 + fr)
    y, _ = sample_rows(spec, 256, rng)
    a = rng.uniform(0.9 * spec.ctrl[0], 0.9 * spec.ctrl[1], size=256)  # inside the clamp: the action acts
    J, _, _ = cs_jacobian(spec, y, a, fr)
    graph = E.make(env_id, freq_rate=fr).get_transition_graph(fr).astype(bool)
    assert (graph_support(J) == graph[None]).all()


def test_derivative_entry_points_validate_arguments_without_a_gpu():
    lib = _lib.lib
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 1, 0.02, _lib.IP_BOUNDARY_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q = _lib.I2PParams()
    q.freq_rate, q.dt, q.variant, q.action_kind = 1, 0.02, _lib.I2P_BOUNDARY_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q.mass_cart = q.mass_pole0 = q.mass_pole1 = q.length0 = q.length1 = 1.0
    for prm, jac_fns, vjp_fns, bad_variant in (
        (p, (lib.emei_cartpole_step_jacobian_f32, lib.emei_cartpole_step_jacobian_f64),
         (lib.emei_cartpole_step_vjp_f32, lib.emei_cartpole_step_vjp_f64), _lib.I2P_REBOUND_BALANCING),
        (q, (lib.emei_i2p_step_jacobian_f32, lib.emei_i2p_step_jacobian_f64),
         (lib.emei_i2p_step_vjp_f32, lib.emei_i2p_step_vjp_f64), _lib.IP_BOUNDARY_SWINGUP),
    ):
        ref = ctypes.byref(prm)
        for f in jac_fns:
            assert f(None, None, None, None, -1, ref, None) == -4
            assert f(None, None, None, None, 0, ref, None) == 0  # empty batch: no-op
            assert f(None, None, None, None, 8, None, None) == -1
            assert f(None, None, None, None, 8, ref, None) == -1  # null state
        for f in vjp_fns:
            assert f(*[None] * 7, -1, ref, None) == -4
            assert f(*[None] * 7, 0, ref, None) == 0
            assert f(*[None] * 7, 8, None, None) == -1
            assert f(*[None] * 7, 8, ref, None) == -1
        v = prm.variant
        prm.variant = bad_variant  # the other family's variant
        assert jac_fns[0](None, None, None, None, 8, ref, None) == -2
        assert vjp_fns[1](*[None] * 7, 8, ref, None) == -2
        prm.variant = 99
        assert jac_fns[1](None, None, None, None, 8, ref, None) == -2
        prm.variant = v
        prm.freq_rate = 0
        assert jac_fns[0](None, None, None, None, 8, ref, None) == -6
        prm.freq_rate = 1
        prm.action_kind = 9
        assert jac_fns[0](None, None, None, None, 8, ref, None) == -3
        prm.action_kind = _lib.ACTION_DISCRETE_U8  # a discrete action has no gradient: g_action must be NULL
        g = (ctypes.c_double * 8)()
        for f in vjp_fns:
            assert f(None, None, None, None, None, None, ctypes.addressof(g), 8, ref, None) == -3
            assert f(None, None, None, None, None, None, None, 8, ref, None) == -1  # without g_action: the null state
        prm.action_kind = _lib.ACTION_CONTINUOUS_F32
    buf = (ctypes.c_float * 64)()
    addr = ctypes.addressof(buf)
    mis = addr + 4 if addr % 16 == 0 else addr
    if mis % 16 != 0:  # cart-pole rows are 16-byte aligned, as for emei_cartpole_step_*
        assert lib.emei_cartpole_step_jacobian_f32(mis, addr, addr, None, 8, ctypes.byref(p), None) == -5
        assert lib.emei_cartpole_step_vjp_f32(addr, addr, None, None, None, mis, None, 8, ctypes.byref(p), None) == -5


def test_families_without_derivatives_say_why():
    for env_id, why in (("ChargedBallCentering-v0", "discontinuous"), ("ContinuousChargedBallCentering-v0", "discontinuous"),
                        ("HopperRunning-v0", "mj_step"), ("HalfCheetahRunning-v0", "mj_step")):
        env = E.make(env_id)
        for fn in (env.get_batch_transition, env.get_batch_jacobian):
            with pytest.raises(NotImplementedError, match=why):
                fn(np.zeros((2, env.observation_space.shape[0])), np.zeros(2))


# =============================================================================================
# GPU
# =============================================================================================
DEV = "cuda:0"
N_PAST_GRID = 148 * 2048 + 1  # one more env than a B200 can hold resident (148 SMs x 2048 threads): the grid-stride tail runs

# |kernel - complex step| / (1 + |complex step|) over the matrices below, measured on a B200: float64 at most 7.7e-14
# (I2P swing-up, fr 4; cart-pole and IP <= 2.7e-15), float32 at most 3.8e-5 (I2P swing-up, fr 4; cart-pole and IP <= 9.1e-7)
F64_TOL = 1e-12
F32_TOL = 2e-4


def _env(env_id, fr, dtype, n=1):
    return E.make(env_id, freq_rate=fr, num_envs=n, dtype=dtype, device=DEV)


def _action_tensor(spec, a, dtype):
    if spec.continuous:
        return torch.as_tensor(a, dtype=dtype, device=DEV)
    return torch.as_tensor(a.astype(np.uint8), device=DEV)


def _check_rows(spec, y, a, fr, jac, rg, tol):
    """compare kernel rows with the complex-step oracle; -> the largest scaled error"""
    J, _, RG = cs_jacobian(spec, y, a, fr)
    err = 0.0
    for got, ref in ((jac, J), (rg, RG)):
        e = np.abs(got - ref) / (1.0 + np.abs(ref))
        err = max(err, float(np.nanmax(e)))
        assert np.isfinite(got).all()
        assert (e <= tol).all(), f"{spec.id} fr={fr}: max scaled error {e.max():.3g} at {np.unravel_index(e.argmax(), e.shape)}"
    return err


def _subsample(n):
    return np.concatenate([np.arange(1024), np.arange(n - 1024, n)])  # the head and the grid-stride tail


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ALL_IDS)
@pytest.mark.parametrize("fr", [1, 2, 4])
def test_jacobian_f64_matches_complex_step(env_id, fr):
    spec = Spec(env_id)
    rng = np.random.default_rng(10 + fr)
    y, a = sample_rows(spec, N_PAST_GRID, rng)
    env = _env(env_id, fr, torch.float64)
    jac, rg = env.get_batch_jacobian(torch.as_tensor(y, device=DEV), _action_tensor(spec, a, torch.float64))
    idx = _subsample(N_PAST_GRID)
    err = _check_rows(spec, y[idx], a[idx], fr, jac.cpu().numpy()[idx], rg.cpu().numpy()[idx], F64_TOL)
    print(f"f64 {env_id} fr={fr}: max scaled error {err:.3g}")
    if not spec.continuous:
        assert (jac[:, :, -1] == 0).all() and (rg[:, -1] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ALL_IDS)
@pytest.mark.parametrize("fr", [1, 2, 4])
def test_jacobian_f32_matches_complex_step(env_id, fr):
    spec = Spec(env_id)
    rng = np.random.default_rng(20 + fr)
    y, a = sample_rows(spec, N_PAST_GRID, rng)
    y32, a32 = y.astype(np.float32), a.astype(np.float32)  # the oracle differentiates at the rounded inputs
    env = _env(env_id, fr, torch.float32)
    jac, rg = env.get_batch_jacobian(torch.as_tensor(y32, device=DEV), _action_tensor(spec, a32, torch.float32))
    idx = _subsample(N_PAST_GRID)
    err = _check_rows(spec, y32[idx].astype(np.float64), a32[idx].astype(np.float64), fr, jac.cpu().numpy()[idx].astype(np.float64),
                      rg.cpu().numpy()[idx].astype(np.float64), F32_TOL)
    print(f"f32 {env_id} fr={fr}: max scaled error {err:.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ALL_IDS)
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_vjp_is_g_transpose_j_for_every_cotangent_subset(env_id, dtype):
    spec = Spec(env_id)
    rng = np.random.default_rng(3)
    n, D = 4097, spec.D
    y, a = sample_rows(spec, n, rng)
    env = _env(env_id, 2, dtype)
    eng, s, act, _ = autodiff._inputs(env, torch.as_tensor(y, dtype=dtype, device=DEV), _action_tensor(spec, a, dtype))
    jac, rg = eng.jacobian(s, act)
    J, RG = jac.double(), rg.double()
    slope = torch.ones(D, dtype=torch.float64, device=DEV)
    if spec.fam == "i2p":
        slope[1:3] = math.pi
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    for use in itertools.product([False, True], repeat=3):
        gs = torch.randn(n, D, dtype=dtype, device=DEV) if use[0] else None
        go = torch.randn(n, D, dtype=dtype, device=DEV) if use[1] else None
        gr = torch.randn(n, dtype=dtype, device=DEV) if use[2] else None
        g_in, g_act = eng.vjp(s, act, gs, go, gr, spec.continuous)
        w = torch.zeros(n, D, dtype=torch.float64, device=DEV)
        want = torch.zeros(n, D + 1, dtype=torch.float64, device=DEV)
        if gs is not None:
            w += gs.double()
        if go is not None:
            w += slope * go.double()
        want += torch.einsum("nr,nrc->nc", w, J)
        if gr is not None:
            want += gr.double()[:, None] * RG
        scale = 1.0 + torch.einsum("nr,nrc->nc", w.abs(), J.abs()) + (gr.double().abs()[:, None] * RG.abs() if gr is not None else 0)
        assert ((g_in.double() - want[:, :D]).abs() <= tol * scale[:, :D]).all(), f"{env_id} {use}"
        if spec.continuous:
            assert ((g_act.double() - want[:, D]).abs() <= tol * scale[:, D]).all(), f"{env_id} {use}"
        else:
            assert g_act is None


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", IP_IDS + I2P_IDS)
def test_gradcheck_get_batch_transition_f64(env_id):
    spec = Spec(env_id)
    rng = np.random.default_rng(4)
    y, _ = sample_rows(spec, 6, rng, swing_omega=5.0)
    if spec.fam == "ip":
        y[:, 1] = rng.uniform(-2.5, 2.5, 6)  # away from the wrap
    else:
        y[:, 1:3] = rng.uniform(0.3, 1.7, (6, 2)) - np.pi  # (th + pi) mod 2 away from its jumps
    a = rng.uniform(0.8 * spec.ctrl[0], 0.8 * spec.ctrl[1], size=(6, 1))  # [B,1]: the gradient keeps the shape
    env = _env(env_id, 3, torch.float64)
    st = torch.tensor(y, dtype=torch.float64, device=DEV, requires_grad=True)
    at = torch.tensor(a, dtype=torch.float64, device=DEV, requires_grad=True)
    assert torch.autograd.gradcheck(lambda s, u: env.get_batch_transition(s, u)[:3], (st, at), eps=1e-6, atol=1e-6, rtol=1e-5)
    _, obs, rew, done = env.get_batch_transition(st, at.float())  # a float32 action: its gradient comes back in float32
    assert done.dtype == torch.bool and not done.requires_grad


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", IP_IDS + I2P_IDS)
@pytest.mark.parametrize("fr", [1, 2, 3, 4])
def test_kernel_jacobian_support_is_the_reference_transition_graph(env_id, fr):
    spec = Spec(env_id)
    rng = np.random.default_rng(5 + fr)
    y, _ = sample_rows(spec, 4096, rng)
    a = rng.uniform(0.9 * spec.ctrl[0], 0.9 * spec.ctrl[1], size=4096)
    env = _env(env_id, fr, torch.float64)
    jac, _ = env.get_batch_jacobian(torch.as_tensor(y, device=DEV), torch.as_tensor(a, device=DEV))
    graph = env.get_transition_graph(fr).astype(bool)
    assert (graph_support(jac.cpu().numpy()) == graph[None]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["ContinuousCartPoleSwingUp-v0"] + IP_IDS[2:] + I2P_IDS[2:])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_action_gradient_at_the_control_clamp(env_id, dtype):
    """zero outside [ctrl_low, ctrl_high], passed through on its boundary and inside (torch.clamp's rule); the
    cart-pole force has no clamp"""
    spec = Spec(env_id)
    lo, hi = spec.ctrl
    a_np = np.array([hi + 0.5, hi, 0.5 * hi, lo, lo - 0.5, 3 * hi, 3 * lo], dtype=np.float64)
    rng = np.random.default_rng(6)
    y, _ = sample_rows(spec, a_np.size, rng, swing_omega=3.0)
    env = _env(env_id, 2, dtype)
    st = torch.tensor(y, dtype=dtype, device=DEV)
    at = torch.tensor(a_np, dtype=dtype, device=DEV, requires_grad=True)
    jac, rg = env.get_batch_jacobian(st, at.detach())
    nxt, obs, rew, _ = env.get_batch_transition(st, at)
    (nxt.sum() + rew.sum()).backward()
    outside = np.array([True, False, False, False, True, True, True]) if spec.fam != "cp" else np.zeros(7, bool)
    col = jac[:, :, -1].cpu().numpy()
    assert (col[outside] == 0).all() and (rg[:, -1].cpu().numpy()[outside] == 0).all()
    assert (np.abs(col[~outside]).sum(axis=1) > 0).all()
    assert (at.grad.cpu().numpy()[outside] == 0).all() and (at.grad.cpu().numpy()[~outside] != 0).all()
    J, _, RG = cs_jacobian(spec, st.double().cpu().numpy(), at.detach().double().cpu().numpy(), 2)
    tol = F64_TOL if dtype == torch.float64 else F32_TOL
    assert np.allclose(col, J[:, :, -1], rtol=tol, atol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["CartPoleBalancing-v0", "CartPoleSwingUp-v0"])
def test_discrete_cartpole_state_gradient(env_id):
    spec = Spec(env_id)
    rng = np.random.default_rng(7)
    y, a = sample_rows(spec, 33, rng)
    env = _env(env_id, 2, torch.float64)
    st = torch.tensor(y, device=DEV, requires_grad=True)
    act = torch.as_tensor(a.astype(np.int64), device=DEV)  # no gradient for a discrete action
    nxt, obs, rew, _ = env.get_batch_transition(st, act)
    (nxt[:, 2].sum() + obs[:, 0].sum() + rew.sum()).backward()
    jac, rg = env.get_batch_jacobian(st.detach(), act)
    want = jac[:, 2, :4] + jac[:, 0, :4] + rg[:, :4]
    assert torch.allclose(st.grad, want, rtol=1e-12, atol=1e-12)
    assert (jac[:, :, 4] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["ContinuousCartPoleSwingUp-v0", "BoundaryInvertedPendulumSwingUp-v0", "ReboundInvertedDoublePendulumSwingUp-v0"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("n", [37, 9001])
def test_transition_is_stateless_and_bit_equal_to_the_step(env_id, dtype, n):
    """the env's state, stats and frozen snapshot do not move; the outputs equal get_batch_next_obs and step() from the
    same rows, bit for bit (9001 envs: the float32 cart-pole step takes its TMA kernel)"""
    spec = Spec(env_id)
    env = _env(env_id, 2, dtype, n=n)
    env.reset(seed=3)
    env.step(torch.zeros(n, device=DEV))
    env.freeze()
    before = env.state.clone()
    snap = [t.clone() for t in env.frozen_state]
    stats = env.stats.clone()
    rng = np.random.default_rng(8)
    y, a = sample_rows(spec, n, rng, swing_omega=5.0)
    rows = torch.as_tensor(y, dtype=dtype, device=DEV)
    act = torch.as_tensor(a, dtype=torch.float32, device=DEV)
    nxt, obs, rew, done = env.get_batch_transition(rows, act)
    jac, rg = env.get_batch_jacobian(rows, act)
    torch.cuda.synchronize()
    assert torch.equal(env.state, before) and torch.equal(env.stats, stats)
    assert all(torch.equal(x, s) for x, s in zip(env.frozen_state, snap))
    ref_obs = env.get_batch_next_obs(rows, action=act) if spec.fam != "i2p" else env.get_batch_next_obs(rows, action=act, state=rows)
    assert torch.equal(obs, ref_obs)
    other = _env(env_id, 2, dtype, n=n)
    other.state = rows
    o2, r2, d2, _, _ = other.step(act)
    assert torch.equal(nxt, other.state) and torch.equal(obs, o2) and torch.equal(rew, r2) and torch.equal(done, d2)
    assert jac.shape == (n, spec.D, spec.D + 1) and rg.shape == (n, spec.D + 1)


def _rollout_sum_model(spec, y0, acts, fr):
    """complex: sum of 50 rewards of the chained step"""
    y, total = y0, 0
    for t in range(acts.shape[0]):
        y, _, r = model_step(spec, y, acts[t], fr)
        total = total + r
    return total


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["ReboundInvertedPendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"])
def test_fifty_step_bptt_matches_complex_step(env_id):
    """d(sum of 50 rewards) / d(state_0, actions) through 50 chained get_batch_transition calls (the supported
    backpropagation-through-time path) against the complex-step derivative of the same 50-step sum"""
    spec = Spec(env_id)
    T, B, fr = 50, 8, 2
    rng = np.random.default_rng(9)
    y0 = rng.uniform(-1, 1, size=(B, spec.D)) * 0.3
    acts = rng.uniform(0.5 * spec.ctrl[0], 0.5 * spec.ctrl[1], size=(T, B))
    env = _env(env_id, fr, torch.float64)
    st = torch.tensor(y0, device=DEV, requires_grad=True)
    at = torch.tensor(acts, device=DEV, requires_grad=True)
    s, total = st, 0
    for t in range(T):
        s, _, r, _ = env.get_batch_transition(s, at[t])
        total = total + r.sum()
    total.backward()
    g_state = np.zeros((B, spec.D))
    for c in range(spec.D):
        yc = y0.astype(np.complex128)
        yc[:, c] += 1j * H_CS
        g_state[:, c] = _rollout_sum_model(spec, yc, acts.astype(np.complex128), fr).imag / H_CS
    g_act = np.zeros((T, B))
    for t in range(T):
        ac = acts.astype(np.complex128)
        ac[t] += 1j * H_CS
        g_act[t] = _rollout_sum_model(spec, y0.astype(np.complex128), ac, fr).imag / H_CS
    np.testing.assert_allclose(st.grad.cpu().numpy(), g_state, rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(at.grad.cpu().numpy(), g_act, rtol=1e-8, atol=1e-10)
