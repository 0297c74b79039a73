"""Differentiable open-loop trajectories: emei_*_trajectory_* / emei_*_trajectory_vjp_* and env.get_batch_trajectory.

The forward is checked bit for bit against T chained get_batch_transition calls, the reverse sweep against the chained
autograd path and against the complex-step derivative of test_autodiff's model (imported, not copied).
"""
import ctypes
import itertools

import numpy as np
import pytest
import torch

import emei_b200 as E
from emei_b200 import _lib
from test_autodiff import H_CS, Spec, model_step, sample_rows

CARTPOLE_IDS = ["CartPoleBalancing-v0", "CartPoleSwingUp-v0", "ContinuousCartPoleBalancing-v0", "ContinuousCartPoleSwingUp-v0"]
IP_IDS = ["ReboundInvertedPendulumBalancing-v0", "BoundaryInvertedPendulumBalancing-v0", "ReboundInvertedPendulumSwingUp-v0",
          "BoundaryInvertedPendulumSwingUp-v0"]
I2P_IDS = ["ReboundInvertedDoublePendulumBalancing-v0", "BoundaryInvertedDoublePendulumBalancing-v0",
           "ReboundInvertedDoublePendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"]
ALL_IDS = CARTPOLE_IDS + IP_IDS + I2P_IDS


# =============================================================================================
# CPU
# =============================================================================================
def _validation_cases():
    """(entry base, is_vjp, params, pointer args, n, horizon, expected code, what): every row is rejected (or is a no-op)
    before any launch, so the table runs without a device."""
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 1, 0.02, _lib.IP_BOUNDARY_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q = _lib.I2PParams()
    q.freq_rate, q.dt, q.variant, q.action_kind = 1, 0.02, _lib.I2P_BOUNDARY_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q.mass_cart = q.mass_pole0 = q.mass_pole1 = q.length0 = q.length1 = 1.0
    buf = (ctypes.c_double * 256)()
    al = (ctypes.addressof(buf) + 15) & ~15  # 16-byte aligned, valid host memory (never dereferenced: no launch happens)
    mis = al + 4
    cases = []
    for base, prm, other_variant in (("emei_cartpole_trajectory", p, _lib.I2P_REBOUND_BALANCING),
                                     ("emei_i2p_trajectory", q, _lib.IP_BOUNDARY_SWINGUP)):
        for vjp in (False, True):
            entry = base + ("_vjp" if vjp else "")
            npt = 7 if vjp else 6
            required = (0, 1, 5) if vjp else (0, 1, 2, 4)  # states, actions, g_state0 / state0, actions, states, rewards
            full = [al] * npt
            if vjp:
                full[6] = None  # g_actions
            none = [None] * npt

            def with_params(**kw):
                c = type(prm)()
                ctypes.memmove(ctypes.byref(c), ctypes.byref(prm), ctypes.sizeof(c))
                for k, v in kw.items():
                    setattr(c, k, v)
                return c

            cases += [
                (entry, prm, none, -1, 4, -4, "negative n"),
                (entry, prm, none, 8, -1, -4, "negative horizon"),
                (entry, None, none, -1, 4, -4, "negative n before the params check"),
                (entry, prm, none, 0, 4, 0, "empty batch: no-op"),
                (entry, prm, none, 8, 0, 0, "zero horizon: no-op"),
                (entry, None, none, 8, 4, -1, "null params"),
                (entry, prm, none, 8, 4, -1, "every pointer null"),
                (entry, with_params(variant=other_variant), none, 8, 4, -2, "the other family's variant"),
                (entry, with_params(variant=99), none, 8, 4, -2, "unknown variant"),
                (entry, with_params(freq_rate=0), none, 8, 4, -6, "freq_rate 0"),
                (entry, with_params(action_kind=9), none, 8, 4, -3, "bad action kind"),
            ]
            for j in required:
                args = list(full)
                args[j] = None
                cases.append((entry, prm, args, 8, 4, -1, f"null required pointer {j}"))
            if vjp:
                disc = with_params(action_kind=_lib.ACTION_DISCRETE_U8)
                cases.append((entry, disc, [None] * 6 + [al], 8, 4, -3, "discrete kind with g_actions"))
                cases.append((entry, disc, [None] * 7, 8, 4, -1, "discrete kind without g_actions: the null states"))
            if base == "emei_cartpole_trajectory":  # cart-pole rows are 16-byte aligned, as for emei_cartpole_step_*
                rows = (0, 2, 3, 5) if vjp else (0, 2, 3)  # states, g_states, g_obs, g_state0 / state0, states, obs
                for j in rows:
                    args = list(full)
                    args[j] = mis
                    cases.append((entry, prm, args, 8, 4, -5, f"misaligned row array {j}"))
    return cases, buf


def test_trajectory_entry_points_validate_arguments_without_a_gpu():
    cases, _buf = _validation_cases()
    for entry, prm, ptrs, n, horizon, want, what in cases:
        for sfx in ("_f32", "_f64"):
            f = getattr(_lib.lib, entry + sfx)
            got = f(*ptrs, n, horizon, ctypes.byref(prm) if prm is not None else None, None)
            assert got == want, f"{entry}{sfx} {what}: got {got}, want {want}"


def test_families_without_derivatives_have_no_trajectory():
    for env_id, why in (("ChargedBallCentering-v0", "discontinuous"), ("ContinuousChargedBallCentering-v0", "discontinuous"),
                        ("HopperRunning-v0", "mj_step"), ("HalfCheetahRunning-v0", "mj_step")):
        env = E.make(env_id)
        with pytest.raises(NotImplementedError, match=why):
            env.get_batch_trajectory(np.zeros((2, env.observation_space.shape[0])), np.zeros((3, 2)))


# =============================================================================================
# GPU
# =============================================================================================
DEV = "cuda:0"
T_STEPS = 12
N_PAST_GRID = 148 * 2048 + 1  # one more env than a B200 can hold resident: the grid-stride tail runs


def _env(env_id, fr, dtype, n=1):
    return E.make(env_id, freq_rate=fr, num_envs=n, dtype=dtype, device=DEV)


def _problem(spec, n, T, dtype, seed, swing_omega=5.0):
    """rows [n, D] and actions [T, n] (on both sides of and exactly on the clamp; discrete: uint8)"""
    rng = np.random.default_rng(seed)
    y, _ = sample_rows(spec, n, rng, swing_omega=swing_omega)
    acts = np.stack([sample_rows(spec, n, rng)[1] for _ in range(T)]) if T else np.zeros((0, n))
    st = torch.as_tensor(y, dtype=dtype, device=DEV)
    at = torch.as_tensor(acts, dtype=dtype, device=DEV) if spec.continuous else torch.as_tensor(acts.astype(np.uint8), device=DEV)
    return st, at


def _bits(t):
    return t.contiguous().view({8: torch.int64, 4: torch.int32, 1: torch.uint8}[t.element_size()])


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _chained(env, st, at):
    """T chained get_batch_transition calls -> stacked (states [T+1], obs [T], rewards [T], dones [T])"""
    s, S, O, R, Dn = st, [st], [], [], []
    for t in range(at.shape[0]):
        s, o, r, d = env.get_batch_transition(s, at[t])
        S.append(s), O.append(o), R.append(r[:, 0]), Dn.append(d[:, 0])
    return torch.stack(S), torch.stack(O), torch.stack(R), torch.stack(Dn)


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ALL_IDS)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("fr", [1, 2, 4])
@pytest.mark.parametrize("n", [37, 9001])
def test_forward_is_bit_equal_to_chained_transitions(env_id, dtype, fr, n):
    """9001 envs: the chained float32 cart-pole steps take the TMA kernel, 37 the small-batch kernel"""
    spec = Spec(env_id)
    env = _env(env_id, fr, dtype)
    st, at = _problem(spec, n, T_STEPS, dtype, seed=fr * 100 + n % 97)
    with torch.no_grad():
        got = env.get_batch_trajectory(st, at)
        want = _chained(env, st, at)
    assert got[3].dtype == torch.bool and got[2].shape == (T_STEPS, n) and got[0].shape == (T_STEPS + 1, n, spec.D)
    for name, g, w in zip(("states", "obs", "rewards", "dones"), got, want):
        assert _same_bits(g, w), f"{env_id} {dtype} fr={fr} n={n}: {name} differs"


@pytest.mark.gpu
@pytest.mark.parametrize("env_id, dtype", [("ContinuousCartPoleSwingUp-v0", torch.float32), ("BoundaryInvertedPendulumSwingUp-v0", torch.float64),
                                           ("BoundaryInvertedDoublePendulumSwingUp-v0", torch.float64),
                                           ("ReboundInvertedDoublePendulumSwingUp-v0", torch.float32)])
def test_forward_past_one_resident_grid(env_id, dtype):
    spec = Spec(env_id)
    env = _env(env_id, 4, dtype)
    st, at = _problem(spec, N_PAST_GRID, 3, dtype, seed=11)
    with torch.no_grad():
        got = env.get_batch_trajectory(st, at)
        want = _chained(env, st, at)
    assert all(_same_bits(g, w) for g, w in zip(got, want))


def _weights(spec, n, T, dtype, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(T + 1, n, spec.D, dtype=dtype, device=DEV, generator=gen), torch.randn(T, n, spec.D, dtype=dtype, device=DEV, generator=gen),
            torch.randn(T, n, dtype=dtype, device=DEV, generator=gen))


def _grads(fn, env, st, at, w, rewards_only=False):
    """d loss / d (state, actions) of loss = <w_s, states> + <w_o, obs> + <w_r, rewards> through fn"""
    s = st.clone().requires_grad_(True)
    a = at.clone().requires_grad_(at.is_floating_point())
    states, obs, rewards, _ = fn(env, s, a)
    loss = (rewards * w[2]).sum()
    if not rewards_only:
        loss = loss + (states * w[0]).sum() + (obs * w[1]).sum()
    loss.backward()
    return s.grad, a.grad


def _fused(env, s, a):
    return env.get_batch_trajectory(s, a)


# |fused - chained| / (1 + |chained|) over the matrix below, measured on a B200: float64 at most 2.4e-14, float32 at most 9.6e-6
# (cart-pole: obs = states[1:] reassociates one cotangent sum; IP and I2P are bit-equal in both precisions)
BWD_TOL = {torch.float64: 1e-12, torch.float32: 1e-5}


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ALL_IDS)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("fr", [1, 2, 4])
@pytest.mark.parametrize("n", [37, 9001])
def test_backward_matches_the_chained_autograd_path(env_id, dtype, fr, n):
    spec = Spec(env_id)
    env = _env(env_id, fr, dtype)
    st, at = _problem(spec, n, T_STEPS, dtype, seed=fr * 10 + n % 89)
    w = _weights(spec, n, T_STEPS, dtype, seed=fr + n)
    gs_f, ga_f = _grads(_fused, env, st, at, w)
    gs_c, ga_c = _grads(_chained, env, st, at, w)
    tol = BWD_TOL[dtype]
    errs = []
    for got, ref in ((gs_f, gs_c), (ga_f, ga_c)):
        if ref is None:
            assert got is None and not spec.continuous  # a discrete action has no gradient
            continue
        assert got.dtype == ref.dtype == dtype and got.shape == ref.shape
        e = (got.double() - ref.double()).abs() / (1 + ref.double().abs())
        errs.append(float(e.max()))
        assert torch.isfinite(ref).all() and errs[-1] <= tol, f"{env_id} {dtype} fr={fr} n={n}: max scaled error {errs[-1]:.3g}"
    print(f"{dtype} {env_id} fr={fr} n={n}: max scaled error (state, action) {', '.join(f'{x:.3g}' for x in errs)}")
    if dtype == torch.float64:  # rewards only: the same device functions, compiled with -fmad=false, in the same term order
        gs_f, ga_f = _grads(_fused, env, st, at, w, rewards_only=True)
        gs_c, ga_c = _grads(_chained, env, st, at, w, rewards_only=True)
        assert torch.equal(gs_f, gs_c) and (ga_c is None or torch.equal(ga_f, ga_c)), f"{env_id} fr={fr} n={n}: rewards-only not bit-equal"


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["ReboundInvertedPendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"])
def test_fifty_step_trajectory_gradient_matches_complex_step(env_id):
    """d(sum of 50 rewards) / d(state_0, actions) through one get_batch_trajectory against the complex-step derivative of
    the same sum (one task per kernel family: emei_cartpole_trajectory_* / emei_i2p_trajectory_*)"""
    spec = Spec(env_id)
    T, B, fr = 50, 8, 2
    rng = np.random.default_rng(9)
    y0 = rng.uniform(-1, 1, size=(B, spec.D)) * 0.3
    acts = rng.uniform(0.5 * spec.ctrl[0], 0.5 * spec.ctrl[1], size=(T, B))
    env = _env(env_id, fr, torch.float64)
    st = torch.tensor(y0, device=DEV, requires_grad=True)
    at = torch.tensor(acts, device=DEV, requires_grad=True)
    env.get_batch_trajectory(st, at)[2].sum().backward()

    def total(y, a):
        out = 0
        for t in range(T):
            y, _, r = model_step(spec, y, a[t], fr)
            out = out + r
        return out

    g_state = np.zeros((B, spec.D))
    for c in range(spec.D):
        yc = y0.astype(np.complex128)
        yc[:, c] += 1j * H_CS
        g_state[:, c] = total(yc, acts.astype(np.complex128)).imag / H_CS
    g_act = np.zeros((T, B))
    for t in range(T):
        ac = acts.astype(np.complex128)
        ac[t] += 1j * H_CS
        g_act[t] = total(y0.astype(np.complex128), ac).imag / H_CS
    np.testing.assert_allclose(st.grad.cpu().numpy(), g_state, rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(at.grad.cpu().numpy(), g_act, rtol=1e-8, atol=1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", IP_IDS + I2P_IDS)
def test_gradcheck_get_batch_trajectory_f64(env_id):
    spec = Spec(env_id)
    T, B = 3, 4
    rng = np.random.default_rng(4)
    y, _ = sample_rows(spec, B, rng, swing_omega=2.0)
    if spec.fam == "ip":
        y[:, 1] = rng.uniform(-1.5, 1.5, B)  # away from the wrap
        y[:, 3] = rng.uniform(-2.0, 2.0, B)
    else:
        y[:, 1:3] = rng.uniform(0.5, 1.5, (B, 2)) - np.pi  # (th + pi) mod 2 away from its jumps
        y[:, 4:6] = rng.uniform(-0.5, 0.5, (B, 2))
    a = rng.uniform(0.8 * spec.ctrl[0], 0.8 * spec.ctrl[1], size=(T, B, 1))  # [T,B,1]: the gradient keeps the shape
    env = _env(env_id, 2, torch.float64)
    st = torch.tensor(y, dtype=torch.float64, device=DEV, requires_grad=True)
    at = torch.tensor(a, dtype=torch.float64, device=DEV, requires_grad=True)
    assert torch.autograd.gradcheck(lambda s, u: env.get_batch_trajectory(s, u)[:3], (st, at), eps=1e-6, atol=1e-6, rtol=1e-5)
    a32 = at.detach().float().requires_grad_(True)  # a float32 action leaf on the float64 env: its gradient comes back in float32
    states, obs, rew, done = env.get_batch_trajectory(st, a32)
    rew.sum().backward()
    assert done.dtype == torch.bool and not done.requires_grad
    assert a32.grad.dtype == torch.float32 and a32.grad.shape == (T, B, 1) and torch.isfinite(a32.grad).all()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["CartPoleBalancing-v0", "CartPoleSwingUp-v0"])
def test_discrete_cartpole_state_gradient(env_id):
    spec = Spec(env_id)
    env = _env(env_id, 2, torch.float64)
    st, at = _problem(spec, 33, 7, torch.float64, seed=7)
    at = at.long()  # int64 actions: no gradient
    w = _weights(spec, 33, 7, torch.float64, seed=5)
    gs_f, ga_f = _grads(_fused, env, st, at, w)
    gs_c, _ = _grads(_chained, env, st, at, w)
    assert ga_f is None
    assert torch.allclose(gs_f, gs_c, rtol=1e-12, atol=1e-12)
    eng = env._ensure_engine()
    states = env.get_batch_trajectory(st, at)[0]
    g0, g_act = eng.trajectory_vjp(states, at.contiguous(), None, None, w[2].contiguous(), False)
    assert g_act is None and torch.isfinite(g0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["ContinuousCartPoleSwingUp-v0", "BoundaryInvertedPendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_null_cotangents_equal_zero_cotangents(env_id, dtype):
    spec = Spec(env_id)
    n, T = 513, 9
    env = _env(env_id, 2, dtype)
    st, at = _problem(spec, n, T, dtype, seed=12)
    eng = env._ensure_engine()
    states, _, _, _ = eng.trajectory(st, at)
    w = _weights(spec, n, T, dtype, seed=13)
    for use in itertools.product([False, True], repeat=3):
        args = [x if u else None for x, u in zip(w, use)]
        zeros = [x if u else torch.zeros_like(x) for x, u in zip(w, use)]
        g0, ga = eng.trajectory_vjp(states, at, *args, True)
        z0, za = eng.trajectory_vjp(states, at, *zeros, True)
        assert torch.equal(g0, z0) and torch.equal(ga, za), f"{env_id} {use}"
    # the forward's nullable outputs: without obs and dones it writes the same states and rewards
    s2, r2 = torch.empty_like(states), torch.empty(T, n, dtype=dtype, device=DEV)
    env._call(eng._trajectory_entry, st.data_ptr(), at.data_ptr(), s2.data_ptr(), None, r2.data_ptr(), None, n, T,
              ctypes.byref(eng.params), env._stream())
    ref = eng.trajectory(st, at)
    assert _same_bits(s2, ref[0]) and _same_bits(r2, ref[2])


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", ["ContinuousCartPoleSwingUp-v0", "ReboundInvertedPendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_trajectory_is_stateless(env_id, dtype):
    """the env's state, stats and frozen snapshot do not move; horizon 0 returns state[None] and empty outputs; numpy in,
    numpy out"""
    spec = Spec(env_id)
    n = 64
    env = _env(env_id, 2, dtype, n=n)
    env.reset(seed=3)
    env.step(torch.zeros(n, device=DEV))
    env.freeze()
    before, stats = env.state.clone(), env.stats.clone()
    snap = [t.clone() for t in env.frozen_state]
    st, at = _problem(spec, n, 5, dtype, seed=14)
    states, obs, rew, done = env.get_batch_trajectory(st, at)
    torch.cuda.synchronize()
    assert torch.equal(env.state, before) and torch.equal(env.stats, stats)
    assert all(torch.equal(x, s) for x, s in zip(env.frozen_state, snap))
    s = st.clone().requires_grad_(True)
    states0, obs0, rew0, done0 = env.get_batch_trajectory(s, at[:0])
    assert states0.shape == (1, n, spec.D) and torch.equal(states0[0], st)
    assert obs0.shape == (0, n, spec.D) and rew0.shape == (0, n) and done0.shape == (0, n) and done0.dtype == torch.bool
    states0.sum().backward()
    assert torch.equal(s.grad, torch.ones_like(st))
    np_out = env.get_batch_trajectory(st.cpu().numpy(), at.cpu().numpy())
    assert all(isinstance(x, np.ndarray) for x in np_out)
    assert np.array_equal(np_out[0], states.cpu().numpy()) and np.array_equal(np_out[2], rew.cpu().numpy())
    with pytest.raises(ValueError):
        env.get_batch_trajectory(st, at.T.contiguous())  # [B, T] is not [T, B]
