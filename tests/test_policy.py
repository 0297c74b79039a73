"""Policy search over the true dynamics: emei_*_policy_eval_* / emei_policy_perturb / emei_policy_update and
env.get_batch_policy_returns / env.policy_search.

The closed-loop returns are checked bit for bit against teacher-forced rollout() calls of the eval's actions, the actions against
a numpy float64 restatement of the linear policy on that rollout's recorded observations, the directions against the numpy
mirror of their Philox stream below, the update against a float64 restatement of ARS V1-t.
"""
import ctypes

import numpy as np
import pytest
import torch

import emei_b200 as E
from emei_b200 import _lib
from oracle.philox import philox4x32_10, u01

PURPOSE_POLICY_PERTURB = 8
PURPOSE_PLAN_ACTION = 7

CARTPOLE_IDS = ["CartPoleBalancing-v0", "CartPoleSwingUp-v0", "ContinuousCartPoleBalancing-v0", "ContinuousCartPoleSwingUp-v0"]
IP_IDS = ["ReboundInvertedPendulumBalancing-v0", "BoundaryInvertedPendulumBalancing-v0", "ReboundInvertedPendulumSwingUp-v0",
          "BoundaryInvertedPendulumSwingUp-v0"]
I2P_IDS = ["ReboundInvertedDoublePendulumBalancing-v0", "BoundaryInvertedDoublePendulumBalancing-v0",
           "ReboundInvertedDoublePendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"]
CB_IDS = ["ChargedBallCentering-v0", "ContinuousChargedBallCentering-v0"]
ALL_IDS = CARTPOLE_IDS + IP_IDS + I2P_IDS + CB_IDS


# =============================================================================================
# host mirrors
# =============================================================================================
def policy_directions(seed, N, P, purpose=PURPOSE_POLICY_PERTURB):
    """[N, P] directions delta_k: Philox (seed, k, block j, purpose 8); block j gives delta_{2j} = rad cos, delta_{2j+1} = rad sin."""
    k = np.arange(N, dtype=np.uint64)
    out = np.empty((N, 2 * ((P + 1) // 2)))
    for j in range((P + 1) // 2):
        w = philox4x32_10(seed, k, np.full(N, j), purpose)
        rad = np.sqrt(-2.0 * np.log(1.0 - u01(w[0], w[1])))
        u2 = u01(w[2], w[3])
        out[:, 2 * j], out[:, 2 * j + 1] = rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)
    return out[:, :P]


def perturb(theta, seed, N, noise):
    """[2N, P]: rows 2k / 2k + 1 = theta +- noise delta_k"""
    d = policy_directions(seed, N, len(theta))
    out = np.empty((2 * N, len(theta)))
    out[0::2], out[1::2] = theta + noise * d, theta - noise * d
    return out


def policy_actions(params, obs, discrete, low=-1.0, high=1.0, dtype=np.float64):
    """the policy of params [C, P] on observations [..., C, E, D] (any float dtype) in the kernel's operation order:
    u = c; u = u + w_j obs_j (numpy float64 rounds every operation); continuous: clip(dtype(u)), discrete: u > 0."""
    params = np.asarray(params, dtype=np.float64)
    o = np.asarray(obs).astype(np.float64)
    D = o.shape[-1]
    u = np.broadcast_to(params[:, None, D], o.shape[:-1]).copy()
    for j in range(D):
        u = u + params[:, None, j] * o[..., j]
    if discrete:
        return (u > 0).astype(np.float64)
    return np.clip(u.astype(dtype), dtype(low), dtype(high)).astype(np.float64)


def ars_update(returns, theta, seed, top, step_size):
    """float64 restatement of the update -> (theta, stats, chosen directions in rank order)"""
    r = np.asarray(returns, dtype=np.float64)
    N2, E_ = r.shape
    N = N2 // 2
    m = np.cumsum(r, axis=1)[:, -1] / E_  # ascending over e
    rp, rm = m[0::2], m[1::2]
    fin = np.isfinite(m)
    elig = np.isfinite(rp) & np.isfinite(rm)
    mx = np.where(elig, np.maximum(rp, rm), -np.inf)
    order = [k for k in np.lexsort((np.arange(N), -mx)) if elig[k]]
    chosen = np.array(order[:top], dtype=np.int64)
    b = len(chosen)
    nan = float("nan")
    mean_fin = m[fin].mean() if fin.any() else nan
    if b == 0:
        return np.array(theta, dtype=np.float64), np.array([0, nan, nan, mean_fin]), chosen
    both = torch.as_tensor(np.concatenate([rp[chosen], rm[chosen]]))
    sigma = float(both.std(unbiased=False))
    th = torch.as_tensor(np.array(theta, dtype=np.float64))
    if sigma > 0 and np.isfinite(sigma):
        d = torch.as_tensor(policy_directions(seed, N, len(theta))[chosen])
        th = th + step_size / (b * sigma) * ((torch.as_tensor(rp[chosen] - rm[chosen]))[:, None] * d).sum(0)
    return th.numpy(), np.array([b, sigma, mx[chosen[0]], mean_fin]), chosen


# =============================================================================================
# CPU
# =============================================================================================
def test_policy_params_layout():
    assert ctypes.sizeof(_lib.PolicyParams) == 4 * 8 + 2 * 4 + 2 * 4
    offs = {f: getattr(_lib.PolicyParams, f).offset for f, _ in _lib.PolicyParams._fields_}
    assert offs == dict(seed=0, gamma=8, noise=16, step_size=24, action_low=32, action_high=36, action_kind=40, top=44)


def _q(**kw):
    q = _lib.PolicyParams()
    q.seed, q.gamma, q.noise, q.step_size, q.action_low, q.action_high = 1, 1.0, 0.1, 0.02, -1.0, 1.0
    q.action_kind, q.top = _lib.ACTION_CONTINUOUS_F32, 2
    for k, v in kw.items():
        setattr(q, k, v)
    return q


def _family_params():
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 1, 0.02, _lib.CARTPOLE_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q = _lib.I2PParams()
    q.freq_rate, q.dt, q.variant, q.action_kind = 1, 0.02, _lib.I2P_BOUNDARY_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q.mass_cart = q.mass_pole0 = q.mass_pole1 = q.length0 = q.length1 = 1.0
    c = _lib.ChargedBallParams()
    c.gravity_acc, c.mass_ball, c.radius, c.charge, c.time_step, c.freq_rate, c.action_kind = 9.8, 1.0, 1.0, 10.0, 0.02, 1, 3
    return {"emei_cartpole_policy_eval": p, "emei_i2p_policy_eval": q, "emei_charged_ball_policy_eval": c}


def _validation_cases():
    """(entry, family params, policy params, pointers, sizes, expected code, what).  Every row is rejected, or is a no-op,
    before any launch, so the table runs without a device."""
    buf = (ctypes.c_double * 256)()
    al = (ctypes.addressof(buf) + 15) & ~15  # valid, 16-byte aligned host memory (never dereferenced)
    mis = al + 4
    cases = []
    for base, prm in _family_params().items():
        for entry in (base + "_f32", base + "_f64"):
            nst = 3 if "charged_ball" in entry else 1
            full = [al] * (nst + 2) + [None]  # state pointers, params, returns, actions_out
            none = [None] * len(full)
            rows = [
                (prm, _q(), none, (-1, 4, 8), -4, "negative C"),
                (prm, _q(), none, (4, -1, 8), -4, "negative E"),
                (prm, _q(), none, (4, 4, -1), -4, "negative H"),
                (prm, _q(), none, (2 ** 31 + 1, 4, 8), -4, "C > 2^31"),
                (prm, _q(), none, (4, 2 ** 31 + 1, 8), -4, "E > 2^31"),
                (prm, _q(), none, (4, 4, 2 ** 31), -4, "H = 2^31"),
                (prm, None, none, (4, 4, 8), -1, "null policy params"),
                (None, _q(), none, (4, 4, 8), -1, "null family params"),
                (prm, _q(action_kind=9), none, (4, 4, 8), -3, "unknown action kind"),
                (prm, _q(gamma=1.5), none, (4, 4, 8), -6, "gamma > 1"),
                (prm, _q(gamma=float("nan")), none, (4, 4, 8), -6, "gamma NaN"),
                (prm, _q(action_low=1.0, action_high=-1.0), none, (4, 4, 8), -6, "empty action box"),
                (prm, _q(), none, (0, 4, 8), 0, "C = 0: no-op"),
                (prm, _q(), none, (4, 0, 8), 0, "E = 0: no-op"),
                (prm, _q(), none, (4, 4, 0), 0, "H = 0: no-op"),
                (prm, _q(), none, (4, 4, 8), -1, "every pointer null"),
            ]
            bad = type(prm)()
            ctypes.memmove(ctypes.byref(bad), ctypes.byref(prm), ctypes.sizeof(bad))
            bad.freq_rate = 0
            rows.append((bad, _q(), full, (4, 4, 8), -6, "family params: freq_rate 0"))
            for j, what in [(i, f"null state pointer {i}") for i in range(nst)] + [(nst, "null params"), (nst + 1, "null returns")]:
                args = list(full)
                args[j] = None
                rows.append((prm, _q(), args, (4, 4, 8), -1, what))
            if "i2p" in entry:
                rows.append((prm, _q(action_kind=_lib.ACTION_DISCRETE_U8), full, (4, 4, 8), -3, "discrete kind on the double pendulum"))
            else:
                rows.append((prm, _q(action_kind=_lib.ACTION_DISCRETE_U8, action_low=1.0, action_high=-1.0), none, (4, 4, 0), 0,
                             "discrete kind ignores the box"))
            for j in ((1, 2) if nst == 3 else (0,)):
                args = list(full)
                args[j] = mis
                rows.append((prm, _q(), args, (4, 4, 8), -5, f"misaligned state pointer {j}"))
            cases += [(entry,) + r for r in rows]
    # perturb: theta, params ; (N, P)
    for r in [
        (_q(), [None, None], (0, 5), -4, "N = 0"), (_q(), [None, None], (4097, 5), -4, "N = 4097"),
        (_q(), [None, None], (4, 0), -4, "P = 0"), (_q(), [None, None], (4, 9), -4, "P = 9"),
        (None, [al, al], (4, 5), -1, "null policy params"),
        (_q(noise=-0.1), [al, al], (4, 5), -6, "negative noise"), (_q(noise=float("inf")), [al, al], (4, 5), -6, "infinite noise"),
        (_q(noise=float("nan")), [al, al], (4, 5), -6, "NaN noise"),
        (_q(), [None, al], (4, 5), -1, "null theta"), (_q(), [al, None], (4, 5), -1, "null params"),
    ]:
        cases.append(("emei_policy_perturb", None) + r)
    # update: returns, theta, stats ; (N, E, P)
    for r in [
        (_q(), [None] * 3, (0, 4, 5), -4, "N = 0"), (_q(), [None] * 3, (4097, 4, 5), -4, "N = 4097"),
        (_q(), [None] * 3, (4, 0, 5), -4, "E = 0"), (_q(), [None] * 3, (4, 2 ** 31 + 1, 5), -4, "E > 2^31"),
        (_q(), [None] * 3, (4, 4, 0), -4, "P = 0"), (_q(), [None] * 3, (4, 4, 9), -4, "P = 9"),
        (None, [al, al, None], (4, 4, 5), -1, "null policy params"),
        (_q(top=0), [al, al, None], (4, 4, 5), -6, "top = 0"), (_q(top=5), [al, al, None], (4, 4, 5), -6, "top > N"),
        (_q(step_size=float("nan")), [al, al, None], (4, 4, 5), -6, "NaN step size"),
        (_q(step_size=float("-inf")), [al, al, None], (4, 4, 5), -6, "infinite step size"),
        (_q(), [None, al, None], (4, 4, 5), -1, "null returns"), (_q(), [al, None, None], (4, 4, 5), -1, "null theta"),
    ]:
        cases.append(("emei_policy_update", None) + r)
    return cases


@pytest.mark.parametrize("case", _validation_cases(), ids=lambda c: f"{c[0]}-{c[6]}")
def test_policy_validation(case):
    entry, prm, q, ptrs, sizes, code, what = case
    fn = getattr(_lib.lib, entry)
    qa = ctypes.byref(q) if q is not None else None
    if entry.startswith("emei_policy_"):
        got = fn(*ptrs, *sizes, qa, None)
    else:
        got = fn(*ptrs, *sizes, qa, ctypes.byref(prm) if prm is not None else None, None)
    assert got == code, f"{entry}: {what}: got {got}, expected {code}"


def test_policy_direction_mirror():
    theta = np.array([0.5, -1.0, 2.0, 0.25, -3.0, 1.5, 0.0])
    p = perturb(theta, 17, 300, 0.1)
    # antithetic pairing is exact: rows 2k and 2k + 1 step by the same nu delta_k in opposite directions
    d = policy_directions(17, 300, 7)
    assert np.array_equal(p[0::2], theta + 0.1 * d) and np.array_equal(p[1::2], theta - 0.1 * d)
    # a direction's first coordinates do not depend on P
    assert np.array_equal(policy_directions(17, 300, 5), d[:, :5])
    # N(0, 1) moments
    z = policy_directions(3, 40000, 8).reshape(-1)
    assert abs(z.mean()) < 5 / np.sqrt(z.size) and abs(z.std() - 1) < 0.01
    assert abs(np.mean(z ** 3)) < 0.05 and abs(np.mean(z ** 4) - 3) < 0.1
    # purpose 8 is its own stream: the planner's purpose-7 words for the same key differ everywhere
    assert not np.any(policy_directions(3, 1000, 8) == policy_directions(3, 1000, 8, purpose=PURPOSE_PLAN_ACTION))
    # another seed, another stream
    assert not np.any(policy_directions(4, 1000, 8) == policy_directions(3, 1000, 8))


def test_policy_restatement_branches():
    """the restatement's own cases: fewer eligible directions than top, sigma = 0 and no eligible direction"""
    r = np.array([[1.0, 3.0], [0.0, 0.0], [np.nan, 1.0], [2.0, 2.0], [5.0, 5.0], [-np.inf, 0.0]])
    th, st, ch = ars_update(r, np.zeros(5), 1, 3, 0.1)
    assert list(ch) == [0] and st[0] == 1 and st[2] == 2.0
    th, st, ch = ars_update(np.ones((4, 3)), np.ones(5), 1, 2, 0.1)
    assert st[1] == 0 and np.array_equal(th, np.ones(5))
    th, st, ch = ars_update(np.full((4, 3), np.nan), np.ones(5), 1, 2, 0.1)
    assert st[0] == 0 and np.isnan(st[3])


def test_policy_raises_without_dynamics_kernel():
    for eid in ("HopperRunning-v0", "HalfCheetahRunning-v0"):
        env = E.make(eid)
        with pytest.raises(NotImplementedError):
            env.policy_search(10)
        with pytest.raises(NotImplementedError):
            env.get_batch_policy_returns(np.zeros((1, 13)), np.zeros((1, 12)), 5)


# =============================================================================================
# GPU
# =============================================================================================
def _starts(eid, n, dtype, fr, seed=0, perturb=True):
    """n start states of task ``eid``: the reset states, perturbed (balancing tasks then terminate inside the horizon)."""
    env = E.make(eid, freq_rate=fr, num_envs=n, dtype=dtype, device="cuda:0")
    env.reset(seed=seed)
    st = env.state
    if isinstance(st, dict):
        return {k: v.clone() for k, v in st.items()}
    st = st.clone()
    if perturb:
        g = torch.Generator(device="cpu").manual_seed(seed + 1)
        st += (0.3 * torch.randn(st.shape, generator=g, dtype=torch.float64)).to(st)
    return st


def _tile(st, C):
    """the starts of C candidates, candidate-major: row c E + e is start e"""
    if isinstance(st, dict):
        return {k: v.repeat((C,) + (1,) * (v.dim() - 1)) for k, v in st.items()}
    return st.repeat(C, 1)


def _params(env, C, seed):
    P = env.observation_space.shape[0] + 1
    g = torch.Generator(device="cpu").manual_seed(seed)
    scale = 2.0 if len(env.action_space.shape) else 1.0
    return (scale * torch.randn((C, P), generator=g, dtype=torch.float64)).to("cuda:0")


def _masked_return(rewards, dones, gamma):
    """float64 host restatement in the kernel's operation order: ret = ret + disc r; disc = disc gamma; stop after a done."""
    r = rewards.double().cpu().numpy()
    d = dones.cpu().numpy().astype(bool)
    ret = np.zeros(r.shape[1])
    disc, alive = 1.0, np.ones(r.shape[1], dtype=bool)
    for t in range(r.shape[0]):
        ret = np.where(alive, ret + disc * r[t], ret)
        disc = disc * gamma
        alive &= ~d[t]
    return ret


def _box(env):
    if len(env.action_space.shape) == 0:
        return True, 0.0, 1.0
    return False, float(env.action_space.low[0]), float(env.action_space.high[0])


@pytest.mark.gpu
@pytest.mark.parametrize("H", [1, 17])
@pytest.mark.parametrize("CE", [(1, 300), (37, 29)])
@pytest.mark.parametrize("fr", [1, 4])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eid", ALL_IDS)
def test_policy_returns_equal_rollout(eid, dtype, fr, CE, H):
    C, En = CE
    env = E.make(eid, freq_rate=fr, num_envs=En, dtype=dtype, device="cuda:0")
    st = _starts(eid, En, dtype, fr, seed=C + H)
    params = _params(env, C, seed=H + fr)
    discrete, lo, hi = _box(env)
    twin = E.make(eid, freq_rate=fr, num_envs=C * En, dtype=dtype, device="cuda:0")
    terminated = 0
    for gamma in (1.0, 0.97):
        ret, act = env.get_batch_policy_returns(params, st, H, gamma=gamma, return_actions=True)
        assert ret.shape == (C, En) and ret.dtype == torch.float64 and act.shape == (H, C, En)
        twin.state = _tile(st, C)
        rec = twin.rollout(H, actions=act.view(H, C * En), record=True, auto_reset=False, max_episode_steps=0)
        ref = _masked_return(rec["rewards"], rec["dones"], gamma)
        assert np.array_equal(ret.cpu().numpy().reshape(-1), ref), f"{eid} {dtype} fr={fr} C={C} E={En} H={H} gamma={gamma}"
        obs = rec["observations"].double().cpu().numpy().reshape(H, C, En, -1)
        host = policy_actions(params.cpu().numpy(), obs, discrete, lo, hi, np.float32 if dtype == torch.float32 else np.float64)
        assert np.array_equal(act.double().cpu().numpy(), host), f"{eid} {dtype} fr={fr}: actions"
        terminated += int(rec["dones"][:-1].any(dim=0).sum())
    if "Balancing" in eid and H == 17 and C * En > 300:
        assert terminated > 0, "perturbed balancing starts should terminate inside the horizon"


def _engine(eid, dtype=torch.float64, n=1):
    env = E.make(eid, num_envs=n, dtype=dtype, device="cuda:0")
    eng, P, q = env._policy_setup()
    return env, eng, P, q


@pytest.mark.gpu
@pytest.mark.parametrize("NP", [(1, 5), (37, 5), (4096, 7), (300, 1), (64, 8)])
def test_policy_perturb_matches_mirror(NP):
    N, P = NP
    env, eng, _, q = _engine("ContinuousCartPoleSwingUp-v0")
    theta = torch.linspace(-2, 3, P, dtype=torch.float64, device="cuda:0")
    q.seed, q.noise = 0xDEADBEEF12345, 0.07
    got = eng.policy_perturb(theta, N, q).cpu().numpy()
    host = perturb(theta.cpu().numpy(), q.seed, N, 0.07)
    assert got.shape == (2 * N, P)
    assert np.all(np.abs(got - host) <= 1e-12 * np.maximum(1.0, np.abs(host)))
    # antithetic pairing is exact: theta - (params[2k] - theta) rounds to params[2k+1] up to one rounding of each side
    th = theta.cpu().numpy()
    assert np.allclose(got[0::2] - th, th - got[1::2], rtol=0, atol=4e-16 * max(1.0, np.abs(th).max()))
    q.noise = 0.0
    z = eng.policy_perturb(theta, N, q).cpu().numpy()
    assert np.array_equal(z, np.broadcast_to(th, z.shape))


def _update(eng, returns, theta, q):
    th = theta.clone()
    stats = torch.full((4,), -1.0, dtype=torch.float64, device="cuda:0")
    eng.policy_update(returns.contiguous(), th, q, stats)
    return th, stats


def _same_bits(x, y):
    return x.dtype == y.dtype and torch.equal(x.contiguous().view(torch.uint8), y.contiguous().view(torch.uint8))


def _check_update(returns, theta, q, tol=1e-12):
    env, eng, P, _ = _engine("ContinuousCartPoleSwingUp-v0")
    th1, st1 = _update(eng, returns, theta, q)
    th2, st2 = _update(eng, returns, theta, q)
    assert _same_bits(th1, th2) and _same_bits(st1, st2), "two calls differ"
    ref_th, ref_st, chosen = ars_update(returns.cpu().numpy(), theta.cpu().numpy(), q.seed, q.top, q.step_size)
    got, gst = th1.cpu().numpy(), st1.cpu().numpy()
    assert np.all(np.abs(got - ref_th) <= tol * np.maximum(np.abs(ref_th), 1e-300) + tol * np.abs(theta.cpu().numpy() - ref_th)), \
        (got, ref_th)
    assert gst[0] == ref_st[0]
    for j in (1, 2, 3):
        assert (np.isnan(gst[j]) and np.isnan(ref_st[j])) or abs(gst[j] - ref_st[j]) <= 1e-12 * max(1.0, abs(ref_st[j])), (j, gst, ref_st)
    return th1, st1, chosen


def _assert_top_set_identified(returns, chosen, top, seed, P):
    """the update pins the chosen set down: swapping the last chosen direction for the best unchosen eligible one moves the
    step direction by more than 100 x the tolerance (the margin test_plan.py uses for CEM elites)."""
    r = np.asarray(returns, dtype=np.float64)
    m = np.cumsum(r, axis=1)[:, -1] / r.shape[1]
    rp, rm = m[0::2], m[1::2]
    elig = np.isfinite(rp) & np.isfinite(rm)
    rest = [k for k in np.lexsort((np.arange(len(rp)), -np.where(elig, np.maximum(rp, rm), -np.inf))) if elig[k] and k not in chosen]
    if len(chosen) < top or not rest:
        return
    d = policy_directions(seed, len(rp), P)
    alt = chosen.copy()
    alt[-1] = rest[0]
    s = lambda ks: ((rp[ks] - rm[ks])[:, None] * d[ks]).sum(0)  # noqa: E731
    gap = np.abs(s(chosen) - s(alt)).max()
    assert gap > 100 * 1e-12 * np.abs(s(chosen)).max(), f"a one-direction swap moves the step by only {gap}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(8, 16, 5, 4), (37, 3, 7, 10), (300, 1, 5, 300), (4096, 2, 5, 64), (1000, 5, 7, 999)],
                         ids=lambda c: f"N{c[0]}-E{c[1]}-P{c[2]}-top{c[3]}")
def test_policy_update_matches_restatement(case):
    N, En, P, top = case
    g = torch.Generator(device="cpu").manual_seed(N + En)
    returns = (100 * torch.randn((2 * N, En), generator=g, dtype=torch.float64)).to("cuda:0")
    theta = torch.randn(P, generator=g, dtype=torch.float64).to("cuda:0")
    _, eng, _, q = _engine("ContinuousCartPoleSwingUp-v0")
    q.seed, q.top, q.step_size = 99 + N, top, 0.3
    _, _, chosen = _check_update(returns, theta, q)
    _assert_top_set_identified(returns.cpu().numpy(), chosen, top, q.seed, P)


@pytest.mark.gpu
def test_policy_update_ties():
    """directions whose max(r+, r-) tie exactly: the chosen set is the smaller k among the tied, checked as a set"""
    N, En, P, top = 300, 4, 5, 40
    g = torch.Generator(device="cpu").manual_seed(5)
    returns = torch.randint(0, 4, (2 * N, En), generator=g).to("cuda:0", torch.float64)
    theta = torch.zeros(P, dtype=torch.float64, device="cuda:0")
    _, eng, _, q = _engine("ContinuousCartPoleSwingUp-v0")
    q.seed, q.top, q.step_size = 7, top, 1.0
    _, _, chosen = _check_update(returns, theta, q)
    m = returns.cpu().numpy().mean(1)
    mx = np.maximum(m[0::2], m[1::2])
    assert len(set(mx[chosen])) < top  # ties inside the chosen set
    _assert_top_set_identified(returns.cpu().numpy(), chosen, top, q.seed, P)


@pytest.mark.gpu
def test_policy_update_nonfinite_and_degenerate():
    N, En, P = 300, 3, 7
    _, eng, _, q = _engine("ContinuousCartPoleSwingUp-v0")
    q.seed, q.step_size = 11, 0.5
    g = torch.Generator(device="cpu").manual_seed(9)
    theta = torch.randn(P, generator=g, dtype=torch.float64).to("cuda:0")
    base = (10 * torch.randn((2 * N, En), generator=g, dtype=torch.float64)).to("cuda:0")
    u = torch.rand((2 * N, En), generator=g).to("cuda:0")
    mixed = base.clone()
    mixed[u < 0.05] = float("nan")
    mixed[(u >= 0.05) & (u < 0.08)] = float("inf")
    mixed[(u >= 0.08) & (u < 0.11)] = float("-inf")
    q.top = 100
    th, st, chosen = _check_update(mixed, theta, q)
    assert 0 < st[0].item() <= 100
    # fewer eligible directions than top
    few = torch.full_like(base, float("nan"))
    few[:20] = base[:20]
    q.top = 50
    th, st, chosen = _check_update(few, theta, q)
    assert st[0].item() == 10 and len(chosen) == 10
    # no eligible direction: theta unchanged, bit for bit
    q.top = 5
    for what in ("nan", "inf", "-inf"):
        th, st, _ = _check_update(torch.full_like(base, float(what)), theta, q)
        assert _same_bits(th, theta) and st[0].item() == 0 and torch.isnan(st[1:3]).all()
    # sigma_R = 0: every chosen return equal, theta unchanged bit for bit
    th, st, _ = _check_update(torch.full_like(base, 3.0), theta, q)
    assert _same_bits(th, theta) and st[1].item() == 0.0 and st[0].item() == 5


@pytest.mark.gpu
def test_policy_invariants():
    eid, H, C = "ContinuousCartPoleBalancing-v0", 23, 19
    env = E.make(eid, num_envs=40, dtype=torch.float32, device="cuda:0")
    env.reset(seed=4)
    env.step(torch.zeros(40, device="cuda:0"))
    env.freeze()
    state0, stats0 = env.state.clone(), env.stats.clone()
    snap0 = [t.clone() for t in env.frozen_state]
    bufs0 = [t.clone() for t in env._engine._bufs]
    params = _params(env, C, seed=1)
    st = _starts(eid, 40, torch.float32, 1)
    r1, a1 = env.get_batch_policy_returns(params, st, H, return_actions=True)
    r2, a2 = env.get_batch_policy_returns(params, st, H, return_actions=True)
    assert torch.equal(r1, r2) and torch.equal(a1, a2)
    assert torch.equal(env.get_batch_policy_returns(params, st, H), r1)
    s1 = env.policy_search(H, iterations=3, directions=16, top=4, episodes=5, seed=6)
    s2 = env.policy_search(H, iterations=3, directions=16, top=4, episodes=5, seed=6)
    for x, y in zip(s1, s2):
        assert torch.equal(x, y)
    assert s1.theta.shape == (5,) and s1.returns.shape == (32, 5) and s1.stats.shape == (3, 4)
    # statelessness
    assert torch.equal(env.state, state0) and torch.equal(env.stats, stats0)
    assert all(torch.equal(x, y) for x, y in zip(env.frozen_state, snap0))
    assert all(torch.equal(x, y) for x, y in zip(env._engine._bufs, bufs0))
    # numpy in, numpy out; a single policy [P]
    rn = env.get_batch_policy_returns(params.cpu().numpy(), st.cpu().numpy(), H)
    assert isinstance(rn, np.ndarray) and np.array_equal(rn, r1.cpu().numpy())
    assert torch.equal(env.get_batch_policy_returns(params[3], st, H), r1[3:4])
    sn = env.policy_search(H, iterations=3, directions=16, top=4, episodes=5, seed=6, theta=np.zeros(5))
    assert isinstance(sn.theta, np.ndarray) and np.array_equal(sn.theta, s1.theta.cpu().numpy())
    # horizon None = max_episode_steps; starts=None draws num_envs starts keyed by seed
    rd = env.get_batch_policy_returns(params, seed=3)
    assert rd.shape == (C, 40) and torch.equal(rd, env.get_batch_policy_returns(params, seed=3, horizon=env.max_episode_steps))
    # unseeded calls draw fresh keys without moving the initial-state stream of a later unseeded reset()
    twin = E.make(eid, num_envs=40, dtype=torch.float32, device="cuda:0")
    env.reset(seed=8)
    twin.reset(seed=8)
    q1 = env.policy_search(200, iterations=1, directions=4, episodes=3, noise=1.0)
    q2 = env.policy_search(200, iterations=1, directions=4, episodes=3, noise=1.0)
    assert not torch.equal(q1.returns, q2.returns)
    u1, u2 = env.get_batch_policy_returns(params, horizon=200), env.get_batch_policy_returns(params, horizon=200)
    assert not torch.equal(u1, u2)
    assert torch.equal(env.reset()[0], twin.reset()[0])
    # the unseeded counter restarts with reset(seed=)
    env.reset(seed=8)
    assert torch.equal(env.policy_search(200, iterations=1, directions=4, episodes=3, noise=1.0).returns, q1.returns)


@pytest.mark.gpu
@pytest.mark.parametrize("eid", ["ChargedBallCentering-v0", "ReboundInvertedDoublePendulumBalancing-v0"])
def test_policy_search_start_states(eid):
    """the starts of an iteration are the initial-state distribution's, keyed by policy_starts_seed: a reset env with the same
    key has them as its state"""
    env = E.make(eid, num_envs=6, dtype=torch.float64, device="cuda:0")
    key = E.policy_starts_seed(E.plan_iteration_seed(21, 0))
    st = env._policy_starts(6, key)
    P = env.observation_space.shape[0] + 1
    params = _params(env, 3, seed=2)
    r = env.get_batch_policy_returns(params, st, 9)
    assert torch.equal(r, env.get_batch_policy_returns(params, env._policy_starts(6, key), 9))
    res = env.policy_search(9, iterations=1, directions=2, top=2, episodes=6, seed=21, theta=np.zeros(P))
    th = torch.zeros(P, dtype=torch.float64, device="cuda:0")
    eng, _, q = env._policy_setup()
    q.seed, q.noise = E.plan_iteration_seed(21, 0), 0.03
    assert np.array_equal(res.returns, env.get_batch_policy_returns(eng.policy_perturb(th, 2, q), st, 9).cpu().numpy())


@pytest.mark.gpu
def test_policy_past_resident_grid():
    eid, H = "ContinuousCartPoleSwingUp-v0", 5
    C, En = 75, 4042  # 303150 pairs > 148 SMs x 2048 threads
    env = E.make(eid, num_envs=En, dtype=torch.float32, device="cuda:0")
    st = _starts(eid, En, torch.float32, 1)
    params = _params(env, C, seed=4)
    ret, act = env.get_batch_policy_returns(params, st, H, return_actions=True)
    twin = E.make(eid, num_envs=C * En, dtype=torch.float32, device="cuda:0")
    twin.state = _tile(st, C)
    rec = twin.rollout(H, actions=act.view(H, C * En), record=True, auto_reset=False, max_episode_steps=0)
    assert np.array_equal(ret.cpu().numpy().reshape(-1), _masked_return(rec["rewards"], rec["dones"], 1.0))


@pytest.mark.gpu
def test_policy_actions_past_2_31_elements():
    eid, C, En, H = "CartPoleSwingUp-v0", 4096, 1024, 513  # H C E = 2.15e9 uint8 actions
    assert H * C * En > 2 ** 31
    env = E.make(eid, num_envs=En, dtype=torch.float32, device="cuda:0")
    st = _starts(eid, En, torch.float32, 1)
    params = _params(env, C, seed=5)
    ret, act = env.get_batch_policy_returns(params, st, H, return_actions=True)
    assert torch.equal(ret, env.get_batch_policy_returns(params, st, H))
    # the last candidates' actions, beyond element 2^31: a teacher-forced rollout of them observes what the policy acted on
    c0 = C - 3
    twin = E.make(eid, num_envs=3 * En, dtype=torch.float32, device="cuda:0")
    twin.state = _tile(st, 3)
    tail = act[:, c0:].reshape(H, 3 * En).contiguous()
    rec = twin.rollout(H, actions=tail, record=True, auto_reset=False, max_episode_steps=0)
    obs = rec["observations"].double().cpu().numpy().reshape(H, 3, En, -1)
    assert np.array_equal(tail.double().cpu().numpy().reshape(H, 3, En), policy_actions(params[c0:].cpu().numpy(), obs, True))
    assert np.array_equal(ret[c0:].cpu().numpy().reshape(-1), _masked_return(rec["rewards"], rec["dones"], 1.0))


# pinned hyperparameters of the efficacy test: (iterations, directions, top, step_size, noise, episodes)
EFFICACY = {
    "CartPoleBalancing-v0": (80, 32, 16, 0.05, 0.1, 8),
    "ContinuousCartPoleBalancing-v0": (80, 32, 16, 0.05, 0.1, 8),
    "BoundaryInvertedPendulumBalancing-v0": (80, 32, 16, 0.05, 0.1, 8),
}


@pytest.mark.gpu
@pytest.mark.parametrize("eid", list(EFFICACY))
def test_policy_search_balances(eid):
    iters, N, top, alpha, nu, episodes = EFFICACY[eid]
    env = E.make(eid, num_envs=256, dtype=torch.float32, device="cuda:0")
    env.reset(seed=0)
    res = env.policy_search(iterations=iters, directions=N, top=top, step_size=alpha, noise=nu, episodes=episodes, seed=1)
    assert torch.isfinite(res.theta).all()
    T = env.max_episode_steps
    found = env.get_batch_policy_returns(res.theta, seed=12345)[0].cpu().numpy()
    zero = env.get_batch_policy_returns(torch.zeros_like(res.theta), seed=12345)[0].cpu().numpy()
    survived = (found >= T).mean()  # reward 1 per step: the return is the episode length
    assert survived >= 0.95, (survived, res.theta, res.stats[-5:])
    assert found.mean() > zero.mean()
