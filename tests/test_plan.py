"""Sampling-based planning: emei_*_plan_eval_* / emei_plan_update_* and env.get_batch_plan_returns / env.plan.

The returns are checked bit for bit against teacher-forced rollout() calls of the candidates' actions, the actions against the
numpy mirror of the candidate stream below, the update against a float64 restatement of CEM / MPPI.
"""
import ctypes

import numpy as np
import pytest
import torch

import emei_b200 as E
from emei_b200 import _lib
from oracle.philox import philox4x32_10, u01

PURPOSE_PLAN_ACTION = 7

CARTPOLE_IDS = ["CartPoleBalancing-v0", "CartPoleSwingUp-v0", "ContinuousCartPoleBalancing-v0", "ContinuousCartPoleSwingUp-v0"]
IP_IDS = ["ReboundInvertedPendulumBalancing-v0", "BoundaryInvertedPendulumBalancing-v0", "ReboundInvertedPendulumSwingUp-v0",
          "BoundaryInvertedPendulumSwingUp-v0"]
I2P_IDS = ["ReboundInvertedDoublePendulumBalancing-v0", "BoundaryInvertedDoublePendulumBalancing-v0",
           "ReboundInvertedDoublePendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"]
CB_IDS = ["ChargedBallCentering-v0", "ContinuousChargedBallCentering-v0"]
ALL_IDS = CARTPOLE_IDS + IP_IDS + I2P_IDS + CB_IDS


# =============================================================================================
# host mirror of the candidate stream (plan.cuh)
# =============================================================================================
def plan_actions(seed, mean, std, K, low=-1.0, high=1.0, discrete=False, dtype=np.float64, env_offset=0, rows=None, cols=None):
    """[H, len(rows), len(cols)] actions of candidates (b, k), b in ``rows`` (default all B), k in ``cols`` (default 0..K-1):
    Philox (seed, (env_offset + b) 2^32 + k, purpose 7); continuous: Box-Muller pair of block t >> 1 (cos half for even t),
    a = clamp(dtype(mean + std z)); discrete: word t & 3 of block t >> 2, a = float32((w >> 8) 2^-24) < float32(p)."""
    mean = np.asarray(mean, dtype=np.float64)
    H, B = mean.shape
    rows = np.arange(B) if rows is None else np.asarray(rows)
    cols = np.arange(K) if cols is None else np.asarray(cols)
    env = ((rows.astype(np.uint64)[:, None] + np.uint64(env_offset)) << np.uint64(32)) | cols.astype(np.uint64)[None, :]
    env = env.reshape(-1)
    out = np.empty((H, env.size), dtype=np.float64)
    for t in range(H):
        m = np.repeat(mean[t, rows], cols.size)
        if discrete:
            w = philox4x32_10(seed, env, np.full(env.size, t >> 2), PURPOSE_PLAN_ACTION)[t & 3]
            u = (w >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)
            out[t] = (u < m.astype(np.float32)).astype(np.float64)
        else:
            w = philox4x32_10(seed, env, np.full(env.size, t >> 1), PURPOSE_PLAN_ACTION)
            rad = np.sqrt(-2.0 * np.log(1.0 - u01(w[0], w[1])))
            u2 = u01(w[2], w[3])
            z = rad * (np.cos(2 * np.pi * u2) if t % 2 == 0 else np.sin(2 * np.pi * u2))
            s = np.repeat(np.asarray(std, dtype=np.float64)[t, rows], cols.size)
            a = (m + s * z).astype(dtype)
            out[t] = np.clip(a, dtype(low), dtype(high))
    return out.reshape(H, rows.size, cols.size)


def cem_order(returns):
    """[B, K] candidate indices in the update's total order: return descending, ties to the smaller k, NaN after every number."""
    r = np.asarray(returns, dtype=np.float64)
    B, K = r.shape
    nan = np.isnan(r)
    return np.lexsort((np.broadcast_to(np.arange(K), (B, K)), np.where(nan, np.inf, -r), nan), axis=-1)


def refit(actions, returns, mean, std, method, elites=1, temperature=1.0, momentum=0.0, min_std=0.0, discrete=False):
    """float64 restatement of the update from the candidates' actions [H, B, K] and returns [B, K] -> (mean, std, CEM order or
    None).  MPPI: a weight that is not a number counts 0, and all-zero weights are uniform."""
    a = torch.as_tensor(np.asarray(actions, dtype=np.float64))
    r = torch.as_tensor(np.asarray(returns, dtype=np.float64))
    H, B, K = a.shape
    if method == "cem":
        order = cem_order(returns)
        w = torch.zeros(B, K, dtype=torch.float64)
        w.scatter_(1, torch.as_tensor(order[:, :elites]), 1.0 / elites)
    else:
        order = None
        rmax = torch.nan_to_num(r, nan=float("-inf")).max(dim=1, keepdim=True).values
        w = torch.nan_to_num(torch.exp((r - rmax) / temperature), nan=0.0)
        tot = w.sum(dim=1, keepdim=True)
        w = torch.where(tot > 0, w / tot, torch.full_like(w, 1.0 / K))
    fit_mean = (w[None] * a).sum(-1)
    fit_std = torch.sqrt((w[None] * (a - fit_mean[..., None]) ** 2).sum(-1))
    m = torch.as_tensor(np.asarray(mean, dtype=np.float64))
    new_mean = momentum * m + (1 - momentum) * fit_mean
    new_std = None
    if discrete:
        new_mean = new_mean.clamp(0, 1)
    else:
        s = torch.as_tensor(np.asarray(std, dtype=np.float64))
        new_std = torch.clamp(momentum * s + (1 - momentum) * fit_std, min=min_std)
    return new_mean.numpy(), (new_std.numpy() if new_std is not None else None), order


def assert_elite_set_identified(actions, order, elites, tol):
    """A fit that matches the restatement within ``tol`` pins the elite set down: swapping the last elite for the best
    non-elite moves the fitted mean by more than 100 tol at some step, for every start."""
    a = np.asarray(actions, dtype=np.float64)
    H, B, K = a.shape
    if elites >= K:
        return
    for b in range(B):
        el = order[b, :elites]
        alt = el.copy()
        alt[-1] = order[b, elites]
        gap = np.abs(a[:, b, el].mean(-1) - a[:, b, alt].mean(-1)).max()
        assert gap > 100 * tol, f"start {b}: a one-elite swap moves the mean by only {gap}"


# =============================================================================================
# CPU
# =============================================================================================
def test_plan_params_layout():
    assert ctypes.sizeof(_lib.PlanParams) == 2 * 8 + 4 * 8 + 2 * 4 + 3 * 4 + 4  # natural alignment, padded to 8
    offs = {f: getattr(_lib.PlanParams, f).offset for f, _ in _lib.PlanParams._fields_}
    assert offs == dict(seed=0, env_offset=8, gamma=16, temperature=24, momentum=32, min_std=40, action_low=48, action_high=52,
                        method=56, elites=60, action_kind=64)


def _plan(**kw):
    q = _lib.PlanParams()
    q.seed, q.gamma, q.temperature, q.momentum, q.min_std = 1, 1.0, 1.0, 0.0, 0.0
    q.action_low, q.action_high, q.method, q.elites, q.action_kind = -1.0, 1.0, _lib.PLAN_CEM, 4, _lib.ACTION_CONTINUOUS_F32
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
    return {"emei_cartpole_plan_eval": p, "emei_i2p_plan_eval": q, "emei_charged_ball_plan_eval": c}


def _validation_cases():
    """(entry, family params or None for the update, plan params, pointers, B, K, H, expected code, what).  Every row is
    rejected, or is a no-op, before any launch, so the table runs without a device."""
    buf = (ctypes.c_double * 256)()
    al = (ctypes.addressof(buf) + 15) & ~15  # valid, 16-byte aligned host memory (never dereferenced)
    mis = al + 4
    fam = _family_params()
    cases = []
    entries = [(base + sfx, fam[base]) for base in fam for sfx in ("_f32", "_f64")]
    entries += [("emei_plan_update_f32", None), ("emei_plan_update_f64", None)]
    for entry, prm in entries:
        update = prm is None
        cb = "charged_ball" in entry
        nst = 0 if update else (3 if cb else 1)
        # eval: state pointers, mean, std, returns, actions_out ; update: returns, mean_io, std_io, best_actions, best_return
        full = [al] * (nst + 4) if not update else [al, al, al, None, None]
        if not update:
            full[-1] = None
        none = [None] * len(full)
        rows = [
            (prm, _plan(), none, -1, 8, 4, -4, "negative B"),
            (prm, _plan(), none, 8, 8, -1, -4, "negative H"),
            (prm, _plan(), none, 8, 0, 4, -4, "K = 0"),
            (prm, _plan(), none, 8, 4097, 4, -4, "K = 4097"),
            (prm, None, none, 8, 8, 4, -1, "null plan params"),
            (prm, _plan(action_kind=9), none, 8, 8, 4, -3, "unknown action kind"),
            (prm, _plan(method=2), none, 8, 8, 4, -6, "unknown method"),
            (prm, _plan(elites=0), none, 8, 8, 4, -6, "CEM with E = 0"),
            (prm, _plan(elites=9), none, 8, 8, 4, -6, "CEM with E > K"),
            (prm, _plan(method=_lib.PLAN_MPPI, temperature=0.0), none, 8, 8, 4, -6, "MPPI at temperature 0"),
            (prm, _plan(gamma=1.5), none, 8, 8, 4, -6, "gamma > 1"),
            (prm, _plan(gamma=-0.1), none, 8, 8, 4, -6, "gamma < 0"),
            (prm, _plan(momentum=1.0), none, 8, 8, 4, -6, "momentum 1"),
            (prm, _plan(min_std=-1.0), none, 8, 8, 4, -6, "negative min_std"),
            (prm, _plan(action_low=1.0, action_high=-1.0), none, 8, 8, 4, -6, "empty action box"),
            (prm, _plan(), none, 0, 8, 4, 0, "B = 0: no-op"),
            (prm, _plan(), none, 8, 8, 0, 0, "H = 0: no-op"),
            (prm, _plan(), none, 8, 8, 4, -1, "every pointer null"),
        ]
        if update:
            rows += [
                (prm, _plan(), [None, al, al, None, None], 8, 8, 4, -1, "null returns"),
                (prm, _plan(), [al, None, al, None, None], 8, 8, 4, -1, "null mean"),
                (prm, _plan(), [al, al, None, None, None], 8, 8, 4, -1, "continuous kind without std"),
            ]
        else:
            rows.append((None, _plan(), none, 8, 8, 4, -1, "null family params"))
            bad = type(prm)()
            ctypes.memmove(ctypes.byref(bad), ctypes.byref(prm), ctypes.sizeof(bad))
            bad.freq_rate = 0
            rows.append((bad, _plan(), full, 8, 8, 4, -6, "family params: freq_rate 0"))
            for j, what in [(i, f"null state pointer {i}") for i in range(nst)] + [(nst, "null mean"), (nst + 1, "null std"),
                                                                                  (nst + 2, "null returns")]:
                args = list(full)
                args[j] = None
                rows.append((prm, _plan(), args, 8, 8, 4, -1, what))
            args = list(full)
            args[nst + 1] = None
            if "i2p" in entry:
                rows.append((prm, _plan(action_kind=_lib.ACTION_DISCRETE_U8), args, 8, 8, 4, -3, "discrete kind on the double pendulum"))
            for j in ((1, 2) if cb else (0,)):
                args = list(full)
                args[j] = mis
                rows.append((prm, _plan(), args, 8, 8, 4, -5, f"misaligned state pointer {j}"))
        cases += [(entry,) + r for r in rows]
    return cases


@pytest.mark.parametrize("case", _validation_cases(), ids=lambda c: f"{c[0]}-{c[8]}")
def test_plan_validation(case):
    entry, prm, q, ptrs, B, K, H, code, what = case
    fn = getattr(_lib.lib, entry)
    qa = ctypes.byref(q) if q is not None else None
    if prm is None and entry.startswith("emei_plan_update"):
        got = fn(*ptrs, B, K, H, qa, None)
    else:
        pa = ctypes.byref(prm) if prm is not None else None
        got = fn(*ptrs, B, K, H, qa, pa, None)
    assert got == code, f"{entry}: {what}: got {got}, expected {code}"


def test_plan_mirror_keying():
    H, B, K = 9, 6, 5
    rng = np.random.default_rng(0)
    mean, std = rng.uniform(-0.5, 0.5, (H, B)), rng.uniform(0.1, 1.0, (H, B))
    full = plan_actions(11, mean, std, K, low=-5, high=5)
    # shards keyed by env_offset reproduce the slices of the full draw
    for b0, b1 in ((0, 2), (2, 5), (5, 6)):
        part = plan_actions(11, mean[:, b0:b1], std[:, b0:b1], K, low=-5, high=5, env_offset=b0)
        assert np.array_equal(part, full[:, b0:b1])
    # a different seed or step gives different draws
    other = plan_actions(12, mean, std, K, low=-5, high=5)
    assert not np.any(other == full)
    assert not np.any(full[0] == full[1]) and not np.any(full[1] == full[2])
    # N(0, 1) moments
    z = plan_actions(3, np.zeros((4, 64)), np.ones((4, 64)), 256, low=-1e9, high=1e9).reshape(-1)
    assert abs(z.mean()) < 5 / np.sqrt(z.size) and abs(z.std() - 1) < 0.02
    assert abs(np.mean(z ** 3)) < 0.05 and abs(np.mean(z ** 4) - 3) < 0.1
    # discrete: frequency of action 1 ~ p
    p = np.array([0.1, 0.5, 0.9])[None, :].repeat(8, 0)
    d = plan_actions(5, p, None, 4096, discrete=True)
    assert set(np.unique(d)) <= {0.0, 1.0}
    assert np.allclose(d.mean(axis=(0, 2)), [0.1, 0.5, 0.9], atol=0.01)


def test_plan_raises_without_dynamics_kernel():
    for eid in ("HopperRunning-v0", "HalfCheetahRunning-v0"):
        env = E.make(eid)
        with pytest.raises(NotImplementedError):
            env.plan(5)
        with pytest.raises(NotImplementedError):
            env.get_batch_plan_returns(np.zeros((1, 12)), np.zeros((5, 1)), np.ones((5, 1)), 8)


# =============================================================================================
# GPU
# =============================================================================================
def _starts(eid, B, dtype, fr, seed=0, perturb=True):
    """B start states of task ``eid``: the reset states, perturbed (balancing tasks then terminate inside the horizon)."""
    env = E.make(eid, freq_rate=fr, num_envs=B, dtype=dtype, device="cuda:0")
    env.reset(seed=seed)
    st = env.state
    if isinstance(st, dict):
        return {k: v.clone() for k, v in st.items()}
    st = st.clone()
    if perturb:
        g = torch.Generator(device="cpu").manual_seed(seed + 1)
        st += (0.3 * torch.randn(st.shape, generator=g, dtype=torch.float64)).to(st)
    return st


def _repeat(st, K):
    if isinstance(st, dict):
        return {k: v.repeat_interleave(K, 0) for k, v in st.items()}
    return st.repeat_interleave(K, 0)


def _dist(env, H, B, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    if len(env.action_space.shape) == 0:
        return torch.rand((H, B), generator=g, dtype=torch.float64).to("cuda:0", env.dtype), None
    mean = 0.6 * (2 * torch.rand((H, B), generator=g, dtype=torch.float64) - 1)
    std = 0.2 + torch.rand((H, B), generator=g, dtype=torch.float64)
    return mean.to("cuda:0", env.dtype), std.to("cuda:0", env.dtype)


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


@pytest.mark.gpu
@pytest.mark.parametrize("H", [1, 17])
@pytest.mark.parametrize("BK", [(1, 257), (37, 64)])
@pytest.mark.parametrize("fr", [1, 4])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eid", ALL_IDS)
def test_plan_returns_equal_rollout(eid, dtype, fr, BK, H):
    B, K = BK
    env = E.make(eid, freq_rate=fr, num_envs=B, dtype=dtype, device="cuda:0")
    st = _starts(eid, B, dtype, fr, seed=B + H)
    mean, std = _dist(env, H, B, seed=H)
    twin = E.make(eid, freq_rate=fr, num_envs=B * K, dtype=dtype, device="cuda:0")
    twin.state = _repeat(st, K)
    terminated = 0
    for gamma in (1.0, 0.97):
        ret, act = env.get_batch_plan_returns(st, mean, std, K, seed=99, gamma=gamma, return_actions=True)
        assert ret.shape == (B, K) and ret.dtype == torch.float64 and act.shape == (H, B, K)
        twin.state = _repeat(st, K)
        rec = twin.rollout(H, actions=act.view(H, B * K), record=True, auto_reset=False, max_episode_steps=0)
        ref = _masked_return(rec["rewards"], rec["dones"], gamma)
        assert np.array_equal(ret.cpu().numpy().reshape(-1), ref), f"{eid} {dtype} fr={fr} B={B} K={K} H={H} gamma={gamma}"
        terminated += int(rec["dones"][:-1].any(dim=0).sum())
    if "Balancing" in eid and H == 17 and B > 1:
        assert terminated > 0, "perturbed balancing starts should terminate inside the horizon"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eid", ["CartPoleSwingUp-v0", "ContinuousCartPoleSwingUp-v0", "BoundaryInvertedPendulumSwingUp-v0",
                                 "ReboundInvertedDoublePendulumSwingUp-v0", "ChargedBallCentering-v0",
                                 "ContinuousChargedBallCentering-v0"])
def test_plan_actions_match_host_mirror(eid, dtype):
    H, B, K = 13, 5, 70
    env = E.make(eid, num_envs=B, dtype=dtype, device="cuda:0")
    st = _starts(eid, B, dtype, 1)
    mean, std = _dist(env, H, B, seed=3)
    discrete = std is None
    for off in (0, 3):
        env.env_offset = off
        _, act = env.get_batch_plan_returns(st, mean, std, K, seed=1234, return_actions=True)
        lo, hi = (0.0, 1.0) if discrete else (float(env.action_space.low[0]), float(env.action_space.high[0]))
        host = plan_actions(1234, mean.double().cpu().numpy(), None if discrete else std.double().cpu().numpy(), K, lo, hi,
                            discrete, np.float32 if dtype == torch.float32 else np.float64, env_offset=off)
        got = act.double().cpu().numpy()
        assert got.min() >= lo and got.max() <= hi
        if discrete:
            assert act.dtype == torch.uint8 and np.array_equal(got, host)
        elif dtype == torch.float64:
            scale = np.maximum(1.0, 10 * std.double().cpu().numpy())[:, :, None]
            assert np.all(np.abs(got - host) <= 1e-12 * scale)
        else:
            assert np.all(np.abs(got - host) <= np.spacing(np.abs(host).astype(np.float32)).astype(np.float64))
    env.env_offset = 0


def _eval_update(env, st, mean, std, K, q, seed):
    """one eval (with actions) and one update through the engine -> (returns, actions, new mean, new std, best_a, best_r)"""
    eng, start, B, _, base = env._plan_setup(st)
    for f in ("method", "elites", "temperature", "momentum", "min_std", "gamma"):
        setattr(base, f, getattr(q, f))
    base.seed = seed
    returns, act = eng.plan_eval(start, mean, std, K, base, True)
    m, s = mean.clone(), std.clone() if std is not None else None
    best_a, best_r = eng.plan_update(returns, m, s, base, True)
    return returns, act, m, s, best_a, best_r


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("case", [
    ("ContinuousCartPoleSwingUp-v0", "cem", dict(elites=16)),
    ("ContinuousCartPoleSwingUp-v0", "mppi", dict(temperature=0.5)),
    ("ContinuousCartPoleSwingUp-v0", "mppi", dict(temperature=1e-3)),  # a large return spread: weights far from uniform
    ("BoundaryInvertedPendulumSwingUp-v0", "cem", dict(elites=1, momentum=0.3, min_std=0.2)),
    ("ReboundInvertedDoublePendulumSwingUp-v0", "mppi", dict(temperature=2.0, momentum=0.5)),
    ("CartPoleSwingUp-v0", "cem", dict(elites=40, momentum=0.25)),
    ("ChargedBallCentering-v0", "mppi", dict(temperature=0.1)),
    ("ContinuousChargedBallCentering-v0", "cem", dict(elites=8, min_std=0.5)),
], ids=lambda c: f"{c[0]}-{c[1]}-{'-'.join(f'{k}{v}' for k, v in c[2].items())}")
def test_plan_update_matches_restatement(case, dtype):
    eid, method, kw = case
    H, B, K = 21, 7, 300
    env = E.make(eid, num_envs=B, dtype=dtype, device="cuda:0")
    st = _starts(eid, B, dtype, 1, perturb=False)
    mean, std = _dist(env, H, B, seed=5)
    discrete = std is None
    q = _lib.PlanParams()
    q.method = {"cem": _lib.PLAN_CEM, "mppi": _lib.PLAN_MPPI}[method]
    q.elites, q.temperature, q.momentum, q.min_std, q.gamma = kw.get("elites", 1), kw.get("temperature", 1.0), kw.get("momentum", 0.0), \
        kw.get("min_std", 0.0), 0.99
    returns, act, m, s, best_a, best_r = _eval_update(env, st, mean, std, K, q, seed=77)
    r = returns.cpu().numpy()
    if method == "mppi" and kw["temperature"] < 0.01:
        spread = (r.max(1) - r.min(1)) / kw["temperature"]
        assert spread.min() > 50, "the large-spread case should make most weights underflow"
    ref_m, ref_s, order = refit(act.double().cpu().numpy(), r, mean.double().cpu().numpy(),
                                None if discrete else std.double().cpu().numpy(), method, discrete=discrete, **kw)
    tol = 1e-12 if dtype == torch.float64 else 1e-6
    assert np.allclose(m.double().cpu().numpy(), ref_m, rtol=tol, atol=tol)
    if method == "cem" and kw.get("momentum", 0.0) == 0.0:  # with momentum 0 the new mean is the elites' mean itself
        assert_elite_set_identified(act.double().cpu().numpy(), order, kw["elites"], tol)
    if discrete:
        assert s is None and m.min() >= 0 and m.max() <= 1
    else:
        assert np.allclose(s.double().cpu().numpy(), ref_s, rtol=tol, atol=tol)
        assert s.min() >= kw.get("min_std", 0.0)
    # the argmax candidate under (return desc, k asc)
    arg = np.lexsort((np.arange(K)[None].repeat(B, 0), -r), axis=-1)[:, 0]
    assert np.array_equal(best_r.cpu().numpy(), r[np.arange(B), arg])
    assert best_a.dtype == act.dtype
    assert torch.equal(best_a, act[:, torch.arange(B), torch.as_tensor(arg, device=act.device)])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eid", ["ContinuousCartPoleBalancing-v0", "CartPoleBalancing-v0"])
def test_plan_update_ties(eid, dtype):
    """starts at rest balance for H steps whatever the actions: every return is H, so CEM takes the first E candidates and
    MPPI weighs all candidates the same."""
    H, B, K, Ee = 3, 4, 96, 10
    env = E.make(eid, num_envs=B, dtype=dtype, device="cuda:0")
    st = torch.zeros((B, 4), dtype=dtype, device="cuda:0")
    mean, std = _dist(env, H, B, seed=8)
    discrete = std is None
    for method in ("cem", "mppi"):
        q = _lib.PlanParams()
        q.method, q.elites, q.temperature = {"cem": _lib.PLAN_CEM, "mppi": _lib.PLAN_MPPI}[method], Ee, 1.0
        q.gamma = 1.0
        returns, act, m, s, best_a, _ = _eval_update(env, st, mean, std, K, q, seed=3)
        assert torch.all(returns == H)
        a = act.double().cpu().numpy()
        chosen = a[:, :, :Ee] if method == "cem" else a
        fit = chosen.mean(-1)
        tol = 1e-12 if dtype == torch.float64 else 1e-6
        assert np.allclose(m.double().cpu().numpy(), fit, rtol=tol, atol=tol)
        if not discrete:
            assert np.allclose(s.double().cpu().numpy(), chosen.std(-1), rtol=tol, atol=tol)
        assert torch.equal(best_a, act[:, :, 0])


def _update_twice(env, st, mean, std, K, q, seed, make_returns):
    """one eval (with actions), then two updates from ``make_returns(returns)`` -> (returns used, actions, [(mean, std, best_a,
    best_r)] * 2)"""
    eng, start, B, _, base = env._plan_setup(st)
    for f in ("method", "elites", "temperature", "momentum", "min_std", "gamma"):
        setattr(base, f, getattr(q, f))
    base.seed = seed
    returns, act = eng.plan_eval(start, mean, std, K, base, True)
    r = make_returns(returns).contiguous()
    outs = []
    for _ in range(2):
        m, s = mean.clone(), std.clone() if std is not None else None
        outs.append((m, s) + tuple(eng.plan_update(r, m, s, base, True)))
    return r, act, outs


def _same_bits(x, y):
    if x is None or y is None:
        return x is None and y is None
    return x.dtype == y.dtype and torch.equal(x.contiguous().view(torch.uint8), y.contiguous().view(torch.uint8))


def _plan_params(method, elites, temperature):
    q = _lib.PlanParams()
    q.method, q.elites, q.temperature, q.gamma = {"cem": _lib.PLAN_CEM, "mppi": _lib.PLAN_MPPI}[method], elites, temperature, 1.0
    return q


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eid", ["ContinuousCartPoleSwingUp-v0", "CartPoleSwingUp-v0"])
def test_plan_update_nonfinite_returns(eid, dtype):
    """Returns that are NaN or -inf (a diverged model, a NaN start): NaN ranks below every number and weighs 0; with no finite
    maximum every MPPI weight is 0 and the weights fall back to uniform.  K = 300 spreads the candidates over every warp of
    the CTA; two calls give the same bits."""
    H, B, K, Ee = 9, 5, 300, 24
    env = E.make(eid, num_envs=B, dtype=dtype, device="cuda:0")
    st = _starts(eid, B, dtype, 1, perturb=False)
    mean, std = _dist(env, H, B, seed=11)
    discrete = std is None
    g = torch.Generator(device="cpu").manual_seed(3)

    def mixed(r):
        x = r.clone()
        u = torch.rand(x.shape, generator=g).to(x.device)
        x[u < 0.3] = float("nan")
        x[(u >= 0.3) & (u < 0.4)] = float("-inf")
        return x

    cases = {"all NaN": lambda r: torch.full_like(r, float("nan")), "all -inf": lambda r: torch.full_like(r, float("-inf")),
             "mixed": mixed}
    tol = 1e-12 if dtype == torch.float64 else 1e-6
    for method in ("cem", "mppi"):
        for what, make in cases.items():
            r, act, outs = _update_twice(env, st, mean, std, K, _plan_params(method, Ee, 0.5), 19, make)
            assert all(_same_bits(x, y) for x, y in zip(outs[0], outs[1])), f"{method} {what}: two calls differ"
            m, s, best_a, best_r = outs[0]
            a = act.double().cpu().numpy()
            rn = r.cpu().numpy()
            ref_m, ref_s, order = refit(a, rn, mean.double().cpu().numpy(), None if discrete else std.double().cpu().numpy(),
                                        method, elites=Ee, temperature=0.5, discrete=discrete)
            if what != "mixed":  # no finite return: CEM takes the first E candidates, MPPI weighs all K the same
                chosen = a[:, :, :Ee] if method == "cem" else a
                assert np.allclose(ref_m, chosen.mean(-1), rtol=1e-12, atol=1e-12)
            assert np.allclose(m.double().cpu().numpy(), ref_m, rtol=tol, atol=tol), f"{method} {what}: mean"
            if not discrete:
                assert np.allclose(s.double().cpu().numpy(), ref_s, rtol=tol, atol=tol), f"{method} {what}: std"
            arg = cem_order(rn)[:, 0]
            assert torch.equal(best_a, act[:, torch.arange(B), torch.as_tensor(arg, device=act.device)])
            assert _same_bits(best_r, r[torch.arange(B, device=r.device), torch.as_tensor(arg, device=r.device)])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eid", ["ContinuousCartPoleSwingUp-v0", "CartPoleSwingUp-v0"])
def test_plan_update_cem_tied_returns(eid, dtype):
    """Returns with many exact ties (four distinct values over K = 300): the elite set is the first E candidates in (return
    descending, k ascending) order, checked as a set, not only through the fitted mean."""
    H, B, K, Ee = 13, 6, 300, 50
    env = E.make(eid, num_envs=B, dtype=dtype, device="cuda:0")
    st = _starts(eid, B, dtype, 1, perturb=False)
    mean, std = _dist(env, H, B, seed=12)
    discrete = std is None
    g = torch.Generator(device="cpu").manual_seed(4)
    tied = lambda r: torch.randint(0, 4, r.shape, generator=g).to(r.device, torch.float64)  # noqa: E731
    r, act, outs = _update_twice(env, st, mean, std, K, _plan_params("cem", Ee, 1.0), 23, tied)
    assert all(_same_bits(x, y) for x, y in zip(outs[0], outs[1]))
    m, s, _, _ = outs[0]
    a = act.double().cpu().numpy()
    ref_m, ref_s, order = refit(a, r.cpu().numpy(), mean.double().cpu().numpy(), None if discrete else std.double().cpu().numpy(),
                                "cem", elites=Ee, discrete=discrete)
    tol = 1e-12 if dtype == torch.float64 else 1e-6
    assert np.allclose(m.double().cpu().numpy(), ref_m, rtol=tol, atol=tol)
    if not discrete:
        assert np.allclose(s.double().cpu().numpy(), ref_s, rtol=tol, atol=tol)
    assert_elite_set_identified(a, order, Ee, tol)


@pytest.mark.gpu
def test_plan_invariants():
    eid, H, B, K = "ContinuousCartPoleSwingUp-v0", 11, 19, 128
    env = E.make(eid, num_envs=B, dtype=torch.float32, device="cuda:0")
    env.reset(seed=4)
    env.step(torch.zeros(B, device="cuda:0"))
    env.freeze()
    state0 = env.state.clone()
    stats0 = env.stats.clone()
    snap0 = [t.clone() for t in env.frozen_state]
    bufs0 = [t.clone() for t in env._engine._bufs]
    mean, std = _dist(env, H, B, seed=1)
    # determinism
    r1, a1 = env.get_batch_plan_returns(env.state, mean, std, K, seed=5, return_actions=True)
    r2, a2 = env.get_batch_plan_returns(env.state, mean, std, K, seed=5, return_actions=True)
    assert torch.equal(r1, r2) and torch.equal(a1, a2)
    p1 = env.plan(H, candidates=K, iterations=3, method="mppi", temperature=0.3, seed=6)
    p2 = env.plan(H, candidates=K, iterations=3, method="mppi", temperature=0.3, seed=6)
    for x, y in zip(p1, p2):
        assert torch.equal(x, y)
    # statelessness
    assert torch.equal(env.state, state0) and torch.equal(env.stats, stats0)
    assert all(torch.equal(x, y) for x, y in zip(env.frozen_state, snap0))
    assert all(torch.equal(x, y) for x, y in zip(env._engine._bufs, bufs0))
    # sharding: rows [b0, b1) with env_offset = b0 equal the slice of the full call
    st = env.state.clone()
    for b0, b1 in ((0, 7), (7, 19)):
        env.env_offset = b0
        r, a = env.get_batch_plan_returns(st[b0:b1], mean[:, b0:b1], std[:, b0:b1], K, seed=5, return_actions=True)
        assert torch.equal(r, r1[b0:b1]) and torch.equal(a, a1[:, b0:b1])
    env.env_offset = 0
    # numpy in, numpy out
    rn = env.get_batch_plan_returns(st.cpu().numpy(), mean.cpu().numpy(), std.cpu().numpy(), K, seed=5)
    assert isinstance(rn, np.ndarray) and np.array_equal(rn, r1.cpu().numpy())
    # unseeded planning draws fresh keys without moving the initial-state stream of a later unseeded reset()
    twin = E.make(eid, num_envs=B, dtype=torch.float32, device="cuda:0")
    env.reset(seed=8)
    twin.reset(seed=8)
    q1 = env.plan(H, candidates=K, iterations=1)
    q2 = env.plan(H, candidates=K, iterations=1)
    assert not torch.equal(q1.returns, q2.returns)
    env.get_batch_plan_returns(env.state, mean, std, K)
    assert torch.equal(env.reset()[0], twin.reset()[0])


@pytest.mark.gpu
def test_plan_past_resident_grid():
    eid, H = "ContinuousCartPoleSwingUp-v0", 5
    B, K = 75, 4042  # 303150 candidates > 148 SMs x 2048 threads
    env = E.make(eid, num_envs=B, dtype=torch.float32, device="cuda:0")
    st = _starts(eid, B, torch.float32, 1)
    mean, std = _dist(env, H, B)
    ret, act = env.get_batch_plan_returns(st, mean, std, K, seed=2, return_actions=True)
    twin = E.make(eid, num_envs=B * K, dtype=torch.float32, device="cuda:0")
    twin.state = _repeat(st, K)
    rec = twin.rollout(H, actions=act.view(H, B * K), record=True, auto_reset=False, max_episode_steps=0)
    assert np.array_equal(ret.cpu().numpy().reshape(-1), _masked_return(rec["rewards"], rec["dones"], 1.0))


@pytest.mark.gpu
def test_plan_actions_past_2_31_elements():
    eid, B, K, H = "CartPoleSwingUp-v0", 1024, 4096, 513  # H B K = 2.15e9 uint8 actions
    assert H * B * K > 2 ** 31
    env = E.make(eid, num_envs=B, dtype=torch.float32, device="cuda:0")
    st = _starts(eid, B, torch.float32, 1)
    mean, _ = _dist(env, H, B, seed=2)
    ret, act = env.get_batch_plan_returns(st, mean, None, K, seed=9, return_actions=True)
    ret_only = env.get_batch_plan_returns(st, mean, None, K, seed=9)
    assert torch.equal(ret, ret_only)
    rows, cols = np.array([0, 511, 1023]), np.array([0, 4095])
    host = plan_actions(9, mean.double().cpu().numpy(), None, K, discrete=True, rows=rows, cols=cols)
    got = act[:, torch.as_tensor(rows)][:, :, torch.as_tensor(cols)].double().cpu().numpy()
    assert np.array_equal(got, host)


@pytest.mark.gpu
@pytest.mark.parametrize("eid", ["ContinuousCartPoleSwingUp-v0", "BoundaryInvertedPendulumSwingUp-v0"])
def test_plan_beats_zero_plan(eid):
    H, B = 40, 8
    env = E.make(eid, num_envs=B, dtype=torch.float32, device="cuda:0")
    env.reset(seed=0)
    res = env.plan(H, candidates=512, iterations=5, elites=64, seed=7)
    assert res.mean.shape == (H, B) and res.std.shape == (H, B) and res.returns.shape == (B, 512)

    def score(actions):
        _, _, rew, done = env.get_batch_trajectory(env.state, actions)
        return _masked_return(rew, done, 1.0)

    planned, zero = score(res.mean), score(torch.zeros_like(res.mean))
    assert np.all(planned > zero), (planned, zero)
