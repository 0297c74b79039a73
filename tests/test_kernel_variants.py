"""Every dispatch variant of the float32 kernels against the float64 oracle, on IDENTICAL float32 inputs.

The golden vectors and the older oracle tests run batches below 8192 envs, i.e. the scalar small-batch cart-pole
kernel only.  Here the TMA-staged packed kernel (two envs per thread, per-lane cold redo, ragged last chunk, ring
recycling) meets the oracle in every template variant: the eight cart-pole / inverted-pendulum models x freq_rate
1..4 (the run-time freq_rate instance included) x every action kind x an aligned and an unaligned action pointer,
with rows planted on the cold-path threshold, the sincos ranges, non-finite values and the termination bounds.  Also:
the charged ball's EPT = 4 launch shape, the scoring layouts (trajectory walk, ragged walk, odd offsets, statistics,
trajectory scoring of odd env counts) and the sum-of-squares pass.

Bar (BASELINE.json north star): 1e-5 rel + 1e-6 abs per step; flags exact except within tolerance of a threshold.
Allowances follow tests/test_gpu_parity.py: ulp32(theta) for |theta| beyond the fast sincos range, half an ulp of a
float32-held variable per sub-step for freq_rate > 1, the operand magnitude of the batch-wide control cost; and 2^-20 of
the summed |increments| of a sub-stepped variable (the float32 rounding of accelerations of hundreds of m/s^2).
"""
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import emei_oracle as O

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore", category=RuntimeWarning)

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib  # noqa: E402
from emei_b200.engine import score, score_seq  # noqa: E402

DT = 0.02
COLD_RATE = (math.pi / 4) / DT  # 39.27 rad/s: a sub-step increment beyond pi/4 sends the env to the cold (libm) path
SMALL_BATCH = 8192              # cartpole_tma.cuh kSmallBatch: from here on the TMA kernel steps the batch
CHUNK = 512                     # envs per TMA chunk; lane A of a warp's 64 envs = 64 w + l, lane B = 64 w + 32 + l

CP = {
    "balancing": "CartPoleBalancing-v0",
    "swingup": "CartPoleSwingUp-v0",
    "continuous_balancing": "ContinuousCartPoleBalancing-v0",
    "continuous_swingup": "ContinuousCartPoleSwingUp-v0",
}
IP = {
    "ip_rebound_balancing": "ReboundInvertedPendulumBalancing-v0",
    "ip_boundary_balancing": "BoundaryInvertedPendulumBalancing-v0",
    "ip_rebound_swingup": "ReboundInvertedPendulumSwingUp-v0",
    "ip_boundary_swingup": "BoundaryInvertedPendulumSwingUp-v0",
}
I2P = {
    "i2p_rebound_balancing": "ReboundInvertedDoublePendulumBalancing-v0",
    "i2p_boundary_balancing": "BoundaryInvertedDoublePendulumBalancing-v0",
    "i2p_rebound_swingup": "ReboundInvertedDoublePendulumSwingUp-v0",
    "i2p_boundary_swingup": "BoundaryInvertedDoublePendulumSwingUp-v0",
}
DISCRETE = (torch.uint8, torch.bool, torch.int32, torch.int64)
CONTINUOUS = (torch.float32, torch.float64)


def close64(a, b, tol=1e-12):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    same_inf = np.isinf(a) & (a == b)
    return np.all(both_nan | same_inf | (np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))))


def within32(a, ref, scale=1.0):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(a - ref) <= scale * (1e-6 + 1e-5 * np.abs(ref))


def agree(got, ref, tol):
    """elementwise: within `tol` where the oracle is finite; the same NaN / the same infinity where it is not"""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    fin = np.isfinite(ref)
    with np.errstate(invalid="ignore"):
        return np.where(fin, np.abs(got - ref) <= tol, (np.isnan(got) & np.isnan(ref)) | (got == ref))


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a.view(np.uint8)


# ================================================================================================
# cart-pole / inverted pendulum float32 step
# ================================================================================================
def planted_values(ip):
    """(x, theta, theta_dot) of the rows where these kernels go wrong (None: keep the benign value): both sides of the
    cold-path threshold |theta_dot| dt = pi/4, a rate that only a later sub-step carries over it (|theta_ddot| of
    15-25 rad/s^2 at a horizontal pole), the sincos ranges (fast <= 1e5 < reduced <= 4e6 < libm only), non-finite
    values, and the cart at the termination threshold / rail ends."""
    x_edges = (2.0,) if ip else (2.4, 5.0)
    rows = []
    for w in (39.0, 39.25, 39.3, 40.0, 45.0, 60.0, 78.0):
        rows += [(None, None, w), (None, None, -w)]
    for th in (0.5 * np.pi, -0.5 * np.pi, 2.0, -2.0):
        rows += [(None, th, 39.1), (None, th, -39.1)]
    for th in (1e5 - 1.0, 1e5 + 3.0, -1e5 - 3.0, 3.9e6, -4.1e6, 1e7):
        rows.append((None, th, None))
    for v in (np.nan, np.inf, -np.inf):
        rows += [(None, v, None), (None, None, v), (v, None, None)]
    for e in x_edges:
        rows += [(e, None, None), (-e, None, None), (e - 1e-3, None, None), (-(e - 1e-3), None, None)]
    return rows


def plant(st, row, vals, ip):
    x, th, w = vals
    if x is not None:
        st[row, 0] = x
    if th is not None:
        st[row, 1 if ip else 2] = th
    if w is not None:
        st[row, 3] = w


def cp_ip_inputs(kind, n, seed, chunk_bases):
    """benign float32 states and actions for `n` envs, with every planted value in lane A only, in lane B only and in both
    lanes of a pair, at each chunk base of `chunk_bases`, and cold rows in the lanes of the ragged last chunk.
    -> (state [n,4] float32, action float32 ([n] discrete 0/1 values or [n,1] continuous), planted row indices)"""
    ip = kind in IP
    rng = np.random.default_rng(seed)
    if ip:
        st = rng.uniform(-1, 1, size=(n, 4)) * np.array([1.9, np.pi, 5.0, 8.0])
        act = rng.uniform(-3.5, 3.5, size=(n, 1))  # beyond ctrlrange: clamped like mj_step
    else:
        x_thr = O.cartpole_params(kind).x_threshold
        st = rng.uniform(-1, 1, size=(n, 4)) * np.array([0.9 * x_thr, 2.0, np.pi, 8.0])
        act = rng.uniform(-1, 1, size=(n, 1)) if kind.startswith("continuous") else rng.integers(0, 2, size=n)
    st = st.astype(np.float32)
    vals = planted_values(ip)
    rows = []
    for b in chunk_bases:
        for j, v in enumerate(vals):
            base = (b + j % 17) * CHUNK + 64 * ((j // 17) % 8)  # a (chunk, warp) of its own
            lane = j % 8
            for r in (base + lane, base + 32 + 8 + lane, base + 16 + lane, base + 48 + lane):  # A only, B only, A+B pair
                plant(st, r, v, ip)
                rows.append(r)
    tail = n % CHUNK
    if tail:
        last = n - tail
        cold = [(None, None, 78.0), (None, None, -60.0), (None, 1e7, None), (None, np.nan, None), (None, None, 45.0),
                (None, None, -40.0), (None, None, np.inf), (None, -4.1e6, None)]
        # lane A with a dead lane B (ragged), then pairs
        picks = [p for p in range(tail) if p % 64 < 32 and p + 32 >= tail] + [p for p in range(tail) if p % 64 < 32 and p + 32 < tail]
        for p, v in zip(picks, cold * 4):
            plant(st, last + p, v, ip)
            rows.append(last + p)
    return st, act.astype(np.float32), np.unique(np.array(rows))


def oracle_step(kind, st32, act, fr):
    """the float64 oracle on the float32 inputs, one sub-step at a time (its state is float64 between sub-steps, so this
    is its freq_rate step) -> (state, observation, reward, done, near-threshold mask, per-element peak |value| held
    between sub-steps, per-element sum of |increment| over the sub-steps, peak |theta_dot| at the start of sub-steps
    2..fr)"""
    y = st32.astype(np.float64)
    peak = np.zeros_like(y)
    path = np.zeros_like(y)
    later = np.zeros(y.shape[0])
    if kind in CP:
        p = O.cartpole_params(kind)
        force = O.cartpole_force(act, kind.startswith("continuous"), p)
        for s in range(fr):
            if s:
                peak = np.fmax(peak, np.abs(y))
                later = np.fmax(later, np.abs(y[:, 3]))
            y0, y = y, O.cartpole_step_f64ref(y, force, DT, 1, p)
            path += np.nan_to_num(np.abs(y - y0))
        rew, done = O.cartpole_reward(kind, y), O.cartpole_terminal(kind, y, p)
        near = np.abs(np.abs(y[:, 0]) - p.x_threshold) < 1e-4
        if not kind.endswith("swingup"):
            near |= np.abs(np.abs(y[:, 2]) - p.theta_threshold_radians) < 1e-4
        return y, y, rew, done, near, peak, path, later
    p = O.InvertedPendulumParams()
    ctrl = np.clip(act.astype(np.float64).reshape(-1), p.ctrl_low, p.ctrl_high)
    swing = kind.endswith("swingup")
    for s in range(fr):
        if s:
            peak = np.fmax(peak, np.abs(y))
            later = np.fmax(later, np.abs(y[:, 3]))
        y0 = y
        y, obs = O.ip_step(y, ctrl, DT, 1, swing, p, libm=True)
        path += np.nan_to_num(np.abs(y - y0))
    rew, done = O.ip_reward(kind, obs), O.ip_terminal(kind, obs, p)
    cy = np.cos(obs[:, 1])
    near = np.abs(np.abs(obs[:, 0]) - 2.0) < 1e-4 if "boundary" in kind else np.zeros(y.shape[0], dtype=bool)
    if kind == "ip_rebound_balancing":
        near |= np.abs(cy - 0.9) < 1e-4
    elif kind == "ip_boundary_balancing":
        near |= np.abs(cy) < 1e-4
    return y, obs, rew, done, near, peak, path, later


def assert_step_vs_oracle(got, st32, ref, kind, fr, rows=None):
    """got = (state, obs, reward, done) numpy of the rows `rows` (default all) of st32 / ref"""
    ip = kind in IP
    g_st, g_obs, g_rew, g_done = got
    r_st, r_obs, r_rew, r_done, near, peak, path, _ = (a if rows is None else a[rows] for a in ref)
    s0 = st32 if rows is None else st32[rows]
    th0 = np.abs(s0[:, 1 if ip else 2]).astype(np.float64)
    # beyond the range of the fast sincos (f32math.cuh kSinCosFastMax) the float32 quantisation of theta bounds the
    # agreement (test_gpu_parity.py)
    quant = np.where(th0 > 1e5, np.nan_to_num(np.spacing(th0.astype(np.float32)).astype(np.float64)) * 40.0 * DT * fr, 0.0)[:, None]
    # float32 evaluation of the increments: a few roundings of each sub-step's |increment| (an env at 78 rad/s carries
    # its cart from 3 m/s through 9 m/s back to 0 within one step; 1e-6 absolute is below float32's reach there)
    tol = 1e-6 + 1e-5 * np.abs(r_st) + quant + 2.0 ** -20 * path
    if fr > 1:  # half an ulp of every float32-held variable per sub-step (test_c1_protocol_ip_f32_teacher_forced_200_steps)
        big = np.fmax(np.fmax(np.abs(s0.astype(np.float64)), np.abs(r_st)), peak).astype(np.float32)
        tol = tol + fr * 0.5 * np.nan_to_num(np.spacing(big).astype(np.float64))
    ok = agree(g_st, r_st, tol)
    assert ok.all(), f"state: {(~ok.all(axis=1)).sum()} rows outside the envelope, first {np.argmin(ok.all(axis=1))}"
    if ip:  # observation: theta wrapped to [-pi, pi) -- compare on the circle
        fin = np.isfinite(r_obs[:, 1])
        dth = np.abs((g_obs[:, 1].astype(np.float64) - r_obs[:, 1] + np.pi) % (2 * np.pi) - np.pi)
        assert np.all(dth[fin] <= tol[fin, 1]) and np.all(np.isnan(g_obs[~fin, 1]))
        ok = agree(g_obs[:, [0, 2, 3]], r_obs[:, [0, 2, 3]], tol[:, [0, 2, 3]])
        assert ok.all()
    else:
        assert np.array_equal(bits(g_obs), bits(g_st))
    ok = agree(g_rew, r_rew, 1e-6 + 1e-5 * np.abs(r_rew) + quant)
    assert ok.all(), f"reward: {(~ok).sum()} rows outside the envelope, first {np.argmin(ok)}"
    assert np.array_equal(g_done[~near], r_done[~near]), f"{(g_done[~near] != r_done[~near]).sum()} flags differ"


def cp_ip_env(kind, fr, n):
    return E.make((CP | IP)[kind], freq_rate=fr, num_envs=n, dtype=torch.float32)


def action_tensor(values, dtype, offset):
    """device tensor of `values` in `dtype`; offset 1: a view one element into its allocation (not 16-byte aligned)"""
    v = torch.as_tensor(values).reshape(-1).cuda()
    buf = torch.zeros(v.numel() + offset, dtype=dtype, device="cuda")
    buf[offset:] = v.to(dtype)
    t = buf[offset:]
    assert (t.data_ptr() % 16 == 0) == (offset == 0)
    return t


def run_step(kind, fr, st32, act):
    env = cp_ip_env(kind, fr, st32.shape[0])
    env.state = st32
    obs, rew, done, _, _ = env.step(act)
    return env.state.cpu().numpy(), obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()


def action_kinds(kind):
    return CONTINUOUS if kind in IP or kind.startswith("continuous") else DISCRETE


@pytest.mark.parametrize("fr", (1, 2, 3, 4))
@pytest.mark.parametrize("kind", list(CP) + list(IP))
def test_cartpole_ip_f32_step_matrix(kind, fr):
    """8191 envs (the scalar small-batch kernel) and 8705 envs (the smallest TMA launch: 17 full chunks + a ragged one
    of a single env) for every action kind and an aligned / unaligned action pointer, against the oracle.  The first 8191
    rows of the TMA launch equal the small kernel's bit for bit, and every action encoding of the same values gives the
    same bits.  get_batch_next_obs (stateless) steps through the same kernel."""
    n = SMALL_BATCH + CHUNK + 1
    n_small = SMALL_BATCH - 1
    st, act, rows = cp_ip_inputs(kind, n, 7 * fr + len(kind), chunk_bases=(0,))
    ref = oracle_step(kind, st, act, fr)
    if fr > 1:  # the planted rows include one that only a later sub-step carries over the cold-path threshold
        assert np.any((np.abs(st[rows, 3]) < COLD_RATE) & (ref[7][rows] > COLD_RATE))
    first = None
    for dt in action_kinds(kind):
        for off in (0, 1):
            big = run_step(kind, fr, st, action_tensor(act, dt, off))
            small = run_step(kind, fr, st[:n_small], action_tensor(act[:n_small], dt, off))
            assert_step_vs_oracle(big, st, ref, kind, fr)
            assert_step_vs_oracle(small, st[:n_small], tuple(a[:n_small] for a in ref), kind, fr)
            for a, b in zip(small, big):
                assert np.array_equal(bits(a), bits(b[:n_small])), f"small kernel != TMA kernel ({dt}, offset {off})"
            if first is None:
                first = big
            for a, b in zip(big, first):
                assert np.array_equal(bits(a), bits(b)), f"{dt} offset {off} differs from {action_kinds(kind)[0]} aligned"
    # get_batch_next_obs: the stateless entry point at a TMA size
    env = cp_ip_env(kind, fr, 4)
    env.state = st[:4]
    env.freeze()
    nxt = env.get_batch_next_obs(torch.from_numpy(st).cuda(), action=action_tensor(act, action_kinds(kind)[0], 0))
    assert np.array_equal(bits(nxt.cpu().numpy()), bits(first[1]))
    assert env.num_envs == 4


def ring_slots(action_bytes):
    """cartpole_tma.cuh tma_ring_shape: slots of a launch with more chunks per CTA than the ring holds"""
    budget, slot = 208 * 1024, 2 * 256 * (16 + action_bytes)
    s = min(budget // slot, 32)
    s = -(-s // 4) * 4
    while s * slot > budget:
        s -= 4
    return s


@pytest.mark.parametrize("kind,dtype,fr", (
    ("swingup", torch.uint8, 4), ("balancing", torch.int32, 3), ("continuous_swingup", torch.float64, 1),
    ("ip_boundary_swingup", torch.float32, 4), ("ip_rebound_swingup", torch.float64, 2),
))
def test_cartpole_ip_f32_ring_recycling(kind, dtype, fr):
    """Just past SMs x slots x 512 envs every consumer group refills its slots (empty barriers, phase flips): planted rows
    at the start, in chunks read through recycled slots and in the ragged last chunk (300 envs), plus a strided
    subsample, against the oracle."""
    assert ring_slots(1) == 24 and ring_slots(4) == 20 and ring_slots(8) == 16
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    width = torch.empty(0, dtype=dtype).element_size()
    n_chunks = sms * ring_slots(width) + 1
    n = n_chunks * CHUNK + 300
    st, act, rows = cp_ip_inputs(kind, n, 11 * fr + width, chunk_bases=(0, n_chunks - 20))
    got = run_step(kind, fr, st, action_tensor(act, dtype, 0))
    idx = np.union1d(np.arange(0, n, 61), rows)
    ref = oracle_step(kind, st[idx], act[idx], fr)
    assert_step_vs_oracle(tuple(a[idx] for a in got), st[idx], ref, kind, fr)


# ================================================================================================
# charged ball float32 step: the EPT = 4 launch shape (n >= 2^24)
# ================================================================================================
def cb_substep_trace(on, ci, fre, Ef, fr, p, f32_force=False):
    """The oracle's env step one sub-step at a time, with the rows whose regime decision lies within tolerance of its
    threshold (take-off, landing radius, landing direction): the only rows where float32 flags may differ
    (tests/test_gpu_parity.py).  Returns (on, circle, free, near, ring): ring = on the ring at the start or end of some
    sub-step (a ball can land and take off again within one step of several sub-steps)."""
    import copy

    ps = copy.copy(p)
    ps.time_step = p.time_step / fr
    near = np.zeros(on.shape[0], dtype=bool)
    ring = on.copy()
    Ef = np.asarray(Ef, dtype=np.float64).reshape(-1)
    for _ in range(fr):
        th, om = ci[:, 0], ci[:, 1]
        lhs = p.mass_ball * om * om * p.radius + np.sin(th) * Ef
        rhs = np.cos(th) * p.mass_ball * p.gravity_acc
        near |= on & (np.abs(lhs - rhs) < 1e-4 * (1.0 + np.abs(lhs) + np.abs(rhs)))
        was_free = ~on
        on, ci, fre = O.charged_ball_step(on, ci, fre, Ef, 1, ps, f32_force=f32_force)
        r2 = fre[:, 0] ** 2 + fre[:, 1] ** 2
        near |= was_free & (np.abs(r2 - (p.radius ** 2 + 0.001)) < 1e-5)
        cross = fre[:, 2] * fre[:, 1] - fre[:, 3] * fre[:, 0]
        vp = np.hypot(fre[:, 2], fre[:, 3]) * np.sqrt(r2)
        near |= was_free & on & (np.abs(cross) < 1e-4 * vp)
        ring |= on
    return on, ci, fre, near, ring


def cb_assert_f32_step(got, ring, ci_in, ref_on, ref_ci, ref_fr, near):
    """flags exact except on `near` rows; state within 1.0 x (1e-6 + 1e-5 |ref|) plus the half-ulp rounding of the
    stored float32 angle, ulp32(theta) (1 + |w|) (tests/test_gpu_parity.py)"""
    got_on = got["on_circle"].astype(bool)
    bad = (got_on != ref_on) & ~near
    assert not bad.any(), f"{bad.sum()} regime flags differ away from the take-off / landing thresholds"
    ok_rows = (got_on == ref_on) & ~near
    th = np.maximum(np.abs(ref_ci[:, 0]), np.abs(ci_in[:, 0]))
    rep = (np.spacing(th.astype(np.float32)).astype(np.float64) * (1.0 + np.abs(ref_ci[:, 1])))[:, None]
    fr_err = np.abs(got["free_state"].astype(np.float64) - ref_fr)
    fr_tol = 1e-6 + 1e-5 * np.abs(ref_fr) + rep * ring[:, None]
    worst = (fr_err / fr_tol)[ok_rows].max()
    assert worst <= 1.0, f"free state: worst fraction of the envelope {worst}"
    oc = ok_rows & ref_on
    ci_err = np.abs(got["circle_state"].astype(np.float64) - ref_ci)
    worst_c = (ci_err / (1e-6 + 1e-5 * np.abs(ref_ci)))[oc].max() if oc.any() else 0.0
    assert worst_c <= 1.0, f"circle state: worst fraction of the envelope {worst_c}"
    return ok_rows


def cb_step(env, state, act):
    env.state = state
    _, rew, done, _, _ = env.step(act)
    st = env.state
    return [st["on_circle"].clone(), st["circle_state"].clone(), st["free_state"].clone(), rew.clone(), done.clone()]


@pytest.mark.parametrize("cont,fr", ((False, 1), (False, 3), (True, 1), (True, 3)))
def test_charged_ball_f32_ept4_vs_ept1_and_oracle(cont, fr):
    """n = 2^24 + 3 takes the 4-envs-per-thread shape; the same rows stepped as two sub-batches below 2^24 take the
    1-env shape: same bits, for every action kind (discrete kinds give the bits of uint8).  Planted ring rows with
    |theta| around 1e5 (the libm branch of cb_sincos) and NaN theta; all planted rows and a dense subsample against the
    oracle."""
    n = (1 << 24) + 3
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(17 + fr + 2 * cont)
    u = lambda lo, hi: lo + (hi - lo) * torch.rand(n, device=dev, generator=g)  # noqa: E731
    on = (torch.rand(n, device=dev, generator=g) < 0.5).to(torch.uint8)
    circle = torch.stack([u(-4.0, 10.0), u(-4.0, 4.0)], dim=1)
    ang, rad = u(0.0, 2 * math.pi), u(0.3, 1.04)
    free = torch.stack([rad * torch.sin(ang), rad * torch.cos(ang), u(-5.0, 5.0), u(-5.0, 5.0)], dim=1)
    planted = torch.tensor([5, 1029, 2 ** 23 + 1, 2 ** 24 - 7, n - 3, n - 2, n - 1] + list(range(4096, 4096 + 64, 3)), device=dev)
    th_vals = [1e5 - 1.0, 1e5 + 2.0, -1e5 - 5.0, 2.5e5, 1e6, float("nan")]
    on[planted] = 1
    circle[planted, 0] = torch.tensor((th_vals * 8)[: planted.numel()], device=dev)
    state = dict(on_circle=on, circle_state=circle, free_state=free)
    if cont:
        base = u(-1.0, 1.0)
        acts = [base, base.double()]
    else:
        base = torch.randint(0, 2, (n,), device=dev, generator=g, dtype=torch.uint8)
        acts = [base.to(dt) for dt in DISCRETE]
    cls = "ContinuousChargedBallCentering-v0" if cont else "ChargedBallCentering-v0"
    big = E.make(cls, freq_rate=fr, num_envs=n, dtype=torch.float32)
    h = n // 2
    lo = E.make(cls, freq_rate=fr, num_envs=h, dtype=torch.float32)
    hi = E.make(cls, freq_rate=fr, num_envs=n - h, dtype=torch.float32)
    first = None
    for a in acts:
        out = cb_step(big, state, a)
        parts = [cb_step(e, {k: v[s] for k, v in state.items()}, a[s]) for e, s in ((lo, slice(0, h)), (hi, slice(h, n)))]
        for x, y0, y1 in zip(out, *parts):
            assert torch.equal(x.view(torch.uint8), torch.cat([y0, y1]).view(torch.uint8)), f"EPT 4 != EPT 1 ({a.dtype})"
        if first is None:
            first = out
        for x, y in zip(out, first):
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8)), f"{a.dtype} differs from {acts[0].dtype}"
    idx = torch.unique(torch.cat([torch.arange(0, n, 89, device=dev), planted]))
    on0 = on[idx].cpu().numpy().astype(bool)
    ci32, fr32 = circle[idx].cpu().numpy(), free[idx].cpu().numpy()
    a_np = base[idx].cpu().numpy()
    p = O.ChargedBallParams()
    r_on, r_ci, r_fr, near, ring = cb_substep_trace(on0, ci32.astype(np.float64), fr32.astype(np.float64),
                                              O.charged_ball_force(a_np.reshape(-1, 1) if cont else a_np, cont, p), fr, p, f32_force=cont)
    got = {k: v[idx].cpu().numpy() for k, v in zip(("on_circle", "circle_state", "free_state"), first[:3])}
    rew = first[3][idx].cpu().numpy()
    nan_rows = np.isnan(ci32[:, 0])
    assert nan_rows.sum() >= 3 and np.all(np.isnan(got["free_state"][nan_rows])) and np.all(np.isnan(r_fr[nan_rows]))
    assert np.array_equal(got["on_circle"][nan_rows].astype(bool), r_on[nan_rows])
    fin = ~nan_rows
    if fr > 1:
        # Known limit of the float32 kernel: between sub-steps it keeps theta as a float32 and evaluates sincos of that
        # rounded angle (ulp32(1e5) = 0.008 rad), so omega drifts from the oracle by up to ~2e-3 per step at |theta| ~ 1e5
        # (the cart-pole kernels rotate (sin, cos) by the increments instead).  Those rows keep the EPT comparison above
        # and their regime flags; the envelope is asserted where the float32 angle resolves the sub-steps.
        big = fin & (np.abs(ci32[:, 0]) > 1e3)
        assert not ((got["on_circle"][big].astype(bool) != r_on[big]) & ~near[big]).any()
        fin &= ~big
    ok_rows = cb_assert_f32_step({k: v[fin] for k, v in got.items()}, ring[fin], ci32[fin].astype(np.float64), r_on[fin],
                                 r_ci[fin], r_fr[fin], near[fin])
    assert near.mean() < 0.01 and ok_rows.mean() > 0.99
    assert (~nan_rows & on0 & (np.abs(ci32[:, 0]) > 1e5)).sum() >= 20  # ring rows that take the libm branch of cb_sincos
    assert within32(rew[fin][ok_rows], O.charged_ball_reward(r_fr[fin], p)[ok_rows]).all()
    assert not first[4].any()


# ================================================================================================
# scoring (get_batch_reward / get_batch_terminal): every family, both precisions, every layout
# ================================================================================================
SCORING = {"CartPoleBalancing-v0": "balancing", "CartPoleSwingUp-v0": "swingup", "HopperRunning-v0": "hopper",
           "HalfCheetahRunning-v0": "halfcheetah", "ChargedBallCentering-v0": "charged_ball",
           **{v: k for k, v in IP.items()}, **{v: k for k, v in I2P.items()}}
MUJOCO = ("hopper", "halfcheetah")


def scoring_env(env_id, dtype):
    kw = dict(terminate_when_unhealthy=False) if env_id.startswith("Hopper") else {}
    return E.make(env_id, dtype=dtype, **kw)


def obs_dim(env):
    return _lib.lib.emei_family_obs_dim(env._scoring_params().family)


def random_obs(kind, shape, dtype, g):
    """observations that straddle every threshold of the family, with a NaN in one row of ~300"""
    d = shape[-1]
    scale = {"balancing": [3.0, 2.0, 0.3, 2.0], "swingup": [6.0, 2.0, 4.0, 2.0], "charged_ball": [0.7] * 4,
             "hopper": [1.0, 0.4, 0.15] + [60.0] * 9, "halfcheetah": [1.0] * 18}.get(kind)
    if scale is None:
        scale = [1.5, 2.0, 3.0, 5.0] if kind.startswith("ip") else [2.5, 0.8, 0.8, 3.0, 5.0, 5.0]
    o = torch.randn(shape, device="cuda", dtype=dtype, generator=g) * torch.tensor(scale, device="cuda", dtype=dtype)
    if kind == "hopper":
        o[..., 1] += 1.25
    flat = o.view(-1, d)
    rows = torch.randint(0, flat.shape[0], (max(1, flat.shape[0] // 300),), device="cuda", generator=g)
    flat[rows, torch.randint(0, d, rows.shape, device="cuda", generator=g)] = float("nan")
    return o


def oracle_scores(kind, env, o, p=None, a=None):
    if kind in ("balancing", "swingup"):
        return O.cartpole_reward(kind, o), O.cartpole_terminal(kind, o, O.cartpole_params(kind))
    if kind.startswith("ip_"):
        return O.ip_reward(kind, o), O.ip_terminal(kind, o)
    if kind.startswith("i2p_"):
        return O.i2p_reward(kind, o), O.i2p_terminal(kind, o)
    if kind == "hopper":
        hp = O.HopperParams(terminate_when_unhealthy=False, dt=env.dt)
        return O.hopper_reward(o, p, a, hp), O.hopper_terminal(o, hp)
    if kind == "halfcheetah":
        return O.halfcheetah_reward(o, p, a, O.HalfCheetahParams(dt=env.dt)), O.halfcheetah_terminal(o)
    return O.charged_ball_reward(o, O.ChargedBallParams()), O.charged_ball_terminal(o)


def near_threshold(kind, o):
    """rows within 1e-4 of a flag threshold of the family (test_pendulum_scoring_vs_golden)"""
    near = np.zeros(o.shape[0], dtype=bool)
    with np.errstate(invalid="ignore"):
        if kind in ("balancing", "swingup"):
            p = O.cartpole_params(kind)
            near |= np.abs(np.abs(o[:, 0]) - p.x_threshold) < 1e-4
            near |= (kind == "balancing") & (np.abs(np.abs(o[:, 2]) - p.theta_threshold_radians) < 1e-4)
        elif kind.startswith("ip_") or kind.startswith("i2p_"):
            ip = kind.startswith("ip_")
            y = np.cos(o[:, 1]) if ip else np.cos(o[:, 1]) + np.cos(o[:, 1] + o[:, 2])
            y_thr = {"ip_rebound_balancing": 0.9, "ip_boundary_balancing": 0.0, "i2p_rebound_balancing": 1.5,
                     "i2p_boundary_balancing": 0.0}.get(kind)
            if y_thr is not None:
                near |= np.abs(y - y_thr) < 1e-4
            if "boundary" in kind:
                near |= np.abs(np.abs(o[:, 0]) - (2.0 if ip else 3.0)) < 1e-4
        elif kind == "hopper":
            near |= np.abs(o[:, 1] - 0.7) < 1e-4
            near |= (np.abs(np.abs(o[:, 2:]) - 100.0) < 1e-4 * 100.0).any(axis=1)
    return near


def assert_scores(kind, env, r, d, o, p=None, a=None):
    """r, d: device outputs for the rows o (and p, a) -> compare with the oracle on the same values"""
    o64 = o.double().cpu().numpy()
    p64 = p.double().cpu().numpy() if p is not None else None
    a64 = a.double().cpu().numpy() if a is not None else None
    ref_r, ref_d = oracle_scores(kind, env, o64, p64, a64)
    got_r, got_d = r.double().cpu().numpy(), d.cpu().numpy()
    assert got_r.shape == ref_r.shape and got_d.shape == ref_d.shape
    if env.dtype == torch.float64:
        assert close64(got_r, ref_r), f"reward: worst {np.nanmax(np.abs(got_r - ref_r))}"
        assert np.array_equal(got_d, ref_d)
        return
    if kind in MUJOCO:  # the batch-wide control cost is subtracted from O(1) terms: its magnitude is what float32 resolves
        cc = (1e-3 if kind == "hopper" else 0.1) * float(np.sum(np.square(a64)))
        ok = agree(got_r, ref_r, 1e-6 + 1e-5 * (np.abs(ref_r) + cc))
    else:
        ok = agree(got_r, ref_r, 1e-6 + 1e-5 * np.abs(ref_r))
    assert ok.all(), f"reward: {(~ok).sum()} rows outside the envelope"
    near = near_threshold(kind, o64)
    assert np.array_equal(got_d[~near], ref_d[~near]) and near.mean() < 0.01


def score_checked(kind, env, stats, o, p=None, a=None):
    env.accumulate_scoring_stats = stats
    env.reset_stats()
    r, d, _ = score(env, env._scoring_params(), o, p, a)
    assert_scores(kind, env, r, d, o, p, a)
    if stats:
        rs, dc = env.read_stats()
        tot = float(r.double().sum())
        assert dc == int(d.sum())
        assert (math.isnan(rs) and math.isnan(tot)) or abs(rs - tot) <= 1e-9 * max(1.0, float(r.double().abs().nansum()))
    else:
        assert env.read_stats() == (0.0, 0)


@pytest.mark.parametrize("stats", (False, True))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("env_id", list(SCORING))
def test_scoring_layouts_vs_oracle(env_id, dtype, stats):
    """Separately allocated rows and a slice at an odd offset for every family; for Hopper / HalfCheetah also the two
    shifted views of a trajectory with 255 / 256 / 257 columns (flat kernel / trajectory walk / realigned copy) and a
    buf[:m] / buf[k:] pair whose walk ends in a ragged row (m % k != 0).  With statistics the row kernel runs one
    resident wave; without, a full grid."""
    kind = SCORING[env_id]
    env = scoring_env(env_id, dtype)
    d = obs_dim(env)
    g = torch.Generator(device="cuda").manual_seed(len(env_id) * 7 + (dtype == torch.float32))
    n = 3001
    o = random_obs(kind, (n + 1, d), dtype, g)
    if kind not in MUJOCO:
        score_checked(kind, env, stats, o[:n])
        score_checked(kind, env, stats, o[1:])
        return
    a_dim = 3 if kind == "hopper" else 6
    p = random_obs(kind, (n + 1, d), dtype, g)
    a = torch.rand((n + 1, a_dim), device="cuda", dtype=dtype, generator=g) * 2 - 1
    score_checked(kind, env, stats, o[:n], p[:n], a[:n])
    score_checked(kind, env, stats, o[1:], p[1:], a[1:])  # odd offsets: 48 / 72-byte rows, 12 / 24-byte actions
    T = 5
    for k in (255, 256, 257):
        seq = random_obs(kind, (T + 1, k, d), dtype, g)
        act = torch.rand((T * k, a_dim), device="cuda", dtype=dtype, generator=g) * 2 - 1
        score_checked(kind, env, stats, seq[1:].reshape(T * k, d), seq[:-1].reshape(T * k, d), act)
    k, m = 256, 3 * 256 + 77
    buf = random_obs(kind, (m + k, d), dtype, g)
    act = torch.rand((m, a_dim), device="cuda", dtype=dtype, generator=g) * 2 - 1
    score_checked(kind, env, stats, buf[k:], buf[:m], act)


@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("env_id", list(SCORING))
def test_sequence_scoring_odd_env_count(env_id, dtype):
    """Trajectory scoring of an odd number of envs: rows of t >= 1 lose 16-byte alignment for 24- and 72-byte rows
    (I2P / HalfCheetah in float32), where the flat views are scored instead -- with the [T, n, A] actions of the whole
    batch in the control cost."""
    kind = SCORING[env_id]
    env = scoring_env(env_id, dtype)
    d = obs_dim(env)
    g = torch.Generator(device="cuda").manual_seed(len(env_id) + 3)
    T, n = 3, 301
    seq = random_obs(kind, (T + 1, n, d), dtype, g)
    a = None
    if kind in MUJOCO:
        a = torch.rand((T, n, 3 if kind == "hopper" else 6), device="cuda", dtype=dtype, generator=g) * 2 - 1
    if hasattr(env, "get_batch_reward_terminal_seq"):
        r, dn = env.get_batch_reward_terminal_seq(seq, a)
    else:
        r, dn, _ = score_seq(env, env._scoring_params(), seq)
    assert r.shape == (T, n, 1) and dn.shape == (T, n, 1) and dn.dtype == torch.bool
    flat_a = a.reshape(T * n, -1) if a is not None else None
    assert_scores(kind, env, r.reshape(-1, 1), dn.reshape(-1, 1), seq[1:].reshape(T * n, d), seq[:-1].reshape(T * n, d), flat_a)


@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_sumsq_tails_grid_cap_and_repeat(dtype):
    """emei_sumsq_* against numpy in float64: every tail length numel % V (V = elements per 128-bit load; the tail
    elements are the largest of the batch), sizes above the 1184-CTA grid cap, and three back-to-back calls on one
    workspace giving the same bits (the last CTA leaves the ticket counter at zero)."""
    env = E.make("HopperRunning-v0", dtype=dtype)
    V = 16 // torch.empty(0, dtype=dtype).element_size()
    cap = 148 * 8 * 256 * V  # kSumsqMaxBlocks CTAs of 256 threads, one 128-bit load each
    ws = torch.zeros(_lib.SUMSQ_WORKSPACE_BYTES // 8, dtype=torch.float64, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(23)
    for base in (1000 * V, 8 * cap):
        for tail in range(V):
            x = torch.randn(base + tail, device="cuda", dtype=dtype, generator=g)
            if tail:
                x[-tail:] = 1000.0 + torch.arange(tail, device="cuda", dtype=dtype)
            want = float(np.sum(np.square(x.cpu().numpy().astype(np.float64))))
            got = []
            for _ in range(3):
                out = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
                env._call("emei_sumsq", x.data_ptr(), x.numel(), out.data_ptr(), ws.data_ptr(), env._stream())
                got.append(float(out.item()))
            assert abs(got[0] - want) <= 1e-12 * want, f"numel {x.numel()}: {got[0]} != {want}"
            assert got[0] == got[1] == got[2]


# ================================================================================================
# analytic inverted double pendulum float32 step
# ================================================================================================
@pytest.mark.parametrize("fr", (1, 3))
@pytest.mark.parametrize("kind", ("i2p_boundary_balancing", "i2p_rebound_swingup"))
def test_i2p_step_f32_remaining_models_vs_oracle(kind, fr):
    """the two models that test_gpu_parity.py leaves out, at freq_rate 1 and 3 (tolerance of that file: the float32
    evaluation error of the acceleration, 2e-5 |delta v|, on the velocity rows)"""
    n = 4096
    rng = np.random.default_rng(3003 + fr)
    st = rng.uniform(-1, 1, size=(n, 6)) * np.array([2.9, np.pi, np.pi, 4.0, 8.0, 10.0])
    st[n // 8 : n // 4, 0] = np.sign(st[n // 8 : n // 4, 0]) * rng.uniform(2.95, 3.05, n // 4 - n // 8)  # the rail ends
    st[n // 4 : n // 2, 1:3] *= 0.1  # near upright: the balancing variants' y threshold
    act = rng.uniform(-1.3, 1.3, size=(n, 1)).astype(np.float32)  # beyond ctrlrange: clamped like mj_step
    st32 = st.astype(np.float32)
    p = O.I2PParams()
    ref_state, _ = O.i2p_step(st32.astype(np.float64), act.astype(np.float64), 0.02, fr, kind.endswith("swingup"), p)
    env = E.make(I2P[kind], freq_rate=fr, num_envs=n, dtype=torch.float32)
    env.state = st32
    obs, rew, done, _, _ = env.step(act)
    got = env.state.cpu().numpy()
    acc = np.abs(ref_state[:, 3:] - st32[:, 3:].astype(np.float64))
    tol = 1e-6 + 1e-5 * np.abs(ref_state)
    tol[:, 3:] += 2e-5 * acc
    err = np.abs(got - ref_state) / tol
    assert err.max() <= 1.0, f"worst fraction of the envelope {err.max()}"
    o = obs.cpu().numpy()
    assert np.array_equal(o[:, [0, 3, 4, 5]], got[:, [0, 3, 4, 5]])
    # reward and flags of the kernel's own observation
    o64 = o.astype(np.float64)
    assert within32(rew.cpu().numpy(), O.i2p_reward(kind, o64)).all()
    near = near_threshold(kind, o64)
    assert np.array_equal(done.cpu().numpy()[~near], O.i2p_terminal(kind, o64)[~near]) and near.mean() < 0.01
