"""The float32 reference-arithmetic steps against the float64 oracle, and the rollouts' counter streams past their first
Philox block.

Each cart-pole / inverted-pendulum / charged-ball task has two float32 implementations: the lean kernels (cartpole_tma.cuh,
cartpole_f32.cuh, charged_ball_f32.cuh) and the generic device step of kernels.cuh instantiated with float.  The generic
one serves emei_ip_step_noisy_f32 (every float32 inverted pendulum built with obs_noise_params),
emei_cartpole_rollout_ref_f32 (with and without noise) and emei_charged_ball_rollout_ref_f32.  It is held here to the bar
the lean kernels meet on the same rows: 1.0 x (1e-5 |ref| + 1e-6) per teacher-forced step, from the identical
float32-rounded input, on the inputs where float32 goes wrong -- un-reset 200-step trajectories at freq_rate 4, unwrapped
angles of hundreds of radians and landings at every position on the ring.

A call with horizon 1, no auto-reset, no TimeLimit and teacher-forced actions is one step per env from caller rows, so
one launch evaluates many independent teacher-forced steps.  Each check prints the worst fraction of its envelope."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from oracle import emei_oracle as O
from oracle import philox as P
from oracle import rollout_oracle as RO

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib  # noqa: E402
from test_gpu_parity import CARTPOLE, IP, _noise_seed, cb_assert_f32_step, cb_substep_trace, ip_inputs, within32  # noqa: E402

pytestmark = pytest.mark.gpu

SIG = np.array([0.01, 0.01, 0.03, 0.03])  # obs_noise_params=(0.01, 0.03): sigma of [x, theta, v, omega]


def _env_params(env):
    """A private copy of the env's C parameter struct (the engine sets action_kind per call)."""
    src = env._ensure_engine().params
    p = type(src)()
    ctypes.memmove(ctypes.byref(p), ctypes.byref(src), ctypes.sizeof(p))
    return p


def _action_array(act, continuous):
    """[T, n] actions -> (device tensor, EMEI_ACTION_* kind): float32 for a Box, uint8 for Discrete(2)."""
    if continuous:
        return torch.as_tensor(np.ascontiguousarray(act, dtype=np.float32)).cuda(), _lib.ACTION_CONTINUOUS_F32
    return torch.as_tensor(np.ascontiguousarray(act, dtype=np.uint8)).cuda(), _lib.ACTION_DISCRETE_U8


def _one_step_rp():
    rp = _lib.RolloutParams()
    rp.horizon, rp.max_episode_steps, rp.auto_reset, rp.random_policy = 1, 0, 0, 0
    return rp


def _rollout_call(entry, state_ptrs, n, T, p, rp, actions, act_dtype, extra=()):
    """One call of a rollout entry point with records on -> (records dict, stats [6], episode buffers)."""
    dev = "cuda"
    ep = dict(ep_step=torch.zeros(n, dtype=torch.int32, device=dev), ep_return=torch.zeros(n, dtype=torch.float32, device=dev),
              ep_index=torch.zeros(n, dtype=torch.int32, device=dev))
    rec = dict(observations=torch.empty((T, n, 4), dtype=torch.float32, device=dev),
               next_observations=torch.empty((T, n, 4), dtype=torch.float32, device=dev),
               actions=torch.empty((T, n), dtype=act_dtype, device=dev), rewards=torch.empty((T, n), dtype=torch.float32, device=dev),
               dones=torch.empty((T, n), dtype=torch.uint8, device=dev), timeouts=torch.empty((T, n), dtype=torch.uint8, device=dev))
    stats = torch.zeros(6, dtype=torch.float64, device=dev)
    ptrs = [rec[k].data_ptr() for k in ("observations", "next_observations", "actions", "rewards", "dones", "timeouts")]
    rc = getattr(_lib.lib, entry)(*state_ptrs, ep["ep_step"].data_ptr(), ep["ep_return"].data_ptr(), ep["ep_index"].data_ptr(),
                                  actions.data_ptr() if actions is not None else None, *ptrs, stats.data_ptr(), n, ctypes.byref(p),
                                  ctypes.byref(rp), *extra, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, f"{entry} returned {rc}"
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in rec.items()}, stats.cpu().numpy(), {k: v.cpu().numpy() for k, v in ep.items()}


def cartpole_ref_f32_step(p, st32, act, continuous, noise=None):
    """emei_cartpole_rollout_ref_f32, one teacher-forced step per row -> (state, next_obs, reward, done) as numpy."""
    n = st32.shape[0]
    state = torch.as_tensor(np.ascontiguousarray(st32, dtype=np.float32)).cuda()
    a, p.action_kind = _action_array(np.asarray(act).reshape(1, n), continuous)
    z = ctypes.byref(noise) if noise is not None else None
    rec, _, _ = _rollout_call("emei_cartpole_rollout_ref_f32", [state.data_ptr()], n, 1, p, _one_step_rp(), a, a.dtype, extra=(z,))
    assert np.array_equal(rec["observations"][0][:, [0, 2, 3]], st32[:, [0, 2, 3]])
    return state.cpu().numpy(), rec["next_observations"][0], rec["rewards"][0], rec["dones"][0].astype(bool)


def _noise_params(seed, step, env_offset=0):
    z = _lib.NoiseParams()
    for j in range(4):
        z.sigma[j] = SIG[j]
    z.seed, z.step, z.env_offset = seed, step, env_offset
    return z


def _frac(err, tol):
    return float((err / tol).max()) if err.size else 0.0


# ================================================================================================
# cart-pole balancing / swing-up (z = NULL: the C ABI only)
# ================================================================================================
@pytest.mark.parametrize("kind", list(CARTPOLE))
@pytest.mark.parametrize("fr", (1, 4))
def test_cartpole_rollout_ref_f32_golden_and_any_angle(golden, kind, fr):
    """The golden vectors' states (unwrapped swing-up angles of hundreds of radians at freq_rate 4: the inputs of
    test_cartpole_step_f32_identical_inputs_any_angle), rounded to float32 and fed to both sides: state and reward at 1.0 x
    the envelope, flags exact off the 1e-4 bands -- the bar of the lean kernel on identical inputs."""
    g = golden("cartpole")
    tag = f"{kind}_fr{fr}"
    st32, act = g[tag + "_state"].astype(np.float32), g[tag + "_action"]
    cont = kind.startswith("continuous")
    cp = O.cartpole_params(kind)
    ref = O.cartpole_step_f64ref(st32.astype(np.float64), O.cartpole_force(act, cont, cp), 0.02, fr, cp)
    p = _env_params(CARTPOLE[kind](freq_rate=fr, num_envs=1, dtype=torch.float32))
    state, nxt, rew, done = cartpole_ref_f32_step(p, st32, act, cont)
    assert np.array_equal(state, nxt)  # the cart-pole's observation is its state
    env_tol = 1e-6 + 1e-5 * np.abs(ref)
    f_state = _frac(np.abs(state - ref), env_tol)
    ref_rew = O.cartpole_reward(kind, ref)[:, 0]
    f_rew = _frac(np.abs(rew - ref_rew), 1e-6 + 1e-5 * np.abs(ref_rew))
    print(f"[envelope] cartpole {tag}: state {f_state:.3g} reward {f_rew:.3g}")
    assert f_state <= 1.0 and f_rew <= 1.0
    near = (np.abs(np.abs(ref[:, 0]) - cp.x_threshold) < 1e-4) | (np.abs(np.abs(ref[:, 2]) - cp.theta_threshold_radians) < 1e-4)
    assert np.array_equal(done[~near], O.cartpole_terminal(kind, ref, cp)[:, 0][~near])


# ================================================================================================
# analytic inverted pendulum: z = NULL, noise through the rollout, noise through the env's step
# ================================================================================================
@functools.lru_cache(maxsize=None)
def _c1_rows(kind, fr):
    """SURVEY 8(d) C1, as test_c1_protocol_ip_f32_teacher_forced_200_steps: 4096 envs, 200 un-reset oracle steps
    -> (float32 rows [200 * 4096, 4], ctrl [200 * 4096, 1])."""
    n, T = 4096, 200
    rng = np.random.default_rng(1001)
    st = rng.uniform(-1, 1, size=(n, 4)) * np.array([1.9, np.pi, 5.0, 8.0])
    acts = rng.uniform(-3, 3, size=(T, n, 1)).astype(np.float32)
    p = O.InvertedPendulumParams()
    ins = []
    for t in range(T):
        ins.append(st)
        st, _ = O.ip_step(st, acts[t].astype(np.float64), 0.02, fr, kind.endswith("swingup"), p)
    s32 = np.concatenate(ins).astype(np.float32)
    assert np.isfinite(s32).all()
    return s32, acts.reshape(T * n, 1)


def ip_assert_f32_step(kind, fr, s32, state, obs, rew, done, ref_state, ref_obs, label):
    """The bar of test_c1_protocol_ip_f32_teacher_forced_200_steps: 1.0 x the envelope; at freq_rate > 1 plus half an
    ulp32 of the variable per sub-step (a float32 value held between the sub-steps of the lean kernel); the wrapped
    observation angle on the circle; the reward at 1.0 x; flags exact off the 1e-4 bands (< 1 % of the rows)."""
    p = O.InvertedPendulumParams()
    err = np.abs(state.astype(np.float64) - ref_state)
    strict = 1e-6 + 1e-5 * np.abs(ref_state)
    tol = strict
    if fr > 1:
        big = np.maximum(np.abs(s32.astype(np.float64)), np.abs(ref_state)).astype(np.float32)
        tol = tol + fr * 0.5 * np.spacing(big).astype(np.float64)
    o = obs.astype(np.float64)
    dth = np.abs((o[:, 1] - ref_obs[:, 1] + np.pi) % (2 * np.pi) - np.pi)
    ref_rew = O.ip_reward(kind, ref_obs).reshape(-1)
    f_rew = _frac(np.abs(rew.astype(np.float64) - ref_rew), 1e-6 + 1e-5 * np.abs(ref_rew))
    print(f"[envelope] {label}: state {_frac(err, tol):.3g} (strict {_frac(err, strict):.3g}) "
          f"obs angle {_frac(dth, 1e-6 + 1e-5 * np.abs(ref_state[:, 1])):.3g} reward {f_rew:.3g}")
    assert _frac(err, tol) <= 1.0, f"{label}: worst fraction of the envelope {_frac(err, tol)}"
    assert np.all(dth <= 1e-6 + 1e-5 * np.abs(ref_state[:, 1]))
    assert np.all((o[:, 1] >= -np.pi - 1e-6) & (o[:, 1] <= np.pi + 1e-6))
    assert np.all(np.abs(o[:, [0, 2, 3]] - ref_obs[:, [0, 2, 3]]) <= tol[:, [0, 2, 3]])
    assert f_rew <= 1.0
    ref_done = O.ip_terminal(kind, ref_obs, p).reshape(-1)
    cy = np.cos(ref_obs[:, 1])
    near = np.abs(np.abs(ref_obs[:, 0]) - 2.0) < 1e-4
    if kind == "ip_rebound_balancing":
        near = np.abs(cy - 0.9) < 1e-4
    elif kind == "ip_boundary_balancing":
        near |= np.abs(cy) < 1e-4
    elif kind == "ip_rebound_swingup":
        near[:] = False
    assert np.array_equal(done.reshape(-1)[~near], ref_done[~near]) and near.mean() < 0.01


def _ip_case(rows, kind, fr):
    if rows == "c1":
        return _c1_rows(kind, fr)
    st, act = ip_inputs(4001, 4096)  # with its x30 unwrapped angles (up to 94 rad) and its rows at the rails
    return st.astype(np.float32), act  # ctrl beyond ctrlrange: clamped like mj_step, on both sides


@pytest.mark.parametrize("kind", list(IP))
@pytest.mark.parametrize("fr", (1, 4))
@pytest.mark.parametrize("rows", ("ip_inputs", "c1"))
@pytest.mark.parametrize("route", ("rollout_ref", "rollout_ref_noise", "env_step_noise"))
def test_ip_f32_reference_arithmetic_vs_oracle(kind, fr, rows, route):
    """All four IP variants, freq_rate 1 and 4, on ip_inputs (with its unwrapped angles) and on the 819,200 C1 rows in
    ONE launch: emei_cartpole_rollout_ref_f32 without noise (C ABI only), with noise, and emei_ip_step_noisy_f32 through
    an env built with obs_noise_params -- each against the float64 oracle from the identical float32 rows, the noisy
    routes with the Philox mirror's draws."""
    s32, act = _ip_case(rows, kind, fr)
    n = s32.shape[0]
    p = O.InvertedPendulumParams()
    ctrl = np.clip(act.astype(np.float64), p.ctrl_low, p.ctrl_high)
    swing = kind.endswith("swingup")
    seed, step = _noise_seed(11), 0
    z = P.obs_noise(n, 4, SIG, seed, step, fr) if route != "rollout_ref" else None
    ref_state, ref_obs = O.ip_step(s32.astype(np.float64), ctrl, 0.02, fr, swing, p, libm=(rows != "c1"), noise=z)
    if route == "env_step_noise":
        env = E.make(IP[kind], freq_rate=fr, num_envs=n, dtype=torch.float32, obs_noise_params=(0.01, 0.03))
        env.reset(seed=11)
        env.state = s32
        obs, rew, done, _, _ = env.step(act)
        state, obs, rew, done = env.state.cpu().numpy(), obs.cpu().numpy(), rew.cpu().numpy()[:, 0], done.cpu().numpy()[:, 0]
    else:
        pp = _env_params(E.make(IP[kind], freq_rate=fr, num_envs=1, dtype=torch.float32))
        noise = _noise_params(seed, step) if z is not None else None
        state, obs, rew, done = cartpole_ref_f32_step(pp, s32, act, True, noise)
    ip_assert_f32_step(kind, fr, s32, state, obs, rew, done, ref_state, ref_obs, f"{kind} fr{fr} {rows} {route}")
    if z is not None:  # the noise is really there
        clean, _ = O.ip_step(s32.astype(np.float64), ctrl, 0.02, fr, swing, p)
        assert (state[:, 2] - clean[:, 2]).std() > 0.5 * SIG[2]


# ================================================================================================
# charged ball (emei_charged_ball_rollout_ref_f32: the C ABI only)
# ================================================================================================
def charged_ball_ref_f32_step(p, on0, ci32, fr32, act, continuous):
    n = on0.shape[0]
    on = torch.as_tensor(on0.astype(np.uint8)).cuda()
    ci = torch.as_tensor(np.ascontiguousarray(ci32, dtype=np.float32)).cuda()
    fr = torch.as_tensor(np.ascontiguousarray(fr32, dtype=np.float32)).cuda()
    a, p.action_kind = _action_array(np.asarray(act).reshape(1, n), continuous)
    rec, _, _ = _rollout_call("emei_charged_ball_rollout_ref_f32", [on.data_ptr(), ci.data_ptr(), fr.data_ptr()], n, 1, p,
                              _one_step_rp(), a, a.dtype)
    got = dict(on_circle=on.cpu().numpy(), circle_state=ci.cpu().numpy(), free_state=fr.cpu().numpy())
    assert np.array_equal(rec["next_observations"][0], got["free_state"]) and not rec["dones"].any()
    return got, rec["rewards"][0]


def _cb_params(fr, cont):
    env_id = "ContinuousChargedBallCentering-v0" if cont else "ChargedBallCentering-v0"
    return _env_params(E.make(env_id, freq_rate=fr, num_envs=1, dtype=torch.float32))


@pytest.mark.parametrize("tag", ("disc_fr1", "disc_fr3", "cont_fr1", "cont_fr3"))
def test_charged_ball_rollout_ref_f32_teacher_forced(golden, tag):
    """Every step of the executed-reference trajectories (golden), teacher-forced from the float32-rounded states:
    cb_assert_f32_step's bar (1.0 x the envelope, flags exact off the thresholds, masks < 1 % of the rows)."""
    c = golden("charged_ball")
    fr, cont = int(tag[-1]), tag.startswith("cont")
    on, ci, fre, act = c[tag + "_on"], c[tag + "_circle"], c[tag + "_free"], c[tag + "_action"]
    T, n = act.shape[0], on.shape[1]
    on0 = on[:-1].reshape(-1)
    ci32, fr32 = ci[:-1].reshape(-1, 2).astype(np.float32), fre[:-1].reshape(-1, 4).astype(np.float32)
    cp = O.ChargedBallParams()
    a = act.reshape(T * n, 1) if cont else act.reshape(-1)
    Ef = O.charged_ball_force(a, cont, cp)
    r_on, r_ci, r_fr, near = cb_substep_trace(on0, ci32.astype(np.float64), fr32.astype(np.float64), Ef, fr, cp, f32_force=cont)
    got, rew = charged_ball_ref_f32_step(_cb_params(fr, cont), on0, ci32, fr32, a, cont)
    ok = (got["on_circle"].astype(bool) == r_on) & ~near
    th = np.maximum(np.abs(r_ci[:, 0]), np.abs(ci32[:, 0]))  # cb_assert_f32_step's representation term of the float32 angle
    rep = (np.spacing(th.astype(np.float32)).astype(np.float64) * (1.0 + np.abs(r_ci[:, 1])))[:, None] * (on0 | r_on)[:, None]
    err = np.abs(got["free_state"] - r_fr)[ok]
    print(f"[envelope] charged ball {tag}: free {_frac(err, (1e-6 + 1e-5 * np.abs(r_fr) + rep)[ok]):.3g} "
          f"(without the angle's representation term {_frac(err, (1e-6 + 1e-5 * np.abs(r_fr))[ok]):.3g})")
    ok_rows = cb_assert_f32_step(got, on0, ci32.astype(np.float64), r_on, r_ci, r_fr, near)
    assert near.mean() < 0.01 and ok_rows.mean() > 0.99
    ref_rew = O.charged_ball_reward(r_fr, cp).reshape(-1)
    assert within32(rew[ok_rows], ref_rew[ok_rows]).all()


def test_charged_ball_rollout_ref_f32_landing():
    """free_to_circle at EVERY position of the ring (the rows of test_charged_ball_f32_landing_vs_oracle), including x ~ +-r
    where asin(x / (scale r + 1e-8)) is ill conditioned and y ~ 0 where float32 drops the 1e-8."""
    n = 1 << 16
    rng = np.random.default_rng(77)
    ang = rng.uniform(0, 2 * np.pi, n)
    ang[: n // 4] = rng.choice([0.5 * np.pi, 1.5 * np.pi], n // 4) + rng.normal(0, 2e-3, n // 4)  # |x| ~ r
    ang[n // 4 : n // 2] = rng.choice([0.0, np.pi], n // 4) + rng.normal(0, 2e-3, n // 4)          # x ~ 0
    rad = rng.uniform(0.97, 0.9999, n)
    pos = np.stack([rad * np.sin(ang), rad * np.cos(ang)], axis=1)
    vdir = ang + rng.uniform(-1.2, 1.2, n)
    speed = rng.uniform(2.5, 6.0, n)
    vel = np.stack([speed * np.sin(vdir), speed * np.cos(vdir)], axis=1)
    fr32 = np.concatenate([pos, vel], axis=1).astype(np.float32)
    on0 = np.zeros(n, dtype=bool)
    ci32 = np.zeros((n, 2), dtype=np.float32)
    act = rng.integers(0, 2, size=n)
    cp = O.ChargedBallParams()
    r_on, r_ci, r_fr, near = cb_substep_trace(on0, ci32.astype(np.float64), fr32.astype(np.float64), O.charged_ball_force(act, False, cp), 1, cp)
    got, _ = charged_ball_ref_f32_step(_cb_params(1, False), on0, ci32, fr32, act, False)
    oc = (got["on_circle"].astype(bool) == r_on) & ~near & r_on
    print(f"[envelope] charged ball landing: circle {_frac(np.abs(got['circle_state'] - r_ci)[oc], (1e-6 + 1e-5 * np.abs(r_ci))[oc]):.3g}")
    ok_rows = cb_assert_f32_step(got, on0, ci32.astype(np.float64), r_on, r_ci, r_fr, near)
    assert 0.3 < r_on.mean() < 1.0 and (ok_rows & r_on).sum() > 10000 and near.mean() < 0.01


# ================================================================================================
# the bookkeeping of the two C-ABI-only entry points: T = 300, random policy, auto-reset, TimeLimit
# ================================================================================================
def _check_bookkeeping(rec, stats, ep, term, max_steps, reset_rows, label):
    """records vs the restated loop (oracle/rollout_oracle.py): dones / timeouts, the observation chain with the reset
    rows of every finished episode, the episode buffers and the six statistics against sums of the records."""
    T, n = rec["rewards"].shape
    ep_step, ep_ret, ep_idx = np.zeros(n, np.int64), np.zeros(n, np.float32), np.zeros(n, np.int64)
    fin, fin_ret, fin_len = 0, 0.0, 0
    for t in range(T):
        done, trunc, ep_step, ep_ret = RO.bookkeeping(term[t], max_steps, ep_step, ep_ret, rec["rewards"][t])
        assert np.array_equal(rec["dones"][t].astype(bool), done) and np.array_equal(rec["timeouts"][t].astype(bool), trunc), f"{label} step {t}"
        idx = np.nonzero(done)[0]
        fin += idx.size
        fin_ret += float(ep_ret[idx].astype(np.float64).sum())
        fin_len += int(ep_step[idx].sum())
        ep_idx[idx] += 1
        expect = rec["next_observations"][t].copy()
        if idx.size:
            expect[idx] = reset_rows(idx, ep_idx[idx])
        ep_step[idx], ep_ret[idx] = 0, 0.0
        if t + 1 < T:
            assert np.allclose(rec["observations"][t + 1], expect, rtol=0, atol=1e-7), f"{label}: observation chain at step {t + 1}"
    assert fin > 0 and rec["timeouts"].any()
    assert np.array_equal(ep["ep_step"], ep_step) and np.array_equal(ep["ep_index"], ep_idx) and np.array_equal(ep["ep_return"], ep_ret)
    rs = float(rec["rewards"].astype(np.float64).sum())
    assert abs(stats[0] - rs) <= 1e-9 * max(1.0, abs(rs))
    assert stats[1] == int(term.sum()) and stats[2] == int(rec["timeouts"].sum()) and stats[3] == fin
    assert abs(stats[4] - fin_ret) <= 1e-9 * max(1.0, abs(fin_ret)) and stats[5] == fin_len


def _random_rp(T, max_steps, seed, env_offset, init_kind, pi_col=-1, lo=-1.0, hi=1.0):
    rp = _lib.RolloutParams()
    rp.horizon, rp.max_episode_steps, rp.auto_reset, rp.random_policy = T, max_steps, 1, 1
    rp.init_kind, rp.init_pi_column, rp.init_low, rp.init_high = init_kind, pi_col, -0.05, 0.05
    rp.seed_reset, rp.seed_action = RO.rollout_seeds(seed)
    rp.env_offset, rp.t0, rp.action_low, rp.action_high = env_offset, 0, lo, hi
    return rp


@pytest.mark.parametrize("env_id,fr,max_steps", (("CartPoleSwingUp-v0", 4, 40), ("ReboundInvertedPendulumSwingUp-v0", 2, 60)))
def test_cartpole_rollout_ref_f32_bookkeeping(env_id, fr, max_steps):
    """emei_cartpole_rollout_ref_f32 without noise over T = 300 steps: random actions = the mirror, in-kernel resets =
    P.init_uniform / P.init_gaussian in float32, records = the restated loop, statistics = sums of the records; the cart-pole's
    transitions against the oracle teacher-forced from the recorded observation (its observation is its state)."""
    n, T, seed = 512, 300, 17
    env = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    p = _env_params(env)
    ip = "Pendulum" in env_id
    cont = ip
    env.reset(seed=seed)
    state = env.state.clone()
    rec0 = np.ascontiguousarray(state.cpu().numpy())
    if ip:
        mean, sigma = env._init_tables()
        rp = _random_rp(T, max_steps, seed, 0, 1, lo=float(env.action_space.low[0]), hi=float(env.action_space.high[0]))
        for j in range(4):
            rp.init_mean[j], rp.init_sigma[j] = mean[j], sigma[j]
    else:
        rp = _random_rp(T, max_steps, seed, 0, 0, pi_col=2)
    p.action_kind = _lib.ACTION_CONTINUOUS_F32 if cont else _lib.ACTION_DISCRETE_U8
    rec, stats, ep = _rollout_call("emei_cartpole_rollout_ref_f32", [state.data_ptr()], n, T, p, rp, None,
                                   torch.float32 if cont else torch.uint8, extra=(None,))
    lo, hi = (rp.action_low, rp.action_high) if cont else (-1.0, 1.0)
    assert np.array_equal(rec["actions"], RO.random_actions(rp.seed_action, n, 0, T, cont, lo, hi))
    assert np.array_equal(rec["observations"][0][:, [0, 2, 3]], rec0[:, [0, 2, 3]])

    def reset_rows(idx, ep_idx):
        out = np.empty((idx.size, 4), np.float32)
        for e in np.unique(ep_idx):
            s = (rp.seed_reset + int(e) * RO.RESET_STRIDE) & RO.MASK64
            if ip:
                rows = P.init_gaussian(n, 4, mean, sigma, s, dtype=np.float32)
                rows[:, 1] = O.ip_wrap_angle(rows[:, 1].astype(np.float64)).astype(np.float32)  # the recorded observation
            else:
                rows = P.init_uniform(n, 4, -0.05, 0.05, 2, s, dtype=np.float32)
            out[ep_idx == e] = rows[idx[ep_idx == e]]
        return out

    if ip:
        term = np.zeros((T, n), dtype=bool)  # Rebound swing-up terminates on non-finite states only (inverted_pendulum.py:139-146)
        assert not rec["dones"][rec["timeouts"] == 0].any()
    else:
        kind, cp = "swingup", O.cartpole_params("swingup")
        term = np.zeros((T, n), dtype=bool)
        worst = 0.0
        for t in range(T):
            obs = rec["observations"][t].astype(np.float64)
            ref = O.cartpole_step_f64ref(obs, O.cartpole_force(rec["actions"][t], False, cp), 0.02, fr, cp)
            worst = max(worst, _frac(np.abs(rec["next_observations"][t] - ref), 1e-6 + 1e-5 * np.abs(ref)))
            term[t] = O.cartpole_terminal(kind, rec["next_observations"][t].astype(np.float64), cp)[:, 0]
            near = np.abs(np.abs(ref[:, 0]) - cp.x_threshold) < 1e-4
            assert np.array_equal(term[t][~near], O.cartpole_terminal(kind, ref, cp)[:, 0][~near])
        print(f"[envelope] cartpole rollout_ref_f32 T={T}: {worst:.3g}")
        assert worst <= 1.0
        assert (rec["dones"] & ~rec["timeouts"]).any()  # both ways of ending an episode
    _check_bookkeeping(rec, stats, ep, term, max_steps, reset_rows, env_id)


def test_charged_ball_rollout_ref_f32_bookkeeping():
    """emei_charged_ball_rollout_ref_f32 over T = 300 steps with the random policy and the TimeLimit: actions = the mirror,
    in-kernel resets = P.init_charged_ball in float32, records = the restated loop, statistics = sums of the records."""
    n, T, seed, max_steps = 512, 300, 19, 70
    env = E.make("ChargedBallCentering-v0", num_envs=n, dtype=torch.float32, freq_rate=2)
    p = _env_params(env)
    env.reset(seed=seed)
    st = {k: v.clone() for k, v in env.state.items()}
    rp = _random_rp(T, max_steps, seed, 0, 0)
    p.action_kind = _lib.ACTION_DISCRETE_U8
    rec, stats, ep = _rollout_call("emei_charged_ball_rollout_ref_f32", [st["on_circle"].data_ptr(), st["circle_state"].data_ptr(),
                                   st["free_state"].data_ptr()], n, T, p, rp, None, torch.uint8)
    assert np.array_equal(rec["actions"], RO.random_actions(rp.seed_action, n, 0, T, False))
    assert 0.45 < rec["actions"].mean() < 0.55

    def reset_rows(idx, ep_idx):
        out = np.empty((idx.size, 4), np.float32)
        for e in np.unique(ep_idx):
            s = (rp.seed_reset + int(e) * RO.RESET_STRIDE) & RO.MASK64
            _, _, free = P.init_charged_ball(n, 1.0, s, dtype=np.float32)
            out[ep_idx == e] = free[idx[ep_idx == e]]
        return out

    assert not rec["dones"][rec["timeouts"] == 0].any()  # the charged ball never terminates (charged_ball.py:110-111)
    _check_bookkeeping(rec, stats, ep, np.zeros((T, n), dtype=bool), max_steps, reset_rows, "charged ball")
    # the reset rows' circle state: P.init_charged_ball bit for bit (final state of every env that was reset in the last step)
    last = np.nonzero(rec["dones"][-1])[0]
    if last.size:
        e_idx = ep["ep_index"][last]
        for e in np.unique(e_idx):
            s = (rp.seed_reset + int(e) * RO.RESET_STRIDE) & RO.MASK64
            _, circle, _ = P.init_charged_ball(n, 1.0, s, dtype=np.float32)
            rows = last[e_idx == e]
            assert np.array_equal(st["circle_state"].cpu().numpy()[rows], circle[rows])


# ================================================================================================
# the counter streams past their first Philox block
# ================================================================================================
STREAM_ENVS = (
    ("CartPoleSwingUp-v0", torch.float32),                     # rollout_f32_kernel, Discrete(2)
    ("CartPoleSwingUp-v0", torch.float64),                     # rollout_ref_kernel, Discrete(2)
    ("ContinuousCartPoleSwingUp-v0", torch.float32),           # rollout_f32_kernel, Box
    ("ContinuousCartPoleSwingUp-v0", torch.float64),           # rollout_ref_kernel, Box
    ("ChargedBallCentering-v0", torch.float32),                # rollout_f32_kernel (charged ball), Discrete(2)
    ("ContinuousChargedBallCentering-v0", torch.float64),      # rollout_ref_kernel (charged ball), Box
)


@pytest.mark.parametrize("env_id,dtype", STREAM_ENVS)
def test_rollout_action_streams_cross_words_blocks_and_env_hi(env_id, dtype):
    """The random policy's actions, bit for bit against RO.random_actions, in launches that start mid-word (t0 = 45) and
    split the horizon into odd lengths, for 140 steps -- crossing the discrete stream's word boundaries (32, 64, 96) and
    its Philox block boundary (128), and the continuous stream's block boundaries (tg & 3) -- for envs whose global ids
    cross 2^32 - 1 -> 2^32, so the counter's env_hi word is non-zero."""
    n, seed, off = 256, 23, (1 << 32) - 100
    env = E.make(env_id, num_envs=n, dtype=dtype, freq_rate=1, env_offset=off)
    env.reset(seed=seed)
    cont = len(env.action_space.shape) > 0
    got = [env.rollout(h, record=True, max_episode_steps=9)["actions"].cpu().numpy() for h in (45, 37, 51, 7)]
    got = np.concatenate(got, axis=0)
    _, seed_action = RO.rollout_seeds(seed)
    lo, hi = (float(env.action_space.low[0]), float(env.action_space.high[0])) if cont else (-1.0, 1.0)
    ref = RO.random_actions(seed_action, n, 0, got.shape[0], cont, lo, hi, env_offset=off)
    assert got.shape[0] == 140 and np.array_equal(got, ref)
    # env_hi is part of the counter: the envs past 2^32 do not draw the stream of their low 32 bits
    assert not np.array_equal(ref[:, 100:], RO.random_actions(seed_action, n - 100, 0, 140, cont, lo, hi, env_offset=0))


def test_rollout_ref_f32_noisy_action_stream_past_first_block():
    """rollout_ref_kernel in float32 (obs_noise_params) draws the same random-policy stream across the word, block and
    env_hi boundaries."""
    n, seed, off = 256, 29, (1 << 32) - 100
    env = E.make("BoundaryInvertedPendulumSwingUp-v0", num_envs=n, dtype=torch.float32, freq_rate=1, env_offset=off,
                 obs_noise_params=0.01)
    env.reset(seed=seed)
    got = np.concatenate([env.rollout(h, record=True, max_episode_steps=11)["actions"].cpu().numpy() for h in (45, 37, 51, 7)])
    _, seed_action = RO.rollout_seeds(seed)
    lo, hi = float(env.action_space.low[0]), float(env.action_space.high[0])
    assert np.array_equal(got, RO.random_actions(seed_action, n, 0, 140, True, lo, hi, env_offset=off))


@pytest.mark.parametrize("sfx", ("_f32", "_f64"))
def test_noise_stream_block_index_past_2_32(sfx):
    """add_state_noise keys sub-step g's pairs by Philox block 4 g + k; from g = 2^30 on the block index needs 33 bits and
    its high bits go to the purpose word (purpose | (blk >> 32) << 8).  From the rest state with zero control one
    sub-step of the Rebound balancing model does not move (sin 0 = 0), so the next state IS the noise: compared with
    P.obs_noise at the step counters 2^30 - 1 (blocks 2^32 - 4, 2^32 - 3) and 2^30 (blocks 2^32, 2^32 + 1), for envs whose
    ids cross 2^32.  The Philox words are the mirror's bit for bit; the device's Box-Muller takes sincospi(2 u) where the
    mirror takes cos(2 pi u), so the float64 draws agree to 1e-12 sigma (a wrong block is off by sigma) and a float32 draw
    to one ulp of its rounding."""
    n, off = 512, (1 << 32) - 256
    dt = torch.float32 if sfx == "_f32" else torch.float64
    p = _env_params(E.make(IP["ip_rebound_balancing"], freq_rate=1, num_envs=1, dtype=dt))
    p.action_kind = _lib.ACTION_CONTINUOUS_F32
    sigma = np.array([0.01, 0.02, 0.03, 0.04])
    seed = _noise_seed(7)
    f = getattr(_lib.lib, "emei_ip_step_noisy" + sfx)
    draws = []
    for step in ((1 << 30) - 1, 1 << 30):
        z = _noise_params(seed, step, off)
        for j in range(4):
            z.sigma[j] = sigma[j]
        s_in = torch.zeros((n, 4), dtype=dt, device="cuda")
        s_out, obs = torch.empty_like(s_in), torch.empty_like(s_in)
        act = torch.zeros(n, dtype=torch.float32, device="cuda")
        rew, done = torch.empty(n, dtype=dt, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
        rc = f(s_in.data_ptr(), s_out.data_ptr(), obs.data_ptr(), act.data_ptr(), rew.data_ptr(), done.data_ptr(), None, n,
               ctypes.byref(p), ctypes.byref(z), torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        ref = P.obs_noise(n, 4, sigma, seed, step, 1, env_offset=off)[0]
        got = s_out.cpu().numpy()
        if sfx == "_f64":  # cos(2 pi u) and cospi(2 u) differ by ~1e-16 absolute, also where the cosine is near 0
            assert np.all(np.abs(got - ref) <= 1e-12 * sigma), f"step {step}"
        else:
            assert np.all(np.abs(got.astype(np.float64) - ref) <= np.spacing(np.abs(ref).astype(np.float32))), f"step {step}"
        draws.append(ref)
    # the two sides of the boundary are different draws, and the high bits matter (without them block 2^32 aliases block 0)
    assert not np.array_equal(draws[0], draws[1])
    assert not np.array_equal(draws[1], P.obs_noise(n, 4, sigma, seed, 0, 1, env_offset=off)[0])
