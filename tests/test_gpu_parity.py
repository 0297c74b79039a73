"""GPU parity tests: the CUDA path (through the C ABI, via the env classes) against the CPU oracle
and the golden vectors of the executed reference.

Tolerances (BASELINE.json north_star):
  * float64 mode: 1e-12 (relative to max(1,|value|)); terminal flags / done counts bit-exact;
  * float32 mode: 1e-5 rel + 1e-6 abs per teacher-forced step; flags exact except where the state
    lies within tolerance of a threshold.
"""
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import emei_oracle as O
from oracle import philox as P

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore", category=RuntimeWarning)

import emei_b200 as E  # noqa: E402
from emei_b200.envs.classic_control import cartpole as CP  # noqa: E402
from emei_b200.envs.classic_control import charged_ball as CB  # noqa: E402

CARTPOLE = {
    "balancing": CP.CartPoleBalancingEnv,
    "swingup": CP.CartPoleSwingUpEnv,
    "continuous_balancing": CP.ContinuousCartPoleBalancingEnv,
    "continuous_swingup": CP.ContinuousCartPoleSwingUpEnv,
}


def close64(a, b, tol=1e-12):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    same_inf = np.isinf(a) & (a == b)
    return np.all(both_nan | same_inf | (np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))))


def within32(a, ref, scale=1.0):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(a - ref) <= scale * (1e-6 + 1e-5 * np.abs(ref))


# ================================================================================================
# cart-pole step
# ================================================================================================
@pytest.mark.parametrize("kind", list(CARTPOLE))
@pytest.mark.parametrize("fr", (1, 4))
def test_cartpole_step_f64_vs_golden(golden, kind, fr):
    g = golden("cartpole")
    tag = f"{kind}_fr{fr}"
    st, act = g[tag + "_state"], g[tag + "_action"]
    env = CARTPOLE[kind](freq_rate=fr, num_envs=st.shape[0], dtype=torch.float64)
    env.state = st
    env.reset_stats()
    obs, rew, done, trunc, info = env.step(act)
    assert trunc is False and info == {}
    assert obs.shape == (st.shape[0], 4) and rew.shape == (st.shape[0], 1) and done.shape == (st.shape[0], 1)
    assert done.dtype == torch.bool and obs.dtype == torch.float64
    obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
    ref = g[tag + "_next"]
    assert close64(obs, ref)
    n_exact = int((obs == ref).all(axis=1).sum())
    assert n_exact >= st.shape[0] - 1, f"only {n_exact}/{st.shape[0]} rows bit-identical"
    assert close64(rew, g[tag + "_reward"])
    assert np.array_equal(done, g[tag + "_done"])
    rs, dc = env.read_stats()
    assert dc == int(g[tag + "_done"].sum())
    assert abs(rs - g[tag + "_reward"].sum()) <= 1e-9


@pytest.mark.parametrize("kind", list(CARTPOLE))
@pytest.mark.parametrize("fr", (1, 4))
def test_cartpole_step_f32_vs_golden(golden, kind, fr):
    g = golden("cartpole")
    tag = f"{kind}_fr{fr}"
    st, act = g[tag + "_state"], g[tag + "_action"]
    env = CARTPOLE[kind](freq_rate=fr, num_envs=st.shape[0], dtype=torch.float32)
    env.state = st  # cast to float32 by the engine
    obs, rew, done, _, _ = env.step(act)
    obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
    ref = g[tag + "_next"]
    small = np.abs(st[:, 2]) <= 4 * np.pi
    ok = within32(obs, ref)
    assert ok[small].all(), f"worst envelope fraction {(np.abs(obs - ref) / (1e-6 + 1e-5 * np.abs(ref)))[small].max()}"
    # outside the working range the float32 quantisation of theta itself bounds the agreement
    quant = np.spacing(np.abs(st[:, 2]).astype(np.float32)).astype(np.float64)[:, None] * 40.0 * 0.02 * fr
    assert np.all(np.abs(obs - ref) <= (1e-6 + 1e-5 * np.abs(ref)) + quant)
    ok_r = np.abs(rew - g[tag + "_reward"]) <= 1e-6 + 1e-5 * np.abs(g[tag + "_reward"]) + quant  # cos(theta): same theta quantisation
    assert ok_r.all() and within32(rew, g[tag + "_reward"])[small].all()
    p = O.cartpole_params(kind)
    near = (np.abs(np.abs(ref[:, 0]) - p.x_threshold) < 1e-4) | (np.abs(np.abs(ref[:, 2]) - p.theta_threshold_radians) < 1e-4)
    assert np.array_equal(done[~near], g[tag + "_done"][~near])


@pytest.mark.parametrize("kind", ("swingup", "continuous_swingup"))
def test_cartpole_step_f32_identical_inputs_any_angle(golden, kind):
    """Same float32 inputs on both sides (oracle in reference arithmetic): strict tolerance for ALL
    angles, including the large unwrapped ones."""
    g = golden("cartpole")
    tag = f"{kind}_fr4"
    st32 = g[tag + "_state"].astype(np.float32)
    act = g[tag + "_action"]
    p = O.cartpole_params(kind)
    ref = O.cartpole_step_f64ref(st32.astype(np.float64), O.cartpole_force(act, kind.startswith("continuous"), p), 0.02, 4, p)
    env = CARTPOLE[kind](freq_rate=4, num_envs=st32.shape[0], dtype=torch.float32)
    env.state = st32
    obs = env.step(act)[0].cpu().numpy()
    frac = np.abs(obs - ref) / (1e-6 + 1e-5 * np.abs(ref))
    assert frac.max() <= 1.0, f"worst envelope fraction {frac.max()}"


def test_cartpole_free_running_trajectory_f64(golden):
    """200 un-forced steps from the reference's reset(seed) states: float64 mode stays on the
    reference trajectory (1e-12 per step compounds to < 1e-9 here; rows are normally bit-identical)."""
    g = golden("cartpole")
    acts, traj = g["traj_swingup_fr4_action"], g["traj_swingup_fr4"]
    env = CP.CartPoleSwingUpEnv(freq_rate=4, num_envs=8, dtype=torch.float64)
    env.state = g["traj_swingup_fr4_init"]
    exact = 0
    for t in range(acts.shape[1]):
        obs, rew, done, _, _ = env.step(acts[:, t])
        o = obs.cpu().numpy()
        assert close64(o, traj[:, t, :4], 1e-9)
        exact += int((o == traj[:, t, :4]).all())
        assert close64(rew.cpu().numpy()[:, 0], traj[:, t, 4], 1e-9)
        assert np.array_equal(done.cpu().numpy()[:, 0], traj[:, t, 5].astype(bool))
    assert exact >= acts.shape[1] - 2, f"{exact}/{acts.shape[1]} steps bit-identical"


def test_cartpole_teacher_forced_f32_trajectory(golden):
    """The north-star protocol: reference states fed back every step, float32 engine."""
    g = golden("cartpole")
    acts, traj = g["traj_swingup_fr4_action"], g["traj_swingup_fr4"]
    env = CP.CartPoleSwingUpEnv(freq_rate=4, num_envs=8, dtype=torch.float32)
    prev = g["traj_swingup_fr4_init"]
    worst = 0.0
    for t in range(acts.shape[1]):
        env.state = prev
        obs = env.step(acts[:, t])[0].cpu().numpy()
        ref = traj[:, t, :4]
        # the un-reset reference trajectory winds theta up to hundreds of radians; casting that theta
        # to float32 (the engine dtype) is an INPUT error of ulp32(theta)/2 that the step propagates
        # (same allowance as test_cartpole_step_f32_vs_golden)
        quant = np.spacing(np.abs(prev[:, 2]).astype(np.float32)).astype(np.float64)[:, None] * 40.0 * 0.02 * 4
        worst = max(worst, (np.abs(obs - ref) / (1e-6 + 1e-5 * np.abs(ref) + quant)).max())
        prev = ref
    assert worst <= 1.0, f"worst envelope fraction {worst}"


def test_cartpole_discrete_action_dtypes_and_int(golden):
    g = golden("cartpole")
    st, act = g["swingup_fr1_state"], g["swingup_fr1_action"]
    outs = []
    for dt in (torch.uint8, torch.int32, torch.int64):
        env = CP.CartPoleSwingUpEnv(num_envs=st.shape[0], dtype=torch.float64)
        env.state = st
        outs.append(env.step(torch.as_tensor(act).to(dt))[0].cpu().numpy())
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[1], outs[2])
    env = CP.CartPoleSwingUpEnv(num_envs=1, dtype=torch.float64)
    env.state = st[:1]
    o = env.step(int(act[0]))[0].cpu().numpy()
    assert np.array_equal(o, outs[0][:1])
    with pytest.raises(AssertionError):
        env.step(torch.tensor([0.5]))
    env2 = CP.CartPoleSwingUpEnv(num_envs=1, dtype=torch.float64, validate_actions=True)
    env2.state = st[:1]
    with pytest.raises(AssertionError):
        env2.step(torch.tensor([3]))
    env3 = CP.CartPoleSwingUpEnv(num_envs=2)
    with pytest.raises(AssertionError):
        env3.step(torch.tensor([0, 1]))  # step before reset (base_control.py:67)


def test_cartpole_reset_freeze_unfreeze_and_liveness():
    """test/test_envs/test_classic_control/test_cartpole.py:14-35 (terminates eventually) +
    test/test_core.py:17-23 (frozen flag) + snapshot/restore semantics."""
    for cls in (CP.CartPoleBalancingEnv, CP.CartPoleSwingUpEnv):
        env = cls(num_envs=64)
        obs, info = env.reset(seed=1)
        assert obs.shape == (64, 4) and info == {}
        env.action_space.seed(0)
        ever_done = torch.zeros(64, dtype=torch.bool, device=obs.device)
        for _ in range(3000):
            o, r, term, trunc, _ = env.step(env.action_space.sample_batch(64))
            ever_done |= term[:, 0]
            if bool(ever_done.all()):
                break
        assert bool(ever_done.all())
    env = CP.CartPoleSwingUpEnv(num_envs=1000, freq_rate=2)
    env.reset(seed=3)
    a = env.action_space.sample_batch(1000)
    env.step(a)
    env.freeze()
    assert env.frozen
    s0 = env.state.clone()
    o1 = env.step(a)[0].clone()
    env.step(a)
    env.unfreeze()
    assert not env.frozen
    assert torch.equal(env.state, s0)
    assert torch.equal(env.step(a)[0], o1)  # deterministic replay from the snapshot
    fresh = CP.CartPoleSwingUpEnv(num_envs=4)
    with pytest.raises(RuntimeError):
        fresh.unfreeze()


def test_cartpole_init_state_philox_bit_exact_and_shard_invariant():
    env = CP.CartPoleSwingUpEnv(num_envs=4096, dtype=torch.float64)
    obs, _ = env.reset(seed=5)
    seed0 = (5 * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    host = P.init_uniform(4096, 4, -0.05, 0.05, 2, seed0)
    assert np.array_equal(obs.cpu().numpy(), host)
    # shard [1024, 2048) of the same global batch
    part = CP.CartPoleSwingUpEnv(num_envs=1024, dtype=torch.float64, env_offset=1024)
    pobs, _ = part.reset(seed=5)
    assert np.array_equal(pobs.cpu().numpy(), host[1024:2048])
    # distribution vs the reference's sampler (golden): moments only
    x = obs.cpu().numpy() - np.array([0, 0, np.pi, 0])
    assert np.all(np.abs(x) <= 0.05)
    assert np.allclose(x.mean(0), 0, atol=3e-3) and np.allclose(x.std(0), 0.1 / np.sqrt(12), atol=1e-3)
    e32 = CP.CartPoleBalancingEnv(num_envs=4096, dtype=torch.float32)
    o32, _ = e32.reset(seed=5)
    assert np.array_equal(o32.cpu().numpy(), P.init_uniform(4096, 4, -0.05, 0.05, -1, seed0, dtype=np.float32))
    o32b, _ = e32.reset()  # second reset draws a fresh stream
    assert not torch.equal(o32, o32b)


def test_cartpole_get_batch_api_numpy_roundtrip(golden):
    g = golden("cartpole")
    for kind in ("balancing", "swingup"):
        tag = f"{kind}_fr1"
        env = CARTPOLE[kind](dtype=torch.float64)
        nxt = g[tag + "_next"]
        r = env.get_batch_reward(nxt)
        d = env.get_batch_terminal(nxt)
        assert isinstance(r, np.ndarray) and r.shape == (nxt.shape[0], 1) and d.dtype == np.bool_
        assert close64(r, g[tag + "_reward"]) and np.array_equal(d, g[tag + "_done"])
        rt, dt = env.get_batch_reward(torch.as_tensor(nxt)), env.get_batch_terminal(torch.as_tensor(nxt))
        assert isinstance(rt, torch.Tensor) and rt.is_cuda and dt.dtype == torch.bool
    # get_batch_next_obs: needs frozen (core.py:190-193); stateless one-step dynamics
    env = CP.CartPoleSwingUpEnv(freq_rate=4, dtype=torch.float64, num_envs=3)
    with pytest.raises(AssertionError):
        env.get_batch_next_obs(g["swingup_fr4_state"], action=g["swingup_fr4_action"])
    env.reset(seed=0)
    env.freeze()
    s_before = env.state.clone()
    nxt = env.get_batch_next_obs(g["swingup_fr4_state"], action=g["swingup_fr4_action"])
    assert close64(nxt, g["swingup_fr4_next"])
    assert torch.equal(env.state, s_before)


# ================================================================================================
# analytic inverted pendulum
# ================================================================================================
IP = {
    "ip_rebound_balancing": "ReboundInvertedPendulumBalancing-v0",
    "ip_boundary_balancing": "BoundaryInvertedPendulumBalancing-v0",
    "ip_rebound_swingup": "ReboundInvertedPendulumSwingUp-v0",
    "ip_boundary_swingup": "BoundaryInvertedPendulumSwingUp-v0",
}


def ip_inputs(seed, n):
    rng = np.random.default_rng(seed)
    st = rng.uniform(-1, 1, size=(n, 4)) * np.array([1.9, np.pi, 5.0, 8.0])  # SURVEY 8(d) C1
    st[: n // 8, 1] *= 30.0  # unwrapped angles
    st[n // 8 : n // 4, 0] = np.sign(st[n // 8 : n // 4, 0]) * rng.uniform(1.95, 2.05, n // 4 - n // 8)
    act = rng.uniform(-3.5, 3.5, size=(n, 1)).astype(np.float32)  # beyond ctrlrange: clamped like mj_step
    return st, act


@pytest.mark.parametrize("kind", list(IP))
@pytest.mark.parametrize("fr", (1, 3))
def test_ip_step_f64_vs_oracle(kind, fr):
    st, act = ip_inputs(1001, 4096)
    p = O.InvertedPendulumParams()
    ctrl = np.clip(act.astype(np.float64), p.ctrl_low, p.ctrl_high)
    ref_state, ref_obs = O.ip_step(st, ctrl, 0.02, fr, kind.endswith("swingup"), p, libm=True)
    env = E.make(IP[kind], freq_rate=fr, num_envs=4096, dtype=torch.float64)
    env.state = st
    obs, rew, done, _, _ = env.step(act)
    assert close64(env.state.cpu().numpy(), ref_state)
    o = obs.cpu().numpy()
    # wrapped angle: compare on the circle (a 1-ulp state difference can land on the other side of +-pi)
    dth = np.abs((o[:, 1] - ref_obs[:, 1] + np.pi) % (2 * np.pi) - np.pi)
    assert dth.max() <= 1e-12 and close64(o[:, [0, 2, 3]], ref_obs[:, [0, 2, 3]])
    assert np.all((o[:, 1] >= -np.pi) & (o[:, 1] < np.pi))
    assert close64(rew.cpu().numpy(), O.ip_reward(kind, ref_obs), 1e-11)
    ref_done = O.ip_terminal(kind, ref_obs, p)
    near = (np.abs(np.abs(ref_obs[:, 0]) - 2.0) < 1e-9) | (np.abs(np.cos(ref_obs[:, 1]) - 0.9) < 1e-9) | (np.abs(np.cos(ref_obs[:, 1])) < 1e-9)
    assert np.array_equal(done.cpu().numpy()[~near], ref_done[~near])
    assert 0 < ref_done.mean() < 1 or kind == "ip_rebound_swingup"


@pytest.mark.parametrize("kind", ("ip_boundary_swingup", "ip_boundary_balancing"))
def test_ip_step_f32_vs_oracle_identical_inputs(kind):
    st, act = ip_inputs(1002, 4096)
    st32 = st.astype(np.float32)
    p = O.InvertedPendulumParams()
    ctrl = np.clip(act.astype(np.float64), p.ctrl_low, p.ctrl_high)
    ref_state, ref_obs = O.ip_step(st32.astype(np.float64), ctrl, 0.02, 1, kind.endswith("swingup"), p)
    env = E.make(IP[kind], num_envs=4096, dtype=torch.float32)
    env.state = st32
    obs, rew, done, _, _ = env.step(act)
    assert within32(env.state.cpu().numpy(), ref_state).all()
    o = obs.cpu().numpy().astype(np.float64)
    dth = np.abs((o[:, 1] - ref_obs[:, 1] + np.pi) % (2 * np.pi) - np.pi)
    assert np.all(dth <= 1e-6 + 1e-5 * np.abs(ref_state[:, 1]))
    assert within32(rew.cpu().numpy(), O.ip_reward(kind, ref_obs), 2.0).all()
    ref_done = O.ip_terminal(kind, ref_obs, p)
    near = (np.abs(np.abs(ref_obs[:, 0]) - 2.0) < 1e-4) | (np.abs(np.cos(ref_obs[:, 1])) < 1e-4)
    assert np.array_equal(done.cpu().numpy()[~near], ref_done[~near])


@pytest.mark.parametrize("kind", list(IP))
@pytest.mark.parametrize("fr", (1, 4))
def test_c1_protocol_ip_f32_teacher_forced_200_steps(kind, fr):
    """SURVEY 8(d) C1: 4096 envs, states U(-1,1) x [1.9, pi, 5, 8], ctrl U(-3,3), 200 teacher-forced steps -- the
    reference (float64 oracle) trajectory is never reset and its state is fed back at every step; the float32 kernel
    steps from the float32-rounded reference state and must meet 1.0 x (1e-5 rel + 1e-6 abs) per step for ALL four
    variants and both freq_rates; flags exact except within 1e-4 of a threshold.  All 200 steps run as ONE batch of
    200 x 4096 envs (one launch of the TMA kernel with the separate observation output)."""
    n, T = 4096, 200
    rng = np.random.default_rng(1001)
    st = rng.uniform(-1, 1, size=(n, 4)) * np.array([1.9, np.pi, 5.0, 8.0])
    acts = rng.uniform(-3, 3, size=(T, n, 1)).astype(np.float32)
    p = O.InvertedPendulumParams()
    swing = kind.endswith("swingup")
    ins = []
    for t in range(T):
        ins.append(st)
        st, _ = O.ip_step(st, acts[t].astype(np.float64), 0.02, fr, swing, p)
    s32 = np.concatenate(ins).astype(np.float32)
    a_all = acts.reshape(T * n, 1)
    assert np.isfinite(s32).all()
    ref_state, ref_obs = O.ip_step(s32.astype(np.float64), a_all.astype(np.float64), 0.02, fr, swing, p)
    env = E.make(IP[kind], freq_rate=fr, num_envs=T * n, dtype=torch.float32)
    env.state = s32
    obs, rew, done, _, _ = env.step(a_all)
    err = np.abs(env.state.cpu().numpy().astype(np.float64) - ref_state)
    tol = 1e-6 + 1e-5 * np.abs(ref_state)
    if fr > 1:
        # The un-reset trajectories reach |omega| = 47 rad/s and accelerations of hundreds of m/s^2 (16 s of random
        # +-300 N on a 15 kg cart): a velocity that sweeps through 4 m/s within the step and ends near zero is held
        # in float32 between the sub-steps, and its grid there (ulp32(4) = 4.8e-7) is already half the ABSOLUTE
        # envelope.  What no float32 step can resolve is added: half an ulp of the variable per sub-step.  (A plain
        # float32 restatement of the reference is off by 129 envelopes on these rows; freq_rate = 1 is asserted strictly.)
        big = np.maximum(np.abs(s32.astype(np.float64)), np.abs(ref_state)).astype(np.float32)
        tol = tol + fr * 0.5 * np.spacing(big).astype(np.float64)
    frac = err / tol
    assert frac.max() <= 1.0, (f"worst fraction of the envelope {frac.max()} at step {np.argmax(frac.max(axis=1)) // n}; "
                               f"strict 1e-5/1e-6: {(err / (1e-6 + 1e-5 * np.abs(ref_state))).max()}")
    o = obs.cpu().numpy().astype(np.float64)
    dth = np.abs((o[:, 1] - ref_obs[:, 1] + np.pi) % (2 * np.pi) - np.pi)  # wrapped angle: compare on the circle
    assert np.all(dth <= 1e-6 + 1e-5 * np.abs(ref_state[:, 1]))
    assert np.all((o[:, 1] >= -np.pi - 1e-6) & (o[:, 1] <= np.pi + 1e-6))
    assert np.all(np.abs(o[:, [0, 2, 3]] - ref_obs[:, [0, 2, 3]]) <= tol[:, [0, 2, 3]])
    assert within32(rew.cpu().numpy(), O.ip_reward(kind, ref_obs)).all()
    ref_done = O.ip_terminal(kind, ref_obs, p)
    cy = np.cos(ref_obs[:, 1])
    near = np.abs(np.abs(ref_obs[:, 0]) - 2.0) < 1e-4
    if kind == "ip_rebound_balancing":
        near = np.abs(cy - 0.9) < 1e-4
    elif kind == "ip_boundary_balancing":
        near |= np.abs(cy) < 1e-4
    elif kind == "ip_rebound_swingup":
        near[:] = False
    assert np.array_equal(done.cpu().numpy()[~near], ref_done[~near]) and near.mean() < 0.01


def test_ip_reset_liveness_graph():
    """test/test_envs/test_mujoco/test_inverted_pendulum.py:14-62: Boundary variants and Rebound
    Balancing terminate eventually; Rebound SwingUp never terminates within 100 steps."""
    for kind, must_end in (("ip_boundary_swingup", True), ("ip_boundary_balancing", True), ("ip_rebound_balancing", True)):
        env = E.make(IP[kind], num_envs=32)
        obs, _ = env.reset(seed=2)
        assert obs.shape == (32, 4) and float(obs.abs().max()) < 0.05
        env.action_space.seed(1)
        ever = torch.zeros(32, dtype=torch.bool, device=obs.device)
        for _ in range(5000):
            ever |= env.step(env.action_space.sample_batch(32))[2][:, 0]
            if bool(ever.all()):
                break
        assert bool(ever.all()) == must_end
    env = E.make(IP["ip_rebound_swingup"], num_envs=32)
    env.reset(seed=2)
    for _ in range(101):
        assert not bool(env.step(env.action_space.sample_batch(32))[2].any())
    assert env.get_transition_graph().shape == (5, 4)


# ================================================================================================
# charged ball
# ================================================================================================
@pytest.mark.parametrize("tag", ("disc_fr1", "disc_fr3", "cont_fr1", "cont_fr3"))
def test_charged_ball_f64_teacher_forced_vs_golden(golden, tag):
    c = golden("charged_ball")
    fr, cont = int(tag[-1]), tag.startswith("cont")
    on, ci, fre, act = c[tag + "_on"], c[tag + "_circle"], c[tag + "_free"], c[tag + "_action"]
    T, n = act.shape[0], on.shape[1]
    # all T teacher-forced steps in ONE batch of T*n envs
    cls = CB.ContinuousChargedBallCenteringEnv if cont else CB.ChargedBallCenteringEnv
    env = cls(freq_rate=fr, num_envs=T * n, dtype=torch.float64)
    env.state = dict(on_circle=on[:-1].reshape(-1).astype(np.uint8), circle_state=ci[:-1].reshape(-1, 2), free_state=fre[:-1].reshape(-1, 4))
    a = act.reshape(T * n, 1) if cont else act.reshape(-1)
    obs, rew, done, _, _ = env.step(a)
    st = env.state
    got_on = st["on_circle"].cpu().numpy().astype(bool)
    ref_on = on[1:].reshape(-1)
    assert np.array_equal(got_on, ref_on)
    assert close64(st["free_state"].cpu().numpy(), fre[1:].reshape(-1, 4))
    # circle state is meaningful while on the circle (it is stale, but still carried, in flight)
    assert close64(st["circle_state"].cpu().numpy(), ci[1:].reshape(-1, 2), 1e-11)
    assert torch.equal(obs, st["free_state"])
    ref_rew = O.charged_ball_reward(fre[1:].reshape(-1, 4), O.ChargedBallParams())
    assert close64(rew.cpu().numpy(), ref_rew)
    assert not bool(done.any())


def cb_substep_trace(on, ci, fre, Ef, fr, p, f32_force=False):
    """The oracle's env step, one sub-step at a time (charged_ball.py:54-82), with the rows whose regime decision of
    some sub-step lies within tolerance of its threshold -- the ONLY rows where float32 flags may differ from float64:
      take-off  m w^2 r + sin(th) E < cos(th) m g     (:75)   margin relative to the terms' magnitude
      landing   x^2 + y^2 > r^2 + 0.001               (:64)   |x^2 + y^2 - (r^2 + 0.001)| < 1e-5
      landing direction: sign of `_angle_greater(v_angle, theta)` (:38-42,48-51) when the velocity is (anti)parallel to
      the position within 1e-4 rad.
    Returns (on, circle, free, near)."""
    import copy

    ps = copy.copy(p)
    ps.time_step = p.time_step / fr
    near = np.zeros(on.shape[0], dtype=bool)
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
    return on, ci, fre, near


def cb_assert_f32_step(got, on0, ci_in, ref_on, ref_ci, ref_fr, near):
    """float32 charged-ball step against the float64 oracle ON IDENTICAL float32 INPUTS, at the north star's bar:
    regime flags exact except on `near` rows; state within 1.0 x (1e-6 + 1e-5 |ref|) plus what float32 cannot
    represent: the stored angle is a float32, so (x, y, vx, vy) = r (sin, cos, w cos, -w sin)(theta) carry its
    half-ulp rounding, ulp32(theta) (1 + |w|) -- zero for the angles of a fresh episode, 2e-6 at |theta| = 30."""
    got_on = got["on_circle"].astype(bool)
    bad = (got_on != ref_on) & ~near
    assert not bad.any(), f"{bad.sum()} regime flags differ away from the take-off / landing thresholds"
    ok_rows = (got_on == ref_on) & ~near
    th = np.maximum(np.abs(ref_ci[:, 0]), np.abs(ci_in[:, 0]))
    rep = (np.spacing(th.astype(np.float32)).astype(np.float64) * (1.0 + np.abs(ref_ci[:, 1])))[:, None]
    fr_err = np.abs(got["free_state"].astype(np.float64) - ref_fr)
    fr_tol = 1e-6 + 1e-5 * np.abs(ref_fr) + rep * (on0 | ref_on)[:, None]
    worst = (fr_err / fr_tol)[ok_rows].max()
    assert worst <= 1.0, f"free state: worst fraction of the envelope {worst}"
    oc = ok_rows & ref_on  # the circle state is meaningful while on the ring
    ci_err = np.abs(got["circle_state"].astype(np.float64) - ref_ci)
    worst_c = (ci_err / (1e-6 + 1e-5 * np.abs(ref_ci)))[oc].max() if oc.any() else 0.0
    assert worst_c <= 1.0, f"circle state: worst fraction of the envelope {worst_c}"
    return ok_rows


@pytest.mark.parametrize("tag", ("disc_fr1", "disc_fr3", "cont_fr1", "cont_fr3"))
def test_charged_ball_f32_teacher_forced(golden, tag):
    """Every step of the executed-reference trajectories (golden), teacher-forced: float32 kernel vs float64 oracle from the
    SAME float32-rounded states, 1.0 x envelope, flags exact except within tolerance of a threshold."""
    c = golden("charged_ball")
    fr, cont = int(tag[-1]), tag.startswith("cont")
    on, ci, fre, act = c[tag + "_on"], c[tag + "_circle"], c[tag + "_free"], c[tag + "_action"]
    T, n = act.shape[0], on.shape[1]
    on0 = on[:-1].reshape(-1)
    ci32, fr32 = ci[:-1].reshape(-1, 2).astype(np.float32), fre[:-1].reshape(-1, 4).astype(np.float32)
    p = O.ChargedBallParams()
    a = act.reshape(T * n, 1) if cont else act.reshape(-1)
    Ef = O.charged_ball_force(a, cont, p)
    r_on, r_ci, r_fr, near = cb_substep_trace(on0, ci32.astype(np.float64), fr32.astype(np.float64), Ef, fr, p, f32_force=cont)
    cls = CB.ContinuousChargedBallCenteringEnv if cont else CB.ChargedBallCenteringEnv
    env = cls(freq_rate=fr, num_envs=T * n, dtype=torch.float32)
    env.state = dict(on_circle=on0.astype(np.uint8), circle_state=ci32, free_state=fr32)
    _, rew, _, _, _ = env.step(a)
    got = {k: v.cpu().numpy() for k, v in env.state.items()}
    ok_rows = cb_assert_f32_step(got, on0, ci32.astype(np.float64), r_on, r_ci, r_fr, near)
    assert near.mean() < 0.01 and ok_rows.mean() > 0.99  # the masks are the exception, not the test
    ref_rew = O.charged_ball_reward(r_fr, p)
    assert within32(rew.cpu().numpy()[ok_rows], ref_rew[ok_rows]).all()


def test_charged_ball_f32_landing_vs_oracle():
    """free_to_circle (charged_ball.py:44-52) in float32: balls in free flight just inside the ring, moving
    outwards, land in this step -- at EVERY position of the ring, including x ~ +-r where the reference's
    asin(x / (scale r + 1e-8)) is ill conditioned (the float32 path evaluates it as atan2 of a cancellation-free
    complement, charged_ball_f32.cuh).  (theta, omega) and the free state at 1.0 x the envelope; flags exact
    except within tolerance of the landing threshold."""
    n = 1 << 16
    rng = np.random.default_rng(77)
    ang = rng.uniform(0, 2 * np.pi, n)
    ang[: n // 4] = rng.choice([0.5 * np.pi, 1.5 * np.pi], n // 4) + rng.normal(0, 2e-3, n // 4)  # |x| ~ r
    ang[n // 4 : n // 2] = rng.choice([0.0, np.pi], n // 4) + rng.normal(0, 2e-3, n // 4)          # x ~ 0
    rad = rng.uniform(0.97, 0.9999, n)
    pos = np.stack([rad * np.sin(ang), rad * np.cos(ang)], axis=1)
    vdir = ang + rng.uniform(-1.2, 1.2, n)  # outward-ish
    speed = rng.uniform(2.5, 6.0, n)
    vel = np.stack([speed * np.sin(vdir), speed * np.cos(vdir)], axis=1)
    fr32 = np.concatenate([pos, vel], axis=1).astype(np.float32)
    on0 = np.zeros(n, dtype=bool)
    ci32 = np.zeros((n, 2), dtype=np.float32)
    act = rng.integers(0, 2, size=n)
    p = O.ChargedBallParams()
    r_on, r_ci, r_fr, near = cb_substep_trace(on0, ci32.astype(np.float64), fr32.astype(np.float64), O.charged_ball_force(act, False, p), 1, p)
    env = CB.ChargedBallCenteringEnv(num_envs=n, dtype=torch.float32)
    env.state = dict(on_circle=on0.astype(np.uint8), circle_state=ci32, free_state=fr32)
    env.step(act)
    got = {k: v.cpu().numpy() for k, v in env.state.items()}
    ok_rows = cb_assert_f32_step(got, on0, ci32.astype(np.float64), r_on, r_ci, r_fr, near)
    assert 0.3 < r_on.mean() < 1.0 and (ok_rows & r_on).sum() > 10000 and near.mean() < 0.01


def test_charged_ball_reset_and_rollout_stats():
    env = CB.ChargedBallCenteringEnv(num_envs=2048, dtype=torch.float64)
    obs, _ = env.reset(seed=9)
    seed0 = (9 * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    h_on, h_ci, h_fr = P.init_charged_ball(2048, 1.0, seed0)
    st = env.state
    assert np.array_equal(st["on_circle"].cpu().numpy(), h_on)
    assert np.array_equal(st["circle_state"].cpu().numpy(), h_ci)
    assert close64(st["free_state"].cpu().numpy(), h_fr, 1e-15)
    # 50-step rollout vs oracle, un-forced, float64
    p = O.ChargedBallParams()
    rng = np.random.default_rng(0)
    on, ci, fre = h_on.astype(bool), h_ci, st["free_state"].cpu().numpy()
    env.reset_stats()
    total = 0.0
    for t in range(50):
        a = rng.integers(0, 2, size=2048)
        obs, rew, done, _, _ = env.step(a)
        on, ci, fre = O.charged_ball_step(on, ci, fre, O.charged_ball_force(a, False, p), 1, p)
        total += O.charged_ball_reward(fre, p).sum()
    assert np.array_equal(env.state["on_circle"].cpu().numpy().astype(bool), on)
    assert close64(obs.cpu().numpy(), fre, 1e-9)
    rs, dc = env.read_stats()
    assert dc == 0 and abs(rs - total) < 1e-6 * abs(total)
    # freeze / unfreeze restores all three arrays
    env.freeze()
    snap = {k: v.clone() for k, v in env.state.items()}
    env.step(rng.integers(0, 2, size=2048))
    env.unfreeze()
    for k in snap:
        assert torch.equal(env.state[k], snap[k])


# ================================================================================================
# scoring (get_batch_reward / get_batch_terminal)
# ================================================================================================
def test_hopper_scoring_f64_vs_golden(golden):
    g = golden("scoring")
    for T in (1, 0):
        tag = f"hopper_T{T}"
        env = E.make("HopperRunning-v0", terminate_when_unhealthy=bool(T), dtype=torch.float64)
        assert env.dt == float(g[tag + "_dt"])
        obs, pre, act = g[tag + "_obs"], g[tag + "_pre_obs"], g[tag + "_action"]
        r = env.get_batch_reward(obs, pre, act)
        d = env.get_batch_terminal(obs, pre, act)
        assert r.shape == (obs.shape[0], 1) and d.shape == (obs.shape[0], 1) and d.dtype == np.bool_
        assert close64(r, g[tag + "_reward"]) and np.array_equal(d, g[tag + "_done"])
        assert np.array_equal(env.is_healthy(obs), g[tag + "_healthy"])
        r2, d2 = env.get_batch_reward_terminal(obs, pre, act)
        assert np.array_equal(r2, r, equal_nan=True) and np.array_equal(d2, d)
    # the reference's own known-answer test (test_hopper.py:6-25)
    env = E.make("HopperRunning-v0", dtype=torch.float64)
    assert env.is_healthy(np.ones([128, 12])).shape == (128,) and np.all(env.is_healthy(np.ones([128, 12])))
    assert not np.any(env.is_healthy(np.ones([128, 12]) * 101))
    r = env.get_batch_reward(obs=np.ones([128, 12]), pre_obs=np.ones([128, 12]), action=np.ones([128, 3]))
    assert r.shape == (128, 1) and close64(r, g["hopper_kat_reward"])
    assert env.get_batch_terminal(obs=np.ones([128, 12])).shape == (128, 1)
    # non-default constructor arguments
    env = E.make(
        "HopperRunning-v0", freq_rate=2, real_time_scale=0.01, forward_reward_weight=1.5, ctrl_cost_weight=2e-3,
        healthy_reward=0.5, terminate_when_unhealthy=False, healthy_state_range=(-50.0, 60.0), healthy_z_range=(0.8, 2.0),
        dtype=torch.float64,
    )
    obs, pre, act = g["hopper_custom_obs"], g["hopper_custom_pre_obs"], g["hopper_custom_action"]
    assert close64(env.get_batch_reward(obs, pre, act), g["hopper_custom_reward"])
    assert np.array_equal(env.get_batch_terminal(obs), g["hopper_custom_done"])


def test_halfcheetah_scoring_f64_vs_golden(golden):
    g = golden("scoring")
    env = E.make("HalfCheetahRunning-v0", dtype=torch.float64)
    obs, pre, act = g["halfcheetah_obs"], g["halfcheetah_pre_obs"], g["halfcheetah_action"]
    assert close64(env.get_batch_reward(obs, pre, act), g["halfcheetah_reward"])
    assert np.array_equal(env.get_batch_terminal(obs, pre, act), g["halfcheetah_done"])


@pytest.mark.parametrize("name", ("hopper", "halfcheetah"))
def test_mujoco_scoring_f32_identical_inputs(golden, name):
    g = golden("scoring")
    tag = "hopper_T0" if name == "hopper" else "halfcheetah"
    obs, pre, act = (g[tag + s].astype(np.float32) for s in ("_obs", "_pre_obs", "_action"))
    if name == "hopper":
        env = E.make("HopperRunning-v0", terminate_when_unhealthy=False, dtype=torch.float32)
        p = O.HopperParams(terminate_when_unhealthy=False)
        ref_r = O.hopper_reward(obs.astype(np.float64), pre.astype(np.float64), act.astype(np.float64), p)
        ref_d = O.hopper_terminal(obs.astype(np.float64), p)
    else:
        env = E.make("HalfCheetahRunning-v0", dtype=torch.float32)
        p = O.HalfCheetahParams()
        ref_r = O.halfcheetah_reward(obs.astype(np.float64), pre.astype(np.float64), act.astype(np.float64), p)
        ref_d = O.halfcheetah_terminal(obs.astype(np.float64))
    r, d = env.get_batch_reward_terminal(obs, pre, act)
    fin = np.isfinite(ref_r)
    # the batch-wide control cost (hundreds) is subtracted from an O(1) term: compare at the
    # magnitude of the operands, which is what float32 arithmetic can resolve
    cc = p.ctrl_cost_weight * float(np.sum(np.square(act.astype(np.float64))))
    assert np.all(np.abs(r.astype(np.float64) - ref_r)[fin] <= 1e-6 + 1e-5 * (np.abs(ref_r[fin]) + cc))
    assert np.array_equal(np.isnan(r), np.isnan(ref_r))
    assert np.array_equal(d, ref_d)


@pytest.mark.parametrize(
    "kind",
    list(IP) + ["i2p_rebound_balancing", "i2p_boundary_balancing", "i2p_rebound_swingup", "i2p_boundary_swingup"],
)
def test_pendulum_scoring_vs_golden(golden, kind):
    g = golden("scoring")
    ids = dict(IP)
    ids.update({k: k.replace("i2p_", "").title().replace("_", "") for k in ()})
    name = {
        "i2p_rebound_balancing": "ReboundInvertedDoublePendulumBalancing-v0",
        "i2p_boundary_balancing": "BoundaryInvertedDoublePendulumBalancing-v0",
        "i2p_rebound_swingup": "ReboundInvertedDoublePendulumSwingUp-v0",
        "i2p_boundary_swingup": "BoundaryInvertedDoublePendulumSwingUp-v0",
        **IP,
    }[kind]
    obs = g[kind + "_obs"]
    env = E.make(name, dtype=torch.float64)
    assert close64(env.get_batch_reward(obs), g[kind + "_reward"])
    assert np.array_equal(env.get_batch_terminal(obs), g[kind + "_done"])
    env32 = E.make(name, dtype=torch.float32)
    o32 = obs.astype(np.float32)
    r32, d32 = env32.get_batch_reward_terminal(o32)
    if kind.startswith("ip"):
        ref_r, ref_d = O.ip_reward(kind, o32.astype(np.float64)), O.ip_terminal(kind, o32.astype(np.float64))
    else:
        ref_r, ref_d = O.i2p_reward(kind, o32.astype(np.float64)), O.i2p_terminal(kind, o32.astype(np.float64))
    fin = np.isfinite(ref_r)
    assert within32(r32[fin], ref_r[fin]).all()
    # flags: exact, except rows within 1e-4 of a threshold of THIS variant (inverted_pendulum.py:73-79,103-111,
    # 139-146,174-183; inverted_double_pendulum.py:84-90,114-122,150-157,185-196)
    o64 = o32.astype(np.float64)
    if kind.startswith("ip"):
        y, x_rail = np.cos(o64[:, 1]), 2.0
        y_thr = {"ip_rebound_balancing": 0.9, "ip_boundary_balancing": 0.0}.get(kind)
    else:
        y, x_rail = np.cos(o64[:, 1]) + np.cos(o64[:, 1] + o64[:, 2]), 3.0
        y_thr = {"i2p_rebound_balancing": 1.5, "i2p_boundary_balancing": 0.0}.get(kind)
    near = np.zeros(o64.shape[0], dtype=bool)
    if y_thr is not None:
        near |= np.abs(y - y_thr) < 1e-4
    if "boundary" in kind:
        near |= np.abs(np.abs(o64[:, 0]) - x_rail) < 1e-4
    assert np.array_equal(d32[~near], ref_d[~near]) and near.mean() < 0.01


def test_mujoco_init_obs_distribution_and_philox():
    for name, d, mean, sigma in (
        ("HopperRunning-v0", 12, [0, 1.25] + [0] * 10, 5e-3),
        ("HalfCheetahRunning-v0", 18, [0] * 18, 0.1),
        ("BoundaryInvertedPendulumSwingUp-v0", 4, [0] * 4, 5e-3),
    ):
        env = E.make(name, dtype=torch.float64)
        env._reseed(11)
        obs = env.get_batch_init_obs(8192)
        assert obs.shape == (8192, d)
        seed0 = (11 * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        host = P.init_gaussian(8192, d, np.array(mean, dtype=np.float64), np.full(d, sigma), seed0)
        assert np.allclose(obs.cpu().numpy(), host, rtol=0, atol=1e-12 * max(1.0, sigma * 10))
        x = obs.cpu().numpy() - np.array(mean)
        assert np.allclose(x.mean(0), 0, atol=5 * sigma / np.sqrt(8192)) and np.allclose(x.std(0), sigma, rtol=0.05)
        pos, vel = env.get_batch_init_state(16)
        assert pos.shape == (16, d // 2) and vel.shape == (16, d // 2)
        assert env.transform_state_to_obs((pos, vel)).shape == (16, d)
        p2, v2 = env.transform_obs_to_state(obs)
        assert p2.shape[1] == d // 2 and v2.shape[1] == d // 2
    env = E.make("HopperRunning-v0", init_noise_params=(0.0, 0.2), dtype=torch.float64)
    o = env.get_batch_init_obs(4096).cpu().numpy()
    assert np.all(o[:, :6] == np.array([0, 1.25, 0, 0, 0, 0])) and abs(o[:, 6:].std() - 0.2) < 0.01
    env = E.make("HopperRunning-v0", init_noise_params={1: (0.3, 0.0)}, dtype=torch.float64)
    o = env.get_batch_init_obs(4096).cpu().numpy()
    assert abs(o[:, 1].std() - 0.3) < 0.02 and np.all(o[:, 2:] == 0)


# ================================================================================================
# BASELINE.json full sizes: size-independent properties + strided oracle subsample
# ================================================================================================
def test_c2_full_size_properties():
    """C2: ContinuousCartPoleSwingUp, 2^20 envs, freq_rate=4 (SURVEY 8(d))."""
    n = 1 << 20
    rng = np.random.default_rng(1002)
    st = (rng.uniform(-1, 1, size=(n, 4)) * np.array([4.0, 5.0, np.pi, 8.0])).astype(np.float32)
    k = n // 100
    st[:k, 0] = np.sign(st[:k, 0]) * rng.uniform(4.99, 5.01, size=k).astype(np.float32)
    act = rng.uniform(-1, 1, size=(n, 1)).astype(np.float32)
    env = CP.ContinuousCartPoleSwingUpEnv(freq_rate=4, num_envs=n, dtype=torch.float32)
    env.state = st
    env.reset_stats()
    obs, rew, done, _, _ = env.step(act)
    # statistics reductions == reductions of the outputs
    rs, dc = env.read_stats()
    assert dc == int(done.sum())
    assert abs(rs - float(rew.double().sum())) < 1e-6 * n
    # strided subsample against the reference-arithmetic oracle
    idx = np.arange(0, n, 16)
    p = O.cartpole_params("continuous_swingup")
    ref = O.cartpole_step_f64ref(st[idx].astype(np.float64), O.cartpole_force(act[idx], True, p), 0.02, 4, p, libm=False)
    o = obs.cpu().numpy()[idx]
    frac = np.abs(o - ref) / (1e-6 + 1e-5 * np.abs(ref))
    assert frac.max() <= 1.0, f"worst envelope fraction {frac.max()}"
    near = np.abs(np.abs(ref[:, 0]) - 5.0) < 1e-4
    assert np.array_equal(done.cpu().numpy()[idx][~near], O.cartpole_terminal("swingup", ref, p)[~near])
    # idempotence of freeze/unfreeze and determinism of the kernel
    env.freeze()
    o2 = env.step(act)[0].clone()
    env.unfreeze()
    assert torch.equal(env.step(act)[0], o2)


def test_c3_full_size_properties():
    """C3: Hopper / HalfCheetah reward+terminal on 2^24 synthetic transitions (float32)."""
    n = 1 << 24
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(1003)
    for name, d, a_dim in (("HopperRunning-v0", 12, 3), ("HalfCheetahRunning-v0", 18, 6)):
        kw = dict(terminate_when_unhealthy=False) if d == 12 else {}
        env = E.make(name, dtype=torch.float32, **kw)
        env.accumulate_scoring_stats = True
        obs = torch.randn((n, d), device=dev, generator=gen)
        if d == 12:
            obs[:, 1] = 1.25 + 0.4 * obs[:, 1]
            obs[:, 2:] *= 30.0
        bad = torch.randint(0, n, (n // 1000,), device=dev, generator=gen)
        obs[bad, 3] = float("nan")
        pre = obs.clone()
        pre[:, 0] -= 0.01 * torch.randn(n, device=dev, generator=gen)
        act = torch.rand((n, a_dim), device=dev, generator=gen) * 2 - 1
        env.reset_stats()
        r, dn = env.get_batch_reward_terminal(obs, pre, act)
        rs, dc = env.read_stats()
        assert dc == int(dn.sum())
        assert int(dn.sum()) >= len(torch.unique(bad))
        # subsample vs oracle with the batch-wide control cost taken from the full batch
        idx = torch.arange(0, n, 256, device=dev)
        sumsq = float((act.double() ** 2).sum())
        o, p_, a = obs[idx].cpu().numpy().astype(np.float64), pre[idx].cpu().numpy().astype(np.float64), act[idx].cpu().numpy().astype(np.float64)
        if d == 12:
            P_ = O.HopperParams(terminate_when_unhealthy=False)
            ref_r, ref_d = O.hopper_reward(o, p_, a, P_, sumsq=sumsq), O.hopper_terminal(o, P_)
        else:
            P_ = O.HalfCheetahParams()
            ref_r, ref_d = O.halfcheetah_reward(o, p_, a, P_, sumsq=sumsq), O.halfcheetah_terminal(o)
        rr = r[idx].cpu().numpy().astype(np.float64)
        fin = np.isfinite(ref_r)
        cc = P_.ctrl_cost_weight * sumsq
        assert np.all(np.abs(rr - ref_r)[fin] <= 1e-6 + 1e-5 * (np.abs(ref_r[fin]) + cc))
        assert np.array_equal(dn[idx].cpu().numpy(), ref_d)
        del obs, pre, act, r, dn
        torch.cuda.empty_cache()


@pytest.mark.parametrize("env_id,n", (("ContinuousCartPoleSwingUp-v0", 1 << 20), ("CartPoleSwingUp-v0", (1 << 21) + 5),
                                      ("BoundaryInvertedPendulumSwingUp-v0", 4096), ("ReboundInvertedPendulumBalancing-v0", 1 << 20)))
def test_step_mirror_symmetry_full_size(env_id, n):
    """A size-independent property of the dynamics (cartpole.py:48-60 is odd in (x, x', theta, theta', F)): stepping
    the mirrored batch with the mirrored actions gives the mirrored result BIT FOR BIT -- every float32 operation of
    the kernel (packed FMAs, Cody-Waite reduction, quadrant logic, angle addition, MUFU.RCP) is sign-symmetric under
    round-to-nearest -- with the same rewards (cos is even) and done flags.  Full BASELINE batch sizes."""
    a = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=4)
    b = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=4)
    g = torch.Generator(device=a.device)
    g.manual_seed(77)
    scale = torch.tensor([4.0, 5.0, 3.14159, 8.0], device=a.device)
    if "InvertedPendulum" in env_id:
        scale = torch.tensor([1.9, 3.14159, 5.0, 8.0], device=a.device)
    st = (torch.rand((n, 4), device=a.device, generator=g) * 2 - 1) * scale
    st[: n // 16] *= 25.0  # un-wrapped angles, envs far outside the rail
    cont = len(a.action_space.shape) > 0
    if cont:
        hi = float(a.action_space.high[0])
        act = (torch.rand(n, device=a.device, generator=g) * 2 - 1) * hi
        act_m = -act
    else:
        act = torch.randint(0, 2, (n,), device=a.device, generator=g, dtype=torch.uint8)
        act_m = 1 - act
    a.state, b.state = st, -st
    o1, r1, d1, _, _ = a.step(act)
    o2, r2, d2, _, _ = b.step(act_m)
    assert torch.equal(a.state, -b.state)
    if "InvertedPendulum" in env_id:  # the observation wraps theta into [-pi, pi): mirrored except exactly at -pi
        inner = o1[:, 1] != -math.pi
        assert torch.equal(o1[inner], -o2[inner])
    else:
        assert torch.equal(o1, -o2)
    assert torch.equal(r1, r2) and torch.equal(d1, d2)


def test_c4_full_size_properties():
    """C4: ChargedBallCentering, 2^26 envs (SURVEY 8(d)): size-independent properties at the full batch -- a fused
    rollout equals the same number of step calls bit for bit, statistics equal the sums of the outputs, sharded
    init equals unsharded init, and a strided subsample follows the float64 oracle step by step."""
    n, T = 1 << 26, 3
    a = CB.ChargedBallCenteringEnv(num_envs=n, dtype=torch.float32)
    a.reset(seed=1004)
    half = CB.ChargedBallCenteringEnv(num_envs=n // 2, dtype=torch.float32, env_offset=n // 2)
    half.reset(seed=1004)
    for k in ("on_circle", "circle_state", "free_state"):
        assert torch.equal(a.state[k][n // 2 :], half.state[k])
    del half
    g = torch.Generator(device=a.device)
    g.manual_seed(4)
    acts = torch.randint(0, 2, (T, n), device=a.device, generator=g, dtype=torch.uint8)
    idx = torch.arange(0, n, 4096, device=a.device)
    sub = {k: v[idx].cpu().numpy() for k, v in a.state.items()}
    b = CB.ChargedBallCenteringEnv(num_envs=n, dtype=torch.float32)
    b.state = {k: v.clone() for k, v in a.state.items()}
    p = O.ChargedBallParams()
    on, ci, fre = sub["on_circle"].astype(bool), sub["circle_state"].astype(np.float64), sub["free_state"].astype(np.float64)
    a.reset_stats()
    total = 0.0
    for t in range(T):
        obs, rew, done, _, _ = a.step(acts[t])
        total += float(rew.double().sum())
        assert not bool(done.any())  # charged_ball.py:110-111
        # teacher-forced subsample: oracle step from the engine's own previous float32 state
        on_in, ci_in = on, ci
        on, ci, fre, near = cb_substep_trace(on, ci, fre, O.charged_ball_force(acts[t][idx].cpu().numpy(), False, p), 1, p)
        got = {k: v[idx].cpu().numpy() for k, v in a.state.items()}
        ok_rows = cb_assert_f32_step(got, on_in, ci_in, on, ci, fre, near)  # 1.0 x envelope, flags exact off the thresholds
        assert ok_rows.mean() > 0.99
        on, ci, fre = got["on_circle"].astype(bool), got["circle_state"].astype(np.float64), got["free_state"].astype(np.float64)
    rs, dc = a.read_stats()
    assert dc == 0 and abs(rs - total) < 1e-6 * abs(total)
    out = b.rollout(T, actions=acts, record=False, auto_reset=False, max_episode_steps=0)
    for k in ("on_circle", "circle_state", "free_state"):
        assert torch.equal(a.state[k], b.state[k]), k
    assert abs(float(out["stats"][0]) - total) < 1e-6 * abs(total)


def test_c5_freeze_unfreeze_full_size():
    """C5's freeze / unfreeze at its per-GPU size (2^26 cart-pole envs, SURVEY 8(d)): freeze -> steps -> unfreeze restores
    the state bit for bit (core.py:18-37, base_control.py:32-36), a second freeze overwrites the snapshot, and stepping
    after the restore reproduces the first trajectory."""
    n = 1 << 26
    env = CP.CartPoleSwingUpEnv(num_envs=n, dtype=torch.float32, freq_rate=1)
    env.reset(seed=1005)
    g = torch.Generator(device=env.device)
    g.manual_seed(9)
    act = torch.randint(0, 2, (n,), device=env.device, generator=g, dtype=torch.uint8)
    s0 = env.state.clone()
    env.freeze()
    o1 = env.step(act)[0].clone()
    env.step(act)
    env.unfreeze()
    assert torch.equal(env.state, s0)
    assert torch.equal(env.step(act)[0], o1)
    env.freeze()  # snapshot of the stepped state replaces the old one
    s1 = env.state.clone()
    env.step(act)
    env.unfreeze()
    assert torch.equal(env.state, s1) and not torch.equal(s1, s0)


def test_empty_and_ragged_batches():
    from emei_b200 import _lib

    # n = 0 is a valid no-op at the C ABI
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant = 1, 0.02, _lib.CARTPOLE_SWINGUP
    import ctypes

    assert _lib.lib.emei_cartpole_step_f32(None, None, None, None, None, None, None, 0, ctypes.byref(p), None) == 0
    # ragged sizes (not multiples of the CTA / vector width)
    for n in (1, 31, 257, 1000003):
        env = CP.CartPoleSwingUpEnv(num_envs=n, freq_rate=2)
        env.reset(seed=n)
        env.reset_stats()
        o, r, d, _, _ = env.step(env.action_space.sample_batch(n))
        assert o.shape == (n, 4) and torch.isfinite(o).all()
        rs, dc = env.read_stats()
        assert abs(rs - float(r.double().sum())) < 1e-6 * n and dc == int(d.sum())
    env = E.make("HalfCheetahRunning-v0", dtype=torch.float64)
    for n in (1, 5, 1025):
        r, d = env.get_batch_reward_terminal(np.zeros((n, 18)), np.zeros((n, 18)), np.ones((n, 6)))
        assert r.shape == (n, 1) and close64(r, np.full((n, 1), -0.1 * 6 * n))


# ================================================================================================
# step_host: the end-to-end host path (chunked multi-stream pipeline) must equal step() bit for bit
# ================================================================================================
# 1000: the kernel reads / writes the pinned host arrays itself (small-batch kernel); 20 000: the same through the TMA kernel (actions by
# DMA, results stored to host memory); 300 000: one range through the copy engines; 1 100 003: two unequal ranges with a ragged end
@pytest.mark.parametrize("n", (1000, 20_000, 300_000, 1_100_003))
@pytest.mark.parametrize("env_id", ("ContinuousCartPoleSwingUp-v0", "CartPoleBalancing-v0", "BoundaryInvertedPendulumSwingUp-v0",
                                    "ChargedBallCentering-v0", "BoundaryInvertedDoublePendulumSwingUp-v0"))
def test_step_host_equals_step(env_id, n):
    rng = np.random.default_rng(5)
    a = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=2)
    b = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=2)
    a.reset(seed=11)
    b.reset(seed=11)
    cont = len(a.action_space.shape) > 0
    for t in range(3):
        if cont:
            lo, hi = float(a.action_space.low[0]), float(a.action_space.high[0])
            act = rng.uniform(lo, hi, size=n).astype(np.float32)
        else:
            act = rng.integers(0, 2, size=n).astype(np.uint8)
        o1, r1, d1, _, _ = a.step(torch.as_tensor(act).cuda())
        o2, r2, d2, tr, info = b.step_host(act)
        assert tr is False and info == {}
        assert isinstance(o2, np.ndarray) and o2.shape == (n, 6 if "Double" in env_id else 4) and r2.shape == (n, 1) and d2.dtype == np.bool_
        assert np.array_equal(o1.cpu().numpy(), o2, equal_nan=True)
        assert np.array_equal(r1.cpu().numpy(), r2, equal_nan=True)
        assert np.array_equal(d1.cpu().numpy(), d2)
    sa, sb = a.state, b.state
    if isinstance(sa, dict):
        for k in sa:
            assert torch.equal(sa[k], sb[k])
    else:
        assert torch.equal(sa, sb)
    assert a.read_stats()[1] == b.read_stats()[1]


@pytest.mark.parametrize("env_id,n", (("ContinuousCartPoleSwingUp-v0", 1 << 19), ("BoundaryInvertedPendulumSwingUp-v0", 4096),
                                      ("ChargedBallCentering-v0", 300_000)))
def test_step_host_graph_replay_equals_step(env_id, n):
    """step_host captures its copy / kernel / copy pipeline into a CUDA graph per (action buffer, ping-pong side) and
    replays it: many steps from ONE pinned buffer rewritten in place, from a second buffer, with device-side step()
    calls in between and with a set_state, must equal step() bit for bit, and the graph path must really be taken."""
    rng = np.random.default_rng(6)
    a = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=2)
    b = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=2)
    a.reset(seed=12)
    b.reset(seed=12)
    cont = len(a.action_space.shape) > 0
    bufs = [torch.empty(n, dtype=torch.float32 if cont else torch.uint8).pin_memory() for _ in range(2)]

    def draw(buf):
        if cont:
            lo, hi = float(a.action_space.low[0]), float(a.action_space.high[0])
            buf.copy_(torch.as_tensor(rng.uniform(lo, hi, size=n).astype(np.float32)))
        else:
            buf.copy_(torch.as_tensor(rng.integers(0, 2, size=n).astype(np.uint8)))

    for t in range(12):
        buf = bufs[0] if t < 8 else bufs[1]
        draw(buf)
        if t == 5:  # a device-side step in between flips the ping-pong side under the staging object
            dev_act = buf.cuda()
            a.step(dev_act)
            b.step(dev_act)
        if t == 9:  # new states written into the live buffers: the captured graphs must still see them
            st = a.state
            st = {k: v.clone() for k, v in st.items()} if isinstance(st, dict) else st.clone()
            a.state = st
            b.state = st
        o1, r1, d1, _, _ = a.step(buf.cuda())
        o2, r2, d2, _, _ = b.step_host(buf)
        assert np.array_equal(o1.cpu().numpy(), o2, equal_nan=True), t
        assert np.array_equal(r1.cpu().numpy(), r2, equal_nan=True) and np.array_equal(d1.cpu().numpy(), d2), t
    assert len(b._staging._graphs) >= 2  # replayed, not only eager
    assert a.read_stats()[1] == b.read_stats()[1]
    b._staging.use_graphs = False  # the eager path stays available and agrees
    draw(bufs[0])
    o1 = a.step(bufs[0].cuda())[0]
    assert np.array_equal(o1.cpu().numpy(), b.step_host(bufs[0])[0], equal_nan=True)


# ================================================================================================
# fused T-step rollout (SURVEY 8f rank 1): zoo/util.py:33-93 batched, TimeLimit + auto-reset in-kernel
# ================================================================================================
from oracle import rollout_oracle as RO  # noqa: E402


@pytest.mark.parametrize("env_id,kind,cont", (
    ("CartPoleSwingUp-v0", "swingup", False),
    ("ContinuousCartPoleSwingUp-v0", "continuous_swingup", True),
    ("CartPoleBalancing-v0", "balancing", False),
))
def test_rollout_teacher_forced_vs_oracle(env_id, kind, cont):
    """Every recorded transition is checked against the oracle's step from the recorded observation
    (teacher-forced), the TimeLimit / done / auto-reset bookkeeping against the restated loop, the
    reset samples against the Philox mirror, and each step bit-for-bit against the step kernel."""
    n, T, fr = 512, 40, 4
    max_steps = 3 if kind == "balancing" else 25  # balancing under random pushes falls within a few steps
    env = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    env.reset(seed=3)
    rng = np.random.default_rng(1)
    acts = rng.uniform(-1, 1, size=(T, n)).astype(np.float32) if cont else rng.integers(0, 2, size=(T, n)).astype(np.uint8)
    st0 = env.state.cpu().numpy().copy()
    if kind != "balancing":  # push a slice near the rail so that terminations happen inside the horizon
        st0[: n // 4, 0] = np.sign(st0[: n // 4, 0] + 1e-9) * 4.9
        st0[: n // 4, 1] = np.sign(st0[: n // 4, 0]) * 3.0
        env.state = st0
    out = env.rollout(T, actions=acts, record=True, max_episode_steps=max_steps)
    obs, nxt, ra = (out[k].cpu().numpy() for k in ("observations", "next_observations", "actions"))
    rew, dones, tmo = (out[k].cpu().numpy() for k in ("rewards", "dones", "timeouts"))
    assert np.array_equal(ra, acts) and np.array_equal(obs[0], st0)
    p = O.cartpole_params(kind)
    seed_reset, _ = RO.rollout_seeds(3)
    pi_col = 2 if "swingup" in kind else -1
    ep_step, ep_ret, ep_idx = np.zeros(n, np.int64), np.zeros(n, np.float32), np.zeros(n, np.int64)
    stepper = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    fin, fin_ret, fin_len, n_term = 0, 0.0, 0, 0
    for t in range(T):
        ref = O.cartpole_step_f64ref(obs[t].astype(np.float64), O.cartpole_force(acts[t].reshape(-1, 1) if cont else acts[t], cont, p), 0.02, fr, p)
        assert within32(nxt[t], ref).all()
        assert within32(rew[t], O.cartpole_reward(kind, ref)[:, 0]).all()
        near = (np.abs(np.abs(ref[:, 0]) - p.x_threshold) < 1e-4) | (np.abs(np.abs(ref[:, 2]) - p.theta_threshold_radians) < 1e-4)
        term = O.cartpole_terminal(kind, nxt[t].astype(np.float64), p)[:, 0]  # flags from the engine's own next_obs
        assert np.array_equal(term[~near], O.cartpole_terminal(kind, ref, p)[:, 0][~near])
        done, trunc, ep_step, ep_ret = RO.bookkeeping(term, max_steps, ep_step, ep_ret, rew[t])
        assert np.array_equal(dones[t], done) and np.array_equal(tmo[t], trunc)
        n_term += int(term.sum())
        # the step kernel computes the same bits
        stepper.state = obs[t]
        o2, r2, d2, _, _ = stepper.step(acts[t])
        assert np.array_equal(o2.cpu().numpy(), nxt[t]) and np.array_equal(r2.cpu().numpy()[:, 0], rew[t])
        assert np.array_equal(d2.cpu().numpy()[:, 0], term)
        # auto-reset: next observation = next_obs, or a fresh Philox reset sample
        idx = np.nonzero(done)[0]
        fin += idx.size
        fin_ret += float(ep_ret[idx].astype(np.float64).sum())
        fin_len += int(ep_step[idx].sum())
        ep_idx[idx] += 1
        expect = nxt[t].copy()
        if idx.size:
            expect[idx] = RO.reset_sample_uniform(idx, ep_idx[idx], seed_reset, pi_column=pi_col)
        ep_step[idx], ep_ret[idx] = 0, 0.0
        nxt_state = obs[t + 1] if t + 1 < T else env.state.cpu().numpy()
        assert np.array_equal(nxt_state, expect)
    assert fin > 0 and tmo.any() and (dones & ~tmo).any()  # both ways of ending an episode were exercised
    info = env.rollout_info(out["stats"])
    assert info["total_episode_num"] == fin and info["terminated"] == n_term
    assert info["truncated"] == int(tmo.sum())
    assert abs(info["reward_sum"] - float(rew.astype(np.float64).sum())) < 1e-3 * max(1.0, abs(float(rew.sum())))
    assert abs(info["avg_length"] - fin_len / fin) < 1e-9 and abs(info["avg_reward"] - fin_ret / fin) < 1e-3
    assert np.array_equal(env._engine.ep_step.cpu().numpy(), ep_step) and np.array_equal(env._engine.ep_index.cpu().numpy(), ep_idx)


def _same_state(a, b):
    if isinstance(a, dict):
        return all(torch.equal(a[k], b[k]) for k in a)
    return torch.equal(a, b)


@pytest.mark.parametrize("env_id,cont", (("CartPoleSwingUp-v0", False), ("ContinuousCartPoleSwingUp-v0", True),
                                         ("BoundaryInvertedPendulumSwingUp-v0", True), ("ChargedBallCentering-v0", False),
                                         ("ContinuousChargedBallCentering-v0", True)))
def test_rollout_random_policy_and_split_horizon(env_id, cont):
    """Built-in random policy = the Philox mirror, bit for bit; one rollout of T steps equals two of T/2
    (state, counters and the action stream continue); records off = records on."""
    n, T = 2048, 24
    a = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=1)
    b = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=1)
    c = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=1)
    for e in (a, b, c):
        e.reset(seed=21)
    full = a.rollout(T, record=True, max_episode_steps=10)
    h1 = b.rollout(T // 2, record=True, max_episode_steps=10)
    h2 = b.rollout(T // 2, record=True, max_episode_steps=10)
    c.rollout(T, record=False, max_episode_steps=10)
    for k in ("observations", "next_observations", "actions", "rewards", "dones", "timeouts"):
        assert torch.equal(full[k], torch.cat([h1[k], h2[k]], dim=0)), k
    assert _same_state(a.state, b.state) and _same_state(a.state, c.state)
    assert torch.allclose(full["stats"], h1["stats"] + h2["stats"], rtol=1e-9)
    _, seed_action = RO.rollout_seeds(21)
    lo, hi = (float(a.action_space.low[0]), float(a.action_space.high[0])) if cont else (0, 1)
    ref = RO.random_actions(seed_action, n, 0, T, cont, lo, hi)
    got = full["actions"].cpu().numpy()
    assert np.array_equal(got, ref)
    if not cont:
        assert 0.45 < got.mean() < 0.55
    assert full["timeouts"].any()


def test_rollout_ip_reset_samples_and_wrap():
    n, T = 1024, 30
    env = E.make("BoundaryInvertedPendulumSwingUp-v0", num_envs=n, dtype=torch.float32)
    env.reset(seed=8)
    st0 = env.state.cpu().numpy().copy()
    st0[:, 1] += 50.0  # un-wrapped angles: the recorded observation must be wrapped, the state not
    env.state = st0
    out = env.rollout(T, record=True, max_episode_steps=7)
    obs, nxt, dones = (out[k].cpu().numpy() for k in ("observations", "next_observations", "dones"))
    assert np.all(np.abs(obs[..., 1]) <= np.pi + 1e-6) and np.all(np.abs(nxt[..., 1]) <= np.pi + 1e-6)
    seed_reset, _ = RO.rollout_seeds(8)
    sp = np.full(4, 5e-3)
    ep_idx = np.zeros(n, np.int64)
    for t in range(T - 1):
        idx = np.nonzero(dones[t])[0]
        ep_idx[idx] += 1
        if idx.size:
            ref = RO.reset_sample_gaussian(idx[:16], ep_idx[idx[:16]], seed_reset, np.zeros(4), sp)
            assert np.allclose(obs[t + 1][idx[:16]], ref, rtol=0, atol=1e-9)
    assert dones.any()


@pytest.mark.parametrize("env_id,cont", (("ChargedBallCentering-v0", False), ("ContinuousChargedBallCentering-v0", True)))
def test_rollout_charged_ball_equals_step_kernel(env_id, cont):
    """A charged-ball rollout = T calls of the (oracle-pinned) step kernel, bit for bit, plus the TimeLimit
    bookkeeping of zoo/util.py:58-73 and in-kernel resets equal to charged_ball.py:84-94 on the Philox mirror."""
    # long enough for take-offs and landings (both branches + free_to_circle); weaker continuous fields need longer
    n, fr = 1024, 2
    T, max_steps = (180, 100) if cont else (70, 30)
    env = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    ref = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    env.reset(seed=5)
    ref.state = {k: v.clone() for k, v in env.state.items()}
    rng = np.random.default_rng(2)
    if cont:  # strong fields, else the ball never leaves the ring within an episode
        acts = (rng.choice([-1.0, 1.0], size=(T, n)) * rng.uniform(0.7, 1.0, size=(T, n))).astype(np.float32)
    else:
        acts = rng.integers(0, 2, size=(T, n)).astype(np.uint8)
    out = env.rollout(T, actions=acts, record=True, max_episode_steps=max_steps)
    obs, nxt, rew = (out[k].cpu().numpy() for k in ("observations", "next_observations", "rewards"))
    dones, tmo = out["dones"].cpu().numpy(), out["timeouts"].cpu().numpy()
    assert np.array_equal(out["actions"].cpu().numpy(), acts) and np.array_equal(dones, tmo)
    seed_reset, _ = RO.rollout_seeds(5)
    ep_step, ep_idx = np.zeros(n, np.int64), np.zeros(n, np.int64)
    saw_free = False
    for t in range(T):
        assert np.array_equal(obs[t], ref.state["free_state"].cpu().numpy())
        o2, r2, d2, _, _ = ref.step(acts[t])
        assert np.array_equal(o2.cpu().numpy(), nxt[t]) and np.array_equal(r2.cpu().numpy()[:, 0], rew[t])
        assert not d2.any()
        saw_free |= bool((ref.state["on_circle"] == 0).any())
        ep_step += 1
        trunc = ep_step >= max_steps
        assert np.array_equal(tmo[t], trunc)
        idx = np.nonzero(trunc)[0]
        if idx.size:
            ep_idx[idx] += 1
            on, circle, free = RO.reset_sample_charged_ball(idx, ep_idx[idx], seed_reset)
            got_free = (obs[t + 1] if t + 1 < T else env.state["free_state"].cpu().numpy())[idx]
            assert np.allclose(got_free, free, rtol=0, atol=3e-7)
            st = {k: v.clone() for k, v in ref.state.items()}
            j = torch.as_tensor(idx, device=st["circle_state"].device)
            st["on_circle"][j] = 1
            st["circle_state"][j] = torch.as_tensor(circle, device=j.device)
            st["free_state"][j] = torch.as_tensor(got_free, device=j.device)
            ref.state = st
            ep_step[idx] = 0
    assert saw_free and tmo.any()
    assert _same_state(env.state, ref.state)
    info = env.rollout_info(out["stats"])
    assert info["truncated"] == int(tmo.sum()) == info["total_episode_num"] and info["terminated"] == 0
    assert abs(info["avg_length"] - max_steps) < 1e-9
    assert abs(info["reward_sum"] - float(rew.astype(np.float64).sum())) < 1e-3 * max(1.0, abs(float(rew.sum())))
    assert np.array_equal(env._engine.ep_step.cpu().numpy(), ep_step) and np.array_equal(env._engine.ep_index.cpu().numpy(), ep_idx)


@pytest.mark.parametrize("env_id,cont,n", (
    ("ContinuousCartPoleSwingUp-v0", True, 148 * 24 * 512 + 1234),   # > 24 chunks per SM: the TMA ring recycles its slots
    ("CartPoleSwingUp-v0", False, 148 * 26 * 512 * 2 + 77),          # uint8 actions, two laps of the ring, ragged tail
    ("BoundaryInvertedPendulumSwingUp-v0", True, 1 << 21),
    ("CartPoleBalancing-v0", False, 513),                             # small-batch kernel: the SCALAR form of the arithmetic
    ("CartPoleBalancing-v0", False, 8192 + 513),                      # smallest TMA batch: 17 chunks on 17 SMs, ragged tail
    ("ContinuousCartPoleSwingUp-v0", True, (1 << 24) + 3),            # 222 chunks per SM: every group's ring laps 11 times
))
def test_step_kernel_large_batches_equal_scalar_rollout(env_id, cont, n):
    """The step kernels (TMA ring with packed f32x2 pairs; the scalar small-batch kernel below 8192 envs) against the
    rollout kernel's one-step arithmetic (packed pairs, different pairing of envs) on the same inputs: bit for bit, at
    sizes that wrap the per-group shared-memory rings, with ragged tails; statistics equal the sums of the outputs."""
    fr = 4
    a = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    b = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    a.reset(seed=11)
    g = torch.Generator(device=a.device)
    g.manual_seed(5)
    st = a.state.clone()
    st.mul_(1.0 + 40.0 * torch.rand(st.shape, device=st.device, generator=g))  # spread the states out
    a.state = st
    b.state = st
    act = (torch.rand(n, device=a.device, generator=g) * 2 - 1) if cont else torch.randint(0, 2, (n,), device=a.device, generator=g, dtype=torch.uint8)
    a.reset_stats()
    obs, rew, done, _, _ = a.step(act)
    out = b.rollout(1, actions=act.reshape(1, n), record=True, auto_reset=False, max_episode_steps=0)
    assert torch.equal(obs, out["next_observations"][0])
    assert torch.equal(rew[:, 0], out["rewards"][0])
    assert torch.equal(done[:, 0], out["dones"][0])
    rs, dc = a.read_stats()
    assert dc == int(done.sum()) and abs(rs - float(rew.double().sum())) <= 1e-6 * max(1.0, abs(rs))
    # misaligned action array (element offset 1): the kernel reads actions directly instead of through TMA
    act2 = torch.empty(n + 1, dtype=act.dtype, device=act.device)[1:]
    act2.copy_(act)
    c = E.make(env_id, num_envs=n, dtype=torch.float32, freq_rate=fr)
    c.state = st
    obs2, rew2, done2, _, _ = c.step(act2)
    assert torch.equal(obs2, obs) and torch.equal(rew2, rew) and torch.equal(done2, done)


# ================================================================================================
# rollout records -> the reference's dataset order (zoo/util.py:33-93,108-111)
# ================================================================================================
@pytest.mark.parametrize("T,n", ((1, 1), (37, 1000), (64, 33), (5, 4097),
                                 (1, 1000), (1000, 1), (45, 77),   # one step, one env; neither dimension a multiple of 16 or 32
                                 (257, 40001)))                    # more tiles than the 148 x 8 CTAs of the grid: grid-stride loop
def test_records_transpose_bit_exact(T, n):
    """every record element size: 1, 4, 8, 16 and the wide observation rows of 24 (6 x float32), 32 (4 x float64) and
    48 bytes (6 x float64), through the C ABI and through offline._transpose"""
    from emei_b200 import _lib, offline

    g = torch.Generator(device="cuda")
    g.manual_seed(T * 7919 + n)
    stream = torch.cuda.current_stream().cuda_stream
    for shape, dtype in (((T, n, 4), torch.float32), ((T, n), torch.float32), ((T, n), torch.uint8), ((T, n), torch.int64), ((T, n), torch.bool),
                         ((T, n), torch.float64), ((T, n, 6), torch.float32), ((T, n, 4), torch.float64), ((T, n, 6), torch.float64)):
        x = torch.randint(0, 250, shape, device="cuda", generator=g).to(dtype)
        want = x.transpose(0, 1).contiguous()
        elem = x.element_size() * (shape[2] if len(shape) > 2 else 1)
        out = torch.empty_like(want)
        assert _lib.lib.emei_records_transpose(x.data_ptr(), out.data_ptr(), T, n, elem, stream) == 0, f"{elem}-byte elements"
        assert torch.equal(out, want), f"{elem}-byte elements"
        y = offline._transpose(x, stream)
        assert y.dtype == x.dtype and torch.equal(y, want)


@pytest.mark.parametrize("env_id", ("CartPoleSwingUp-v0", "ContinuousChargedBallCentering-v0"))
def test_collect_dataset_matches_reference_layout(env_id, tmp_path):
    from emei_b200 import offline

    n, total = 256, 256 * 90
    env = E.make(env_id, num_envs=n, dtype=torch.float32)
    env.max_episode_steps = 40
    env._reseed(4)
    samples, info = offline.collect_dataset(env, total)
    N = samples["observations"].shape[0]
    assert N == total and samples["observations"].shape == (N, 4) and samples["rewards"].shape == (N,)
    assert samples["dones"].dtype == np.float32 and set(np.unique(samples["dones"])) <= {0.0, 1.0}
    cont = env_id.startswith("Continuous")
    assert samples["actions"].shape == ((N, 1) if cont else (N,))
    # env-major: inside one env's trajectory consecutive samples chain unless an episode ended (zoo/util.py:73)
    T = total // n
    obs, nxt = samples["observations"].reshape(n, T, 4), samples["next_observations"].reshape(n, T, 4)
    dones = samples["dones"].reshape(n, T).astype(bool)
    chain = (nxt[:, :-1] == obs[:, 1:]).all(axis=2)
    assert chain[~dones[:, :-1]].all() and not chain[dones[:, :-1]].all()
    assert (samples["timeouts"] <= samples["dones"]).all() and samples["timeouts"].sum() > 0
    assert info["total_episode_num"] == int(dones.sum()) and 1 <= info["avg_length"] <= 40
    path = offline.save_dataset(samples, tmp_path / "random.npz")
    back = offline.load_dataset(path, device=env.device)
    assert all(torch.equal(back[k].cpu(), torch.as_tensor(samples[k])) for k in offline.KEYS)


# ================================================================================================
# analytic inverted double pendulum step (SURVEY 8f rank 3)
# ================================================================================================
I2P = {
    "i2p_rebound_balancing": "ReboundInvertedDoublePendulumBalancing-v0",
    "i2p_boundary_balancing": "BoundaryInvertedDoublePendulumBalancing-v0",
    "i2p_rebound_swingup": "ReboundInvertedDoublePendulumSwingUp-v0",
    "i2p_boundary_swingup": "BoundaryInvertedDoublePendulumSwingUp-v0",
}


def i2p_inputs(seed, n):
    rng = np.random.default_rng(seed)
    st = rng.uniform(-1, 1, size=(n, 6)) * np.array([2.9, np.pi, np.pi, 4.0, 8.0, 10.0])
    st[: n // 8, 1:3] *= 20.0  # unwrapped angles
    st[n // 8 : n // 4, 0] = np.sign(st[n // 8 : n // 4, 0]) * rng.uniform(2.95, 3.05, n // 4 - n // 8)  # the rail ends
    st[n // 4 : n // 2, 1:3] *= 0.1  # near upright: the balancing variants' y threshold
    act = rng.uniform(-1.3, 1.3, size=(n, 1)).astype(np.float32)  # beyond ctrlrange: clamped like mj_step
    return st, act


@pytest.mark.parametrize("kind", list(I2P))
@pytest.mark.parametrize("fr", (1, 3))
def test_i2p_step_f64_vs_oracle(kind, fr):
    n = 4096
    st, act = i2p_inputs(3001, n)
    p = O.I2PParams()
    ref_state, ref_obs = O.i2p_step(st, act.astype(np.float64), 0.02, fr, kind.endswith("swingup"), p, libm=True)
    env = E.make(I2P[kind], freq_rate=fr, num_envs=n, dtype=torch.float64)
    env.state = st
    env.reset_stats()
    obs, rew, done, trunc, info = env.step(act)
    assert trunc is False and info == {}
    assert close64(env.state.cpu().numpy(), ref_state, 1e-11)
    o = obs.cpu().numpy()
    # the observation's "(theta + pi) % 2 * pi - pi" jumps by 2 pi where (theta + pi) crosses an even integer:
    # compare it from the engine's own state, and the state against the oracle
    assert np.allclose(o, O.i2p_wrap_obs(env.state.cpu().numpy()), rtol=0, atol=1e-12)
    assert close64(rew.cpu().numpy(), O.i2p_reward(kind, o), 1e-11)
    ref_done = O.i2p_terminal(kind, o)
    y = np.cos(o[:, 1]) + np.cos(o[:, 1] + o[:, 2])
    near = (np.abs(np.abs(o[:, 0]) - 3.0) < 1e-9) | (np.abs(y - 1.5) < 1e-9) | (np.abs(y) < 1e-9)
    assert np.array_equal(done.cpu().numpy()[~near], ref_done[~near])
    assert 0 < ref_done.mean() < 1 or kind == "i2p_rebound_swingup"
    rs, dc = env.read_stats()
    assert dc == int(done.sum()) and abs(rs - float(rew.sum())) < 1e-6 * max(1.0, abs(rs))


@pytest.mark.parametrize("kind", ("i2p_boundary_swingup", "i2p_rebound_balancing"))
def test_i2p_step_f32_vs_oracle_identical_inputs(kind):
    n = 4096
    st, act = i2p_inputs(3002, n)
    st[: n // 8, 1:3] /= 20.0  # float32 cannot hold angles of tens of radians to 1e-6
    st32 = st.astype(np.float32)
    p = O.I2PParams()
    ref_state, _ = O.i2p_step(st32.astype(np.float64), act.astype(np.float64), 0.02, 1, kind.endswith("swingup"), p)
    env = E.make(I2P[kind], num_envs=n, dtype=torch.float32)
    env.state = st32
    obs, rew, done, _, _ = env.step(act)
    got = env.state.cpu().numpy()
    # accelerations reach 1e3 rad/s^2 near the mass matrix's weak direction: allow the float32 evaluation error of
    # a (relative 1e-5 of |a| h) on the velocity rows
    acc = np.abs(ref_state[:, 3:] - st32[:, 3:].astype(np.float64))
    tol = 1e-6 + 1e-5 * np.abs(ref_state)
    tol[:, 3:] += 2e-5 * acc
    assert (np.abs(got - ref_state) <= tol).all()
    assert np.array_equal(obs.cpu().numpy()[:, [0, 3, 4, 5]], got[:, [0, 3, 4, 5]])
    assert rew.shape == (n, 1) and done.dtype == torch.bool


def test_i2p_reset_freeze_next_obs_and_graph():
    env = E.make("BoundaryInvertedDoublePendulumSwingUp-v0", num_envs=2048, dtype=torch.float64)
    obs, info = env.reset(seed=5)
    assert obs.shape == (2048, 6) and info == {} and float(obs.abs().max()) < 0.05  # N(0, 5e-3) on all six
    assert abs(float(obs.std()) - 5e-3) < 5e-4
    a = torch.rand(2048, device=env.device, dtype=torch.float64) * 2 - 1
    env.freeze()
    snap = env.state.clone()
    nxt = env.get_batch_next_obs(env.state, action=a)  # stateless: the env does not move
    assert torch.equal(env.state, snap)
    # state= takes precedence over obs, any batch size: rows 100..611 step exactly as in the full batch
    part = env.get_batch_next_obs(env.current_obs[:7], action=a[100:612], state=snap[100:612])
    assert torch.equal(part, nxt[100:612]) and env.num_envs == 2048
    o1, _, _, _, _ = env.step(a)
    assert torch.equal(o1, nxt)
    env.step(a)
    env.unfreeze()
    assert torch.equal(env.state, snap) and env.frozen is False
    g = env.get_transition_graph()
    assert g.shape == (7, 6) and g[6].tolist() == [0, 0, 0, 1, 1, 1]


# ================================================================================================
# obs_noise_params: Gaussian state noise after every sub-step (mujoco_env.py:98-104; SURVEY 8f rank 4)
# ================================================================================================
NOISE_MUL, NOISE_ADD = 0xA24BAED4963EE407, 0x9FB21C651E98DF25  # EmeiMujocoEnv._next_obs_noise


def _noise_seed(seed):
    return (seed * NOISE_MUL + NOISE_ADD) & 0xFFFFFFFFFFFFFFFF


@pytest.mark.parametrize("dtype", (torch.float64, torch.float32))
@pytest.mark.parametrize("fr", (1, 4))
def test_ip_obs_noise_vs_oracle_and_philox_mirror(dtype, fr):
    """Two consecutive noisy steps against the oracle fed with the Philox mirror's draws (teacher-forced), in both
    precisions, with ip_inputs' unwrapped angles; the (sigma_pos, sigma_vel) tuple form; sharded == unsharded.  float32 is
    held to the bar of test_c1_protocol_ip_f32_teacher_forced_200_steps (1.0 x the envelope, plus half an ulp32 of the
    variable per sub-step at freq_rate > 1); test_f32_reference_arithmetic.py covers every variant and the C1 rows."""
    n, kind = 2048, "ip_boundary_swingup"
    st, act = ip_inputs(4001, n)
    if dtype == torch.float32:
        st = st.astype(np.float32).astype(np.float64)
    p = O.InvertedPendulumParams()
    ctrl = np.clip(act.astype(np.float64), p.ctrl_low, p.ctrl_high)
    sig = np.array([0.01, 0.01, 0.03, 0.03])
    env = E.make(IP[kind], freq_rate=fr, num_envs=n, dtype=dtype, obs_noise_params=(0.01, 0.03))
    env.reset(seed=11)
    cur = st
    for step in range(2):
        env.state = cur
        obs, rew, done, _, _ = env.step(act)
        z = P.obs_noise(n, 4, sig, _noise_seed(11), step, fr)
        ref_state, ref_obs = O.ip_step(cur, ctrl, 0.02, fr, True, p, libm=True, noise=z)
        got = env.state.cpu().numpy().astype(np.float64)
        if dtype == torch.float64:
            assert close64(got, ref_state, 1e-11)
        else:
            big = np.maximum(np.abs(cur), np.abs(ref_state)).astype(np.float32)
            tol = 1e-6 + 1e-5 * np.abs(ref_state) + (fr * 0.5 * np.spacing(big).astype(np.float64) if fr > 1 else 0.0)
            assert (np.abs(got - ref_state) / tol).max() <= 1.0, f"worst fraction of the envelope {(np.abs(got - ref_state) / tol).max()}"
        clean, _ = O.ip_step(cur, ctrl, 0.02, fr, True, p, libm=True)
        d = got - clean
        assert 0.5 * sig[0] < d[:, 0].std() and d[:, 2].std() > 0.5 * sig[2]  # the noise is really there
        assert within32(rew.cpu().numpy(), O.ip_reward(kind, ref_obs)).all()
        cur = got
    # sharding: the second half of the batch as its own env with env_offset = n/2 draws the same noise
    half = E.make(IP[kind], freq_rate=fr, num_envs=n // 2, dtype=dtype, obs_noise_params=(0.01, 0.03), env_offset=n // 2)
    full = E.make(IP[kind], freq_rate=fr, num_envs=n, dtype=dtype, obs_noise_params=(0.01, 0.03))
    half.reset(seed=11)
    full.reset(seed=11)
    half.state, full.state = st[n // 2 :], st
    half.step(act[n // 2 :])
    full.step(act)
    assert torch.equal(half.state, full.state[n // 2 :])
    # (noise inside fused rollouts: test_rollout_ref_equals_step_calls)
    # the host path draws the same noise (ranges keyed by their global env ids, no graph replay with a moving counter)
    h = E.make(IP[kind], freq_rate=fr, num_envs=n, dtype=dtype, obs_noise_params=(0.01, 0.03))
    g = E.make(IP[kind], freq_rate=fr, num_envs=n, dtype=dtype, obs_noise_params=(0.01, 0.03))
    h.reset(seed=11)
    g.reset(seed=11)
    h.state, g.state = st, st
    for _ in range(3):
        o1 = g.step(act)[0]
        o2 = h.step_host(act[:, 0])[0]
        assert np.array_equal(o1.cpu().numpy(), o2)
    assert torch.equal(h.state, g.state)


def test_obs_noise_forms_moments_and_i2p():
    """scalar / dict forms (mujoco_env.py:217-227), the moments of the added noise, the I2P family, and zero noise
    == the plain step bit for bit."""
    from scipy import stats

    n = 1 << 15
    st, act = ip_inputs(4002, n)
    env = E.make(IP["ip_rebound_swingup"], num_envs=n, dtype=torch.float64, obs_noise_params={1: (0.0, 0.05)})
    clean = E.make(IP["ip_rebound_swingup"], num_envs=n, dtype=torch.float64)
    env.reset(seed=3)
    clean.reset(seed=3)
    env.state, clean.state = st, st
    env.step(act)
    clean.step(act)
    d = (env.state - clean.state).cpu().numpy()
    assert np.all(d[:, [0, 1, 2]] == 0.0)  # only joint 1's velocity is noisy
    assert abs(d[:, 3].std() - 0.05) < 0.002 and abs(d[:, 3].mean()) < 0.002
    assert stats.kstest(d[:, 3] / 0.05, "norm").pvalue > 1e-3
    # I2P, float64, scalar form, two sub-steps
    m = 4096
    st6, act6 = i2p_inputs(4003, m)
    p6 = O.I2PParams()
    e6 = E.make(I2P["i2p_boundary_swingup"], freq_rate=2, num_envs=m, dtype=torch.float64, obs_noise_params=0.02)
    e6.reset(seed=5)
    e6.state = st6
    obs6, rew6, done6, _, _ = e6.step(act6)
    z6 = P.obs_noise(m, 6, np.full(6, 0.02), _noise_seed(5), 0, 2)
    ref6, _ = O.i2p_step(st6, act6.astype(np.float64), 0.02, 2, True, p6, libm=True, noise=z6)
    assert close64(e6.state.cpu().numpy(), ref6, 1e-10)
    assert np.allclose(obs6.cpu().numpy(), O.i2p_wrap_obs(e6.state.cpu().numpy()), rtol=0, atol=1e-12)
    # zero noise takes the plain kernels
    e0 = E.make(I2P["i2p_boundary_swingup"], freq_rate=2, num_envs=m, dtype=torch.float64, obs_noise_params=0.0)
    e1 = E.make(I2P["i2p_boundary_swingup"], freq_rate=2, num_envs=m, dtype=torch.float64)
    e0.state, e1.state = st6, st6
    assert torch.equal(e0.step(act6)[0], e1.step(act6)[0])


def test_obs_noise_step_host_multi_range():
    """step_host with obs_noise_params at a size that is cut into two ranges: every range must draw the streams of its
    own global env ids (NoiseParams.env_offset + lo), i.e. equal the single-launch step() bit for bit."""
    n = (1 << 20) + 48
    st, act = ip_inputs(4004, n)
    a = E.make(IP["ip_rebound_swingup"], num_envs=n, dtype=torch.float32, obs_noise_params=0.02)
    b = E.make(IP["ip_rebound_swingup"], num_envs=n, dtype=torch.float32, obs_noise_params=0.02)
    a.reset(seed=2)
    b.reset(seed=2)
    a.state, b.state = st, st
    for _ in range(2):
        o1, r1, d1, _, _ = a.step(act)
        o2, r2, d2, _, _ = b.step_host(act[:, 0])
        assert np.array_equal(o1.cpu().numpy(), o2) and np.array_equal(r1.cpu().numpy(), r2) and np.array_equal(d1.cpu().numpy(), d2)
    assert len(b._staging.ranges) == 2 and not b._staging._graphs


# ================================================================================================
# round 2: trajectory scoring, scoring cache, slices, reset epochs, output ownership
# ================================================================================================
@pytest.mark.parametrize("name,d,a_dim", (("HopperRunning-v0", 12, 3), ("HalfCheetahRunning-v0", 18, 6)))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("T,n", ((1, 256), (5, 1000), (40, 4096), (3, 100), (257, 512)))
def test_sequence_scoring_equals_flat_scoring(name, d, a_dim, dtype, T, n):
    """emei_reward_terminal_seq_* (obs_seq [T+1, n, D]: pre_obs of step t IS obs of step t-1, hopper.py:95-97 /
    half_cheetah.py:60) == emei_reward_terminal_* on separately allocated obs / pre_obs arrays, BIT FOR BIT, for
    one and several time segments, env counts below / above the coalescing minimum and rows that lose 16-byte
    alignment; and == the float64 oracle."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(T * 1000 + n)
    kw = dict(terminate_when_unhealthy=False) if d == 12 else {}
    env = E.make(name, dtype=dtype, **kw)
    seq = torch.randn((T + 1, n, d), device=dev, dtype=dtype, generator=g)
    if d == 12:
        seq[:, :, 1] += 1.25
        seq[:, :, 2:] *= 60.0  # some rows leave the healthy range
    seq.view(-1)[torch.randint(0, seq.numel(), (max(1, seq.numel() // 500),), device=dev, generator=g)] = float("nan")
    act = torch.rand((T, n, a_dim), device=dev, dtype=dtype, generator=g) * 2 - 1
    r_seq, d_seq = env.get_batch_reward_terminal_seq(seq, act)
    assert r_seq.shape == (T, n, 1) and d_seq.shape == (T, n, 1) and d_seq.dtype == torch.bool
    # (a) separately allocated arrays: the ordinary row kernel
    obs, pre = seq[1:].reshape(T * n, d).clone(), seq[:-1].reshape(T * n, d).clone()
    r_flat, d_flat = env.get_batch_reward_terminal(obs, pre, act.reshape(T * n, a_dim))
    assert torch.equal(torch.nan_to_num(r_seq.reshape(-1, 1), nan=7.0), torch.nan_to_num(r_flat, nan=7.0))
    assert torch.equal(d_seq.reshape(-1, 1), d_flat)
    # (b) the two shifted VIEWS of the trajectory through the reference's one-shot signature: the C side recognises
    # pre_obs + n*D == obs and walks the trajectory (n >= 256), same bits either way
    r_v, d_v = env.get_batch_reward_terminal(seq[1:].reshape(T * n, d), seq[:-1].reshape(T * n, d), act.reshape(T * n, a_dim))
    assert torch.equal(torch.nan_to_num(r_v, nan=7.0), torch.nan_to_num(r_flat, nan=7.0)) and torch.equal(d_v, d_flat)
    # (c) the oracle (float64: 1e-12; float32: envelope)
    o64, p64, a64 = (t.double().cpu().numpy() for t in (obs, pre, act.reshape(T * n, a_dim)))
    if d == 12:
        hp = O.HopperParams(terminate_when_unhealthy=False)
        ref_r, ref_d = O.hopper_reward(o64, p64, a64, hp), O.hopper_terminal(o64, hp)
    else:
        hp = O.HalfCheetahParams()
        ref_r, ref_d = O.halfcheetah_reward(o64, p64, a64, hp), O.halfcheetah_terminal(o64)
    got = r_flat.double().cpu().numpy()
    fin = np.isfinite(ref_r)
    if dtype == torch.float64:
        assert close64(got[fin], ref_r[fin], 1e-11)
    else:
        assert np.all(np.abs(got[fin] - ref_r[fin]) <= 1e-4 * (1.0 + np.abs(ref_r[fin])))  # (o - p)/dt amplifies float32 rounding by 1/dt
    assert np.array_equal(d_flat.cpu().numpy(), ref_d)


def test_sequence_scoring_statistics_and_other_families():
    """the trajectory entry point accumulates the same statistics as the flat one and accepts every family (families
    without a pre_obs term score obs_seq[1:] row by row)."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(5)
    T, n = 6, 2048
    hop = E.make("HopperRunning-v0", dtype=torch.float64, terminate_when_unhealthy=False)
    hop.accumulate_scoring_stats = True
    seq = torch.randn((T + 1, n, 12), device=dev, dtype=torch.float64, generator=g)
    seq[:, :, 1] += 1.25
    act = torch.rand((T, n, 3), device=dev, dtype=torch.float64, generator=g)
    hop.reset_stats()
    r, d = hop.get_batch_reward_terminal_seq(seq, act)
    rs, dc = hop.read_stats()
    assert dc == int(d.sum()) and abs(rs - float(r.sum())) < 1e-9 * max(1.0, abs(rs))
    cp = E.make("CartPoleSwingUp-v0", dtype=torch.float64)
    from emei_b200.engine import score_seq

    s4 = torch.randn((T + 1, n, 4), device=dev, dtype=torch.float64, generator=g) * 3
    r4, d4, _ = score_seq(cp, cp._scoring_params(), s4)
    r_ref, d_ref = cp.get_batch_reward_terminal(s4[1:].reshape(-1, 4).clone())
    assert torch.equal(r4.reshape(-1, 1), r_ref) and torch.equal(d4.reshape(-1, 1), d_ref)


def test_scoring_pair_shares_one_pass_and_slices_are_accepted():
    """The reference's API is two calls (get_batch_reward, get_batch_terminal): made back to back on the same device
    tensors they cost ONE fused pass; an in-place change of an input, or any other emei launch in between, voids the
    cache.  Contiguous slices that start at an odd byte offset (12-byte action rows, 72-byte observation rows) are
    accepted like the reference accepts them."""
    from emei_b200 import _lib

    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(3)
    n = 5000
    env = E.make("HalfCheetahRunning-v0", dtype=torch.float32)
    obs = torch.randn((n, 18), device=dev, generator=g)
    pre = torch.randn((n, 18), device=dev, generator=g)
    act = torch.rand((n, 6), device=dev, generator=g)
    c0 = _lib.launch_count
    r1 = env.get_batch_reward(obs, pre, act)
    c1 = _lib.launch_count
    d1 = env.get_batch_terminal(obs, pre, act)
    assert c1 - c0 == 2 and _lib.launch_count == c1  # sumsq + rows once; the terminal call is served from that pass
    d1b = env.get_batch_terminal(obs)  # the pass is served ONCE: this call runs the row kernel again
    assert _lib.launch_count == c1 + 1
    env.get_batch_reward(obs, pre, act)
    c1 = _lib.launch_count
    assert torch.equal(env.get_batch_terminal(obs), d1) and _lib.launch_count == c1  # obs alone identifies the flags
    env.get_batch_reward(obs, pre, act)
    c1 = _lib.launch_count
    env.get_batch_reward(obs, pre, act)  # the SAME half again is never served from the cache
    assert _lib.launch_count == c1 + 2
    r2, d2 = env.get_batch_reward_terminal(obs.clone(), pre.clone(), act.clone())
    assert torch.equal(r1, r2) and torch.equal(d1, d2) and torch.equal(d1b, d2)
    env.get_batch_reward(obs, pre, act)  # the cache now holds THIS triple
    obs[0, 0] = float("nan")  # torch bumps the tensor's version: the cached pass must not be served
    d3 = env.get_batch_terminal(obs, pre, act)
    assert bool(d3[0, 0]) and not bool(d1[0, 0])
    env.get_batch_reward(obs, pre, act)
    E.make("CartPoleSwingUp-v0", num_envs=8).reset(seed=0)  # any other emei launch in between voids it too
    c2 = _lib.launch_count
    env.get_batch_terminal(obs, pre, act)
    assert _lib.launch_count > c2
    # odd-offset slices
    k = 3
    r_s, d_s = env.get_batch_reward_terminal(obs[k:], pre[k:], act[k:])
    r_c, d_c = env.get_batch_reward_terminal(obs[k:].clone(), pre[k:].clone(), act[k:].clone())
    assert torch.equal(torch.nan_to_num(r_s), torch.nan_to_num(r_c)) and torch.equal(d_s, d_c)
    hop = E.make("HopperRunning-v0", dtype=torch.float32)
    o12, a3 = torch.randn((n, 12), device=dev, generator=g), torch.rand((n, 3), device=dev, generator=g)
    r_s = hop.get_batch_reward(o12[1:], o12[:-1], a3[1:])
    r_c = hop.get_batch_reward(o12[1:].clone(), o12[:-1].clone(), a3[1:].clone())
    assert torch.equal(r_s, r_c)


def test_unseeded_resets_change_the_rollout_streams():
    """reset() zeroes the episode / step counters of the counter-based streams, so every un-seeded reset must move to
    a fresh stream: `env.reset(); env.rollout(T)` cycles (offline.collect_dataset) must not replay the same random
    actions; reset(seed=s) restarts the sequence of streams reproducibly."""
    from oracle import rollout_oracle as RO

    n, T = 512, 16
    env = E.make("ContinuousCartPoleSwingUp-v0", num_envs=n, freq_rate=1)
    env.reset(seed=21)
    a0 = env.rollout(T, record=True)["actions"].clone()
    env.reset()
    a1 = env.rollout(T, record=True)["actions"].clone()
    env.reset()
    a2 = env.rollout(T, record=True)["actions"].clone()
    assert not torch.equal(a0, a1) and not torch.equal(a1, a2) and not torch.equal(a0, a2)
    _, sa1 = RO.rollout_seeds(21, epoch=1)
    assert np.array_equal(a1.cpu().numpy(), RO.random_actions(sa1, n, 0, T, True, -1.0, 1.0))
    env.reset(seed=21)
    b0 = env.rollout(T, record=True)["actions"].clone()
    env.reset()
    b1 = env.rollout(T, record=True)["actions"].clone()
    assert torch.equal(a0, b0) and torch.equal(a1, b1)


def test_rollout_action_validation_matches_step():
    env = E.make("CartPoleSwingUp-v0", num_envs=64, validate_actions=True)
    env.reset(seed=1)
    with pytest.raises(AssertionError):
        env.rollout(4, actions=torch.zeros((4, 64), dtype=torch.float32, device="cuda"))  # floats for Discrete(2)
    with pytest.raises(AssertionError):
        env.rollout(4, actions=torch.full((4, 64), 2, dtype=torch.int64, device="cuda"))  # outside the space
    a16 = torch.randint(0, 2, (4, 64), dtype=torch.int16, device="cuda")  # unsupported width: cast, not KeyError
    env2 = E.make("CartPoleSwingUp-v0", num_envs=64)
    env2.reset(seed=1)
    env.reset(seed=1)
    env.rollout(4, actions=a16)
    env2.rollout(4, actions=a16.to(torch.int64))
    assert torch.equal(env.state, env2.state)


@pytest.mark.parametrize("env_id", ("ContinuousCartPoleSwingUp-v0", "BoundaryInvertedPendulumSwingUp-v0", "ChargedBallCentering-v0",
                                    "BoundaryInvertedDoublePendulumSwingUp-v0"))
def test_step_outputs_are_owned_by_the_caller_by_default(env_id):
    """The reference returns `self.state.copy()` (base_control.py:47,69,76): by default what step() returns is the
    caller's -- the next step does not overwrite it and writing into it does not touch the env; copy_outputs=False is
    the zero-copy opt-in with the documented lifetime."""
    n = 9000
    env = E.make(env_id, num_envs=n)
    obs0, _ = env.reset(seed=4)
    a = env.action_space.sample_batch(n)
    o1, r1, d1, _, _ = env.step(a)
    keep = (o1.clone(), r1.clone(), d1.clone())
    o2, _, _, _, _ = env.step(a)
    env.step(a)
    assert torch.equal(o1, keep[0]) and torch.equal(r1, keep[1]) and torch.equal(d1, keep[2])
    assert o2.data_ptr() != o1.data_ptr()
    ref = E.make(env_id, num_envs=n)
    ref.reset(seed=4)
    for _ in range(3):
        ref.step(a)
    o2.zero_()  # the caller scribbles over what it was given: the env must not notice
    assert all(torch.equal(x, y) for x, y in zip(_state_tensors(env), _state_tensors(ref)))
    fast = E.make(env_id, num_envs=n, copy_outputs=False)
    fast.reset(seed=4)
    of, rf, df, _, _ = fast.step(a)
    assert torch.equal(of, keep[0]) and torch.equal(rf, keep[1])


def _state_tensors(env):
    st = env.state
    return list(st.values()) if isinstance(st, dict) else [st]


# ================================================================================================
# round 2: rollouts in the step entry points' arithmetic (float64, inverted double pendulum, obs_noise_params)
# ================================================================================================
def _device_reset_rows(env, kind, seed_reset, ep_idx_value, n, dtype):
    """Expected in-kernel reset samples of ALL n envs for one episode index, produced by the emei_init_* kernels
    (the reference-arithmetic rollout kernel uses their arithmetic: bit-identical) -- and pinned to the host Philox
    mirror of oracle/philox.py."""
    import ctypes

    seed = (seed_reset + ep_idx_value * RO.RESET_STRIDE) & RO.MASK64
    dev = env.device
    npdt = np.float64 if dtype == torch.float64 else np.float32
    if kind == "uniform":
        pi_col = 2 if "SwingUp" in type(env).__name__ else -1
        out = torch.empty((n, 4), dtype=dtype, device=dev)
        env._call("emei_init_uniform", out.data_ptr(), n, 4, -0.05, 0.05, pi_col, ctypes.c_uint64(seed), ctypes.c_uint64(env.env_offset), env._stream())
        assert np.array_equal(out.cpu().numpy(), P.init_uniform(n, 4, -0.05, 0.05, pi_col, seed, env.env_offset, dtype=npdt))
        return out
    if kind == "gaussian":
        mean, sigma = env._init_tables()
        d = mean.shape[0]
        out = torch.empty((n, d), dtype=dtype, device=dev)
        Arr = ctypes.c_double * d
        env._call("emei_init_gaussian", out.data_ptr(), n, d, Arr(*mean), Arr(*sigma), ctypes.c_uint64(seed), ctypes.c_uint64(env.env_offset), env._stream())
        host = P.init_gaussian(n, d, mean, sigma, seed, env.env_offset)
        assert np.allclose(out.double().cpu().numpy(), host, rtol=0, atol=1e-12 if dtype == torch.float64 else 1e-7)
        return out
    on = torch.empty((n,), dtype=torch.uint8, device=dev)
    ci = torch.empty((n, 2), dtype=dtype, device=dev)
    fr = torch.empty((n, 4), dtype=dtype, device=dev)
    env._call("emei_init_charged_ball", on.data_ptr(), ci.data_ptr(), fr.data_ptr(), n, 1.0, ctypes.c_uint64(seed), ctypes.c_uint64(env.env_offset), env._stream())
    h_on, h_ci, h_fr = P.init_charged_ball(n, 1.0, seed, env.env_offset, dtype=npdt)
    assert np.array_equal(ci.cpu().numpy(), h_ci) and np.allclose(fr.cpu().numpy(), h_fr, rtol=0, atol=1e-15 if dtype == torch.float64 else 1e-7)
    return dict(on_circle=on, circle_state=ci, free_state=fr)


@pytest.mark.parametrize("env_id,dtype,kw,reset_kind,max_steps", (
    ("CartPoleSwingUp-v0", torch.float64, dict(freq_rate=4), "uniform", 7),
    ("ContinuousCartPoleBalancing-v0", torch.float64, dict(freq_rate=1), "uniform", 5),
    ("BoundaryInvertedPendulumSwingUp-v0", torch.float64, dict(freq_rate=2), "gaussian", 6),
    ("BoundaryInvertedPendulumSwingUp-v0", torch.float64, dict(freq_rate=2, obs_noise_params=(0.01, 0.05)), "gaussian", 6),
    ("ReboundInvertedPendulumBalancing-v0", torch.float32, dict(freq_rate=3, obs_noise_params=0.02), "gaussian", 6),
    ("BoundaryInvertedDoublePendulumSwingUp-v0", torch.float32, dict(freq_rate=1), "gaussian", 6),
    ("BoundaryInvertedDoublePendulumBalancing-v0", torch.float64, dict(freq_rate=2), "gaussian", 6),
    ("ReboundInvertedDoublePendulumSwingUp-v0", torch.float64, dict(freq_rate=2, obs_noise_params=(0.01, 0.03)), "gaussian", 6),
    ("ReboundInvertedDoublePendulumBalancing-v0", torch.float32, dict(freq_rate=1, obs_noise_params=0.01), "gaussian", 6),
    ("ChargedBallCentering-v0", torch.float64, dict(freq_rate=2), "charged_ball", 8),
    ("ContinuousChargedBallCentering-v0", torch.float64, dict(freq_rate=1), "charged_ball", 8),
))
@pytest.mark.parametrize("policy", ("teacher", "random"))
def test_rollout_ref_equals_step_calls(env_id, dtype, kw, reset_kind, max_steps, policy):
    """emei_cartpole_rollout_ref_* / emei_i2p_rollout_* / emei_charged_ball_rollout_ref_f64 (zoo/util.py:33-93 in one
    launch, in the arithmetic of the step entry points): every recorded transition equals the step call of a twin env
    BIT FOR BIT -- float64 reference-exact mode, the four inverted-double-pendulum tasks, and obs_noise_params with
    its step counter continued through the rollout (mujoco_env.py:98-104) -- the TimeLimit / done / auto-reset
    bookkeeping equals the restated loop, in-kernel resets equal the emei_init_* kernels (pinned to the Philox mirror),
    a horizon split over two launches continues state, counters and streams, and records on == records off."""
    n, T = 640, 20
    a = E.make(env_id, num_envs=n, dtype=dtype, **kw)
    b = E.make(env_id, num_envs=n, dtype=dtype, **kw)   # split horizon, no records
    twin = E.make(env_id, num_envs=n, dtype=dtype, **kw)
    for e in (a, b, twin):
        e.reset(seed=8)
    cont = len(a.action_space.shape) > 0
    rng = np.random.default_rng(2)
    acts = None
    if policy == "teacher":
        lo, hi = (float(a.action_space.low[0]), float(a.action_space.high[0])) if cont else (0, 2)
        acts = rng.uniform(lo, hi, size=(T, n)).astype(np.float32) if cont else rng.integers(0, 2, size=(T, n)).astype(np.int64)
    out = a.rollout(T, actions=acts, record=True, max_episode_steps=max_steps)
    b.rollout(T // 2, actions=None if acts is None else acts[: T // 2], max_episode_steps=max_steps)
    b.rollout(T - T // 2, actions=None if acts is None else acts[T // 2 :], max_episode_steps=max_steps)
    assert _same_state(a.state, b.state)
    for k in ("ep_step", "ep_index", "ep_return"):
        assert torch.equal(getattr(a._engine, k), getattr(b._engine, k)), k
    rec = {k: v for k, v in out.items() if k != "stats"}
    assert rec["observations"].dtype == dtype and rec["rewards"].dtype == dtype
    D = rec["observations"].shape[2]
    assert D == (6 if "Double" in env_id else 4)
    if policy == "random":
        seed_reset, seed_action = RO.rollout_seeds(8)
        lo, hi = (float(a.action_space.low[0]), float(a.action_space.high[0])) if cont else (-1.0, 1.0)
        ref_a = RO.random_actions(seed_action, n, 0, T, cont, lo, hi)
        assert np.array_equal(rec["actions"].cpu().numpy(), ref_a)
        acts = ref_a
    else:
        seed_reset, _ = RO.rollout_seeds(8)
        assert np.array_equal(rec["actions"].cpu().numpy(), acts)
    ep_step, ep_idx = np.zeros(n, np.int64), np.zeros(n, np.int64)
    ep_ret = torch.zeros(n, dtype=dtype, device=a.device)
    fin = n_trunc = 0
    cache = {}
    for t in range(T):
        # the recorded observation: what the previous step returned, except on rows that were just reset (their
        # observation is re-derived from the fresh state: compared with the env's own current_obs formula)
        cur = twin.current_obs if hasattr(type(twin), "current_obs") else (twin.state["free_state"] if isinstance(twin.state, dict) else twin.state)
        assert torch.allclose(rec["observations"][t], cur, rtol=0, atol=1e-12 if dtype == torch.float64 else 2e-6), f"observation at step {t}"
        if t > 0:
            keep = torch.as_tensor(~prev_done, device=a.device)
            assert torch.equal(rec["observations"][t][keep], rec["next_observations"][t - 1][keep])
        if hasattr(twin, "_noise_step"):
            twin._noise_step = t  # the rollout continues the noise stream's step counter
        act_t = torch.as_tensor(acts[t]).to(a.device)
        o2, r2, d2, _, _ = twin.step(act_t.reshape(n, 1) if cont else act_t)
        assert torch.equal(rec["next_observations"][t], o2), f"next_observation at step {t}"
        assert torch.equal(rec["rewards"][t], r2[:, 0])
        term = d2[:, 0].cpu().numpy()
        ep_step = ep_step + 1
        ep_ret = ep_ret + r2[:, 0]
        trunc = ep_step >= max_steps
        done = term | trunc
        assert np.array_equal(rec["dones"][t].cpu().numpy(), done) and np.array_equal(rec["timeouts"][t].cpu().numpy(), trunc)
        idx = np.nonzero(done)[0]
        prev_done = done
        fin += idx.size
        n_trunc += int(trunc.sum())
        ep_idx[idx] += 1
        for epv in np.unique(ep_idx[idx]):  # resets: rows of the init kernels' samples for that episode index
            rows = idx[ep_idx[idx] == epv]
            if (epv,) not in cache:
                cache[(epv,)] = _device_reset_rows(twin, reset_kind, seed_reset, int(epv), n, dtype)
            fresh = cache[(epv,)]
            sel = torch.as_tensor(rows, device=a.device)
            if isinstance(fresh, dict):
                st = twin.state
                for kk in fresh:
                    st[kk][sel] = fresh[kk][sel]
            else:
                twin.state[sel] = fresh[sel]
        ep_step[idx] = 0
        ep_ret[torch.as_tensor(idx, device=a.device)] = 0
    assert fin > 0 and n_trunc > 0
    assert _same_state(a.state, twin.state)
    assert np.array_equal(a._engine.ep_step.cpu().numpy(), ep_step) and np.array_equal(a._engine.ep_index.cpu().numpy(), ep_idx)
    assert torch.equal(a._engine.ep_return, ep_ret)
    info = a.rollout_info(out["stats"])
    assert info["total_episode_num"] == fin and info["truncated"] == n_trunc
    rs = float(rec["rewards"].double().sum())
    assert abs(info["reward_sum"] - rs) <= 1e-9 * max(1.0, abs(rs)) + (1e-3 if dtype == torch.float32 else 0.0)


@pytest.mark.parametrize("env_id,n", (("ContinuousCartPoleSwingUp-v0", 1_100_003), ("ChargedBallCentering-v0", 4096),
                                      ("BoundaryInvertedDoublePendulumSwingUp-v0", 300_000)))
def test_step_host_outputs_selector(env_id, n):
    """step_host(action, outputs=...) downloads only what the caller consumes (5 bytes per env for reward + done instead
    of 21): same state evolution, same values, None for what stays on the device -- eager and as a replayed graph."""
    rng = np.random.default_rng(6)
    a = E.make(env_id, num_envs=n, dtype=torch.float32)
    b = E.make(env_id, num_envs=n, dtype=torch.float32)
    a.reset(seed=12)
    b.reset(seed=12)
    cont = len(a.action_space.shape) > 0
    lo, hi = (float(a.action_space.low[0]), float(a.action_space.high[0])) if cont else (0, 2)
    act = torch.as_tensor(rng.uniform(lo, hi, size=n).astype(np.float32) if cont else rng.integers(0, 2, size=n).astype(np.uint8)).pin_memory()
    for t in range(8):  # the same pinned buffer: eager, captured, replayed
        o1, r1, d1, _, _ = a.step_host(act)
        o2, r2, d2, _, _ = b.step_host(act, outputs=("reward", "done"))
        assert o2 is None and np.array_equal(r1, r2, equal_nan=True) and np.array_equal(d1, d2)
        assert b._staging.d2h_bytes == 5 * n and a._staging.d2h_bytes == (4 * o1.shape[1] + 5) * n
    o3, r3, d3, _, _ = b.step_host(act, outputs=("obs",))
    o4, _, _, _, _ = a.step_host(act)
    assert r3 is None and d3 is None and np.array_equal(o3, o4, equal_nan=True)
    assert _same_state(a.state, b.state)
    with pytest.raises(ValueError):
        b.step_host(act, outputs=("observation",))


def test_random_policy_test_mirror():
    """emei/util.py:5-41 batched (emei_b200.util.random_policy_test): the reference's report line, the random and the
    constant-action policy, a bounded run."""
    from emei_b200.util import random_policy_test

    env = E.make("CartPoleBalancing-v0", num_envs=256, dtype=torch.float32)
    lines = []
    rep = random_policy_test(env, report_every=50, max_steps=100, out=lines.append)
    assert len(rep) == 2 and sum(r["total_episode_num"] for r in rep) > 0
    assert lines and lines[0].startswith("episode length: ") and "\tepisode rewards: " in lines[0]
    rep = random_policy_test(env, default_action=1, report_every=40, max_steps=40, out=lines.append)
    assert rep[0]["total_episode_num"] >= env.num_envs  # pushing right at every step ends every episode within 40 steps
    assert rep[0]["terminated"] >= env.num_envs and rep[0]["avg_length"] < 40
    with pytest.raises(NotImplementedError):
        random_policy_test(env, is_render=True)


@pytest.mark.parametrize("env_id,cont", (("ChargedBallCentering-v0", False), ("ContinuousCartPoleSwingUp-v0", True)))
def test_rollout_with_host_actions_is_pipelined_and_equal(env_id, cont, monkeypatch):
    """Teacher-forced rollouts whose actions are HOST arrays are cut into pieces (uploads one piece ahead of the kernels):
    same final state, counters and statistics as one launch over the same actions on the device."""
    n, T = 3000, 40
    rng = np.random.default_rng(9)
    acts = rng.uniform(-1, 1, size=(T, n)).astype(np.float32) if cont else rng.integers(0, 2, size=(T, n)).astype(np.uint8)
    a = E.make(env_id, num_envs=n, dtype=torch.float32)
    b = E.make(env_id, num_envs=n, dtype=torch.float32)
    a.reset(seed=4)
    b.reset(seed=4)
    monkeypatch.setattr(type(b), "_ROLLOUT_PIECE_BYTES", 3 * acts[0].nbytes)  # pieces of 3 steps: 14 launches, a ragged last one
    monkeypatch.setattr(type(b), "_ROLLOUT_PIECE_MIN_STEPS", 1)
    launches0 = E._lib.launch_count
    out_b = b.rollout(T, actions=torch.as_tensor(acts).pin_memory(), max_episode_steps=7)
    assert E._lib.launch_count - launches0 == 14
    out_a = a.rollout(T, actions=torch.as_tensor(acts).cuda(), max_episode_steps=7)
    assert _same_state(a.state, b.state)
    assert torch.allclose(out_a["stats"], out_b["stats"], rtol=1e-12, atol=0)
    for k in ("ep_step", "ep_index", "ep_return"):
        assert torch.equal(getattr(a._engine, k), getattr(b._engine, k)), k
    out_c = b.rollout(T, actions=acts, max_episode_steps=7)  # pageable numpy actions take the same path
    out_d = a.rollout(T, actions=torch.as_tensor(acts).cuda(), max_episode_steps=7)
    assert _same_state(a.state, b.state) and torch.allclose(out_c["stats"], out_d["stats"], rtol=1e-12, atol=0)
