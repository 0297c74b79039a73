"""Offline datasets for every task that rolls out (zoo/util.py:33-93,108-111): the wide records transposes at the
edges of alignment and 32-bit offsets against torch (every element size at every shape: test_records_transpose_bit_exact),
and ``collect_dataset`` checked against the rollout's records, a host restatement of the
collection loop and, where the observation determines the state, the float64 oracle transition by transition.

Observation records are D x sizeof(real) bytes per element: 16 (float32 cart-pole, inverted pendulum, charged ball),
24 (float32 inverted double pendulum), 32 (float64, D = 4) and 48 (float64 inverted double pendulum)."""
import numpy as np
import pytest
import torch

from oracle import emei_oracle as O
from oracle import philox as P
from oracle import rollout_oracle as RO

pytestmark = pytest.mark.gpu

import emei_b200 as E  # noqa: E402
from emei_b200 import _lib, offline  # noqa: E402

CARTPOLE = {"CartPoleBalancing-v0": "balancing", "CartPoleSwingUp-v0": "swingup",
            "ContinuousCartPoleBalancing-v0": "continuous_balancing", "ContinuousCartPoleSwingUp-v0": "continuous_swingup"}
IP = {"ReboundInvertedPendulumBalancing-v0": "ip_rebound_balancing", "BoundaryInvertedPendulumBalancing-v0": "ip_boundary_balancing",
      "ReboundInvertedPendulumSwingUp-v0": "ip_rebound_swingup", "BoundaryInvertedPendulumSwingUp-v0": "ip_boundary_swingup"}
I2P = ("ReboundInvertedDoublePendulumBalancing-v0", "BoundaryInvertedDoublePendulumBalancing-v0",
       "ReboundInvertedDoublePendulumSwingUp-v0", "BoundaryInvertedDoublePendulumSwingUp-v0")
CHARGED_BALL = ("ChargedBallCentering-v0", "ContinuousChargedBallCentering-v0")
ROLLOUT_ENVS = tuple(CARTPOLE) + tuple(IP) + I2P + CHARGED_BALL
SEED = 4


def close64(a, b, tol=1e-12):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))


def within32(a, ref, scale=1.0):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(a - ref) <= scale * (1e-6 + 1e-5 * np.abs(ref))


# ================================================================================================
# emei_records_transpose against torch, bit for bit
# ================================================================================================
def _records(shape, dtype, seed):
    """random bits of the given dtype (floats through their integer twins: every bit pattern, NaNs included)"""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    if dtype == torch.uint8:
        return torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=g)
    bits = {torch.float32: torch.int32, torch.float64: torch.int64}[dtype]
    info = torch.iinfo(bits)
    return torch.randint(info.min, info.max, shape, dtype=bits, device="cuda", generator=g).view(dtype)


def _transpose_cabi(x):
    """[T, n, ...] -> [n, T, ...] through the C ABI itself (a refused element size is an error code, not a ValueError)"""
    T, n = x.shape[0], x.shape[1]
    elem = x.element_size() * int(np.prod(x.shape[2:], dtype=np.int64))
    out = torch.empty((n, T) + tuple(x.shape[2:]), dtype=x.dtype, device=x.device)
    code = _lib.lib.emei_records_transpose(x.data_ptr(), out.data_ptr(), T, n, elem, torch.cuda.current_stream().cuda_stream)
    assert code == 0, f"emei_records_transpose({elem}-byte elements) returned {code}"
    return out


def _bits(t):
    return t.view({1: torch.uint8, 4: torch.int32, 8: torch.int64}[t.element_size()])


def test_records_transpose_24_byte_rows_at_8_byte_alignment():
    """a [T, n, 6] float32 tensor is only 8-byte aligned when it starts at an odd pair of floats: the 24-byte path must
    take it (its words are 8 bytes), and write to an 8-byte aligned output too"""
    T, n = 37, 301
    buf = _records((T * n * 6 + 2,), torch.float32, 5)
    x = buf[2:].view(T, n, 6)
    assert x.data_ptr() % 16 == 8
    want = _bits(x).transpose(0, 1).contiguous()
    out_buf = torch.full((n * T * 6 + 4,), -1, dtype=torch.int32, device="cuda")
    out = out_buf[2:-2]
    assert out.data_ptr() % 16 == 8
    code = _lib.lib.emei_records_transpose(x.data_ptr(), out.data_ptr(), T, n, 24, torch.cuda.current_stream().cuda_stream)
    assert code == 0
    assert torch.equal(out.view(n, T, 6), want)
    assert (out_buf[:2] == -1).all() and (out_buf[-2:] == -1).all()  # nothing written outside the output


def test_records_transpose_past_4gib_offsets():
    """48-byte elements, T = 1024, n = 2^17 + 3: about 6.4 GB each way, so the byte offsets of the later rows pass 2^32"""
    T, n = 1024, (1 << 17) + 3
    assert T * n * 48 > (1 << 32)
    x = _records((T, n, 6), torch.float64, 11)
    got = _transpose_cabi(x)
    want = _bits(x).transpose(0, 1).contiguous()
    assert torch.equal(_bits(got), want)
    del got, want, x
    torch.cuda.empty_cache()


# ================================================================================================
# collect_dataset: layout, episodes, values
# ================================================================================================
def _max_steps(env_id):
    # a limit by which some of the balancing tasks' episodes have ended by themselves under random pushes and some not
    # (oracle from the reset distribution, freq_rate 1: the rebound double pendulum falls within 4 steps in 40 % of the
    # episodes, the boundary pendulum within 20 in 11 %, the others within 16 in 14-47 %)
    if env_id == "ReboundInvertedDoublePendulumBalancing-v0":
        return 4
    return 20 if env_id == "BoundaryInvertedPendulumBalancing-v0" else 16


def _teacher_actions(env, T, n, seed):
    rng = np.random.default_rng(seed)
    if len(env.action_space.shape) > 0:
        lo, hi = float(env.action_space.low[0]), float(env.action_space.high[0])
        return rng.uniform(lo, hi, size=(T, n)).astype(np.float32)
    return rng.integers(0, 2, size=(T, n)).astype(np.int64)


def _reset_rows(env_id, dtype, env, seed_reset, ep, ids, n):
    """observations of envs ``ids`` at the start of their ep-th in-rollout episode, from the host Philox mirror:
    (rows [len(ids), D] float64, absolute tolerance).  The float64 rollouts sample like the emei_init_* kernels
    (P.init_*, all n envs at once), the packed float32 rollouts of cart-pole, inverted pendulum and charged ball with
    their own lean samplers (RO.reset_sample_*, env by env)."""
    f64 = dtype == torch.float64
    s = (seed_reset + ep * RO.RESET_STRIDE) & RO.MASK64
    eps = np.full(len(ids), ep)
    if env_id in CARTPOLE:
        pi_col = 2 if "SwingUp" in env_id else -1
        if f64:
            return P.init_uniform(n, 4, -0.05, 0.05, pi_col, s)[ids], 0.0
        return RO.reset_sample_uniform(ids, eps, seed_reset, pi_column=pi_col).astype(np.float64), 0.0
    if env_id in CHARGED_BALL:
        if f64:
            return P.init_charged_ball(n, 1.0, s)[2][ids], 1e-15
        return RO.reset_sample_charged_ball(ids, eps, seed_reset)[2].astype(np.float64), 3e-7
    mean, sigma = env._init_tables()
    if env_id in IP:
        if f64:
            rows = P.init_gaussian(n, 4, mean, sigma, s)[ids]
        else:
            rows = RO.reset_sample_gaussian(ids, eps, seed_reset, mean, sigma).astype(np.float64)
        rows[:, 1] = O.ip_wrap_angle(rows[:, 1])
        return rows, (1e-12 if f64 else 1e-9)
    # the inverted double pendulum's rollout samples like init_gaussian_kernel in both precisions
    rows = P.init_gaussian(n, 6, mean, sigma, s, dtype=np.float64 if f64 else np.float32)[ids].astype(np.float64)
    return O.i2p_wrap_obs(rows), (1e-12 if f64 else 2e-6)


def _check_values(env_id, dtype, env, ds, fr):
    """every transition teacher-forced from its recorded observation through the float64 oracle"""
    obs, nxt = ds["observations"].astype(np.float64), ds["next_observations"]
    act, rew, dones, tmo = ds["actions"], ds["rewards"], ds["dones"].astype(bool), ds["timeouts"].astype(bool)
    f64 = dtype == torch.float64
    if env_id in CARTPOLE:
        kind = CARTPOLE[env_id]
        cont = kind.startswith("continuous")
        p = O.cartpole_params(kind)
        ref = O.cartpole_step_f64ref(obs, O.cartpole_force(act if cont else act.astype(np.int64), cont, p), 0.02, fr, p)
        if f64:  # DESIGN section 2: <= 1e-12 relative to max(1, |value|)
            assert close64(nxt, ref).all()
            assert close64(rew, O.cartpole_reward(kind, ref)[:, 0]).all()
        else:
            assert within32(nxt, ref).all()
            assert within32(rew, O.cartpole_reward(kind, ref)[:, 0]).all()
        term = O.cartpole_terminal(kind, ref, p)[:, 0]
        near = (np.abs(np.abs(ref[:, 0]) - p.x_threshold) < 1e-4) | (np.abs(np.abs(ref[:, 2]) - p.theta_threshold_radians) < 1e-4)
    else:
        kind = IP[env_id]
        p = O.InvertedPendulumParams()
        ctrl = np.clip(act.astype(np.float64).reshape(-1), p.ctrl_low, p.ctrl_high)
        # from the wrapped observation: the state's angle differs from it by a multiple of 2 pi, which moves sin / cos by
        # a few ulp(theta); the angles here stay within a few turns, so that is far below the 1e-12 bar
        _, ref = O.ip_step(obs, ctrl, 0.02, fr, kind.endswith("swingup"), p, libm=True)
        dth = np.abs((nxt[:, 1].astype(np.float64) - ref[:, 1] + np.pi) % (2 * np.pi) - np.pi)  # on the circle
        assert np.all((nxt[:, 1] >= -np.pi) & (nxt[:, 1] <= np.pi))
        cols = [0, 2, 3]
        if f64:
            assert np.all(dth <= 1e-12) and close64(nxt[:, cols], ref[:, cols]).all()
            assert close64(rew, O.ip_reward(kind, ref)[:, 0]).all()
        else:
            assert np.all(dth <= 1e-6 + 1e-5 * np.abs(ref[:, 1])) and within32(nxt[:, cols], ref[:, cols]).all()
            assert within32(rew, O.ip_reward(kind, ref)[:, 0], 2.0).all()
        term = O.ip_terminal(kind, ref, p)[:, 0]
        cy = np.cos(ref[:, 1])
        near = (np.abs(np.abs(ref[:, 0]) - 2.0) < 1e-4) | (np.abs(cy - 0.9) < 1e-4) | (np.abs(cy) < 1e-4)
    # flags: exact away from the threshold bands; a timeout ends the episode whatever the terminal flag says
    free = ~near & ~tmo
    assert np.array_equal(dones[free], term[free])
    assert dones[tmo].all()


def _collect_and_check(env_id, dtype, policy, n, T):
    mes = _max_steps(env_id)
    env = E.make(env_id, num_envs=n, dtype=dtype)
    twin = E.make(env_id, num_envs=n, dtype=dtype)
    for e in (env, twin):
        e.max_episode_steps = mes
        e.reset(seed=SEED)
    acts = _teacher_actions(env, T, n, 7) if policy == "teacher" else None
    samples, info = offline.collect_dataset(env, n * T, actions=acts)
    # the twin repeats collect_dataset's seed history: reset(seed) then one un-seeded reset (stream epoch 1)
    twin.reset()
    rec = twin.rollout(T, actions=acts, record=True)
    D = 6 if env_id in I2P else 4
    npdt = np.float64 if dtype == torch.float64 else np.float32
    cont = len(env.action_space.shape) > 0
    N = n * T

    # ---- layout: the dataset is the records, transposed; env-major = time-major re-laid out
    ds_env = {k: v.cpu().numpy() for k, v in offline.records_to_dataset(rec, "env").items()}
    ds_time = {k: v.cpu().numpy() for k, v in offline.records_to_dataset(rec, "time").items()}
    assert sorted(samples) == sorted(offline.KEYS)
    for k in offline.KEYS:
        assert samples[k].dtype == ds_env[k].dtype and np.array_equal(samples[k], ds_env[k], equal_nan=True), k
        tail = samples[k].shape[1:]
        by_env = ds_env[k].reshape((n, T) + tail)
        by_time = ds_time[k].reshape((T, n) + tail)
        assert np.array_equal(by_env, by_time.swapaxes(0, 1), equal_nan=True), k  # ds_env[i*T + t] == ds_time[t*n + i]
        r = rec[k].cpu().numpy()
        if k in ("dones", "timeouts"):
            r = r.astype(np.float32)
        assert np.array_equal(by_time, r.reshape(by_time.shape), equal_nan=True), k
    assert samples["observations"].shape == (N, D) and samples["next_observations"].shape == (N, D)
    assert samples["observations"].dtype == npdt and samples["next_observations"].dtype == npdt
    assert samples["rewards"].shape == (N,)
    assert samples["dones"].dtype == np.float32 and samples["timeouts"].dtype == np.float32
    assert samples["dones"].shape == (N,) and samples["timeouts"].shape == (N,)
    assert set(np.unique(samples["dones"])) <= {0.0, 1.0} and set(np.unique(samples["timeouts"])) <= {0.0, 1.0}
    assert samples["actions"].shape == ((N, 1) if cont else (N,))
    if acts is not None:
        assert np.array_equal(samples["actions"].reshape(n, T).T, acts.astype(samples["actions"].dtype))

    # ---- episodes, against the restated loop: every env's run is contiguous in the env-major dataset
    obs = samples["observations"].reshape(n, T, D)
    nxt = samples["next_observations"].reshape(n, T, D)
    dones = samples["dones"].reshape(n, T).astype(bool)
    tmo = samples["timeouts"].reshape(n, T).astype(bool)
    rew = samples["rewards"].reshape(n, T).astype(np.float64)
    assert not (tmo & ~dones).any()  # timeouts => dones
    ep_len = np.zeros(n, np.int64)
    ep_idx = np.zeros(n, np.int64)
    seed_reset, _ = RO.rollout_seeds(SEED, epoch=1)
    for t in range(T):
        ep_len += 1
        assert np.array_equal(tmo[:, t], ep_len == mes), f"timeouts at step {t}"
        assert (ep_len <= mes).all()
        d = dones[:, t]
        if t + 1 < T:
            assert np.array_equal(obs[~d, t + 1], nxt[~d, t]), f"chain at step {t}"  # exactly, unless done
        ep_idx[d] += 1
        if t + 1 < T:
            for e in np.unique(ep_idx[d]):
                rows = np.nonzero(d & (ep_idx == e))[0]
                ref, tol = _reset_rows(env_id, dtype, env, seed_reset, int(e), rows, n)
                got = obs[rows, t + 1].astype(np.float64)
                assert np.all(np.abs(got - ref) <= tol), f"reset sample of episode {e} at step {t + 1}"
        ep_len[d] = 0
    assert dones.any() and tmo.any()
    if "Balancing" in env_id:
        assert (dones & ~tmo).any()  # terminations too
    # rollout_info, recomputed in float64 from the flat rows: the finished episodes are everything up to each env's last done
    fin = int(dones.sum())
    last = np.where(dones.any(axis=1), T - 1 - np.argmax(dones[:, ::-1], axis=1), -1)
    fin_len = int((last + 1).sum())
    fin_ret = float(sum(rew[i, : last[i] + 1].sum() for i in range(n)))
    assert info["total_episode_num"] == fin
    assert abs(info["avg_length"] - fin_len / fin) <= 1e-12 * fin_len / fin
    ret_tol = 1e-9 if dtype == torch.float64 else 1e-4  # float32 episode returns are accumulated in float32
    assert abs(info["avg_reward"] - fin_ret / fin) <= ret_tol * max(1.0, abs(fin_ret / fin))

    # ---- values, teacher-forced from the recorded observations (the I2P observation does not determine the state, the
    # charged ball's omits its regime: for those the chain is dataset = records here plus the records-vs-step tests)
    if env_id in CARTPOLE or env_id in IP:
        _check_values(env_id, dtype, env, samples, env.freq_rate)


@pytest.mark.parametrize("policy", ("random", "teacher"))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64), ids=("f32", "f64"))
@pytest.mark.parametrize("env_id", ROLLOUT_ENVS)
def test_collect_dataset(env_id, dtype, policy):
    _collect_and_check(env_id, dtype, policy, n=512, T=64)


@pytest.mark.parametrize("env_id,dtype", (("BoundaryInvertedDoublePendulumBalancing-v0", torch.float64),
                                          ("ContinuousCartPoleSwingUp-v0", torch.float64)))
def test_collect_dataset_past_the_grid_cap(env_id, dtype):
    """40001 envs x 48 steps: more transpose tiles than the grid's 148 x 8 CTAs, a ragged last tile in both dimensions"""
    _collect_and_check(env_id, dtype, "random", n=40001, T=48)
