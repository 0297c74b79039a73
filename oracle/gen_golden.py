"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz by EXECUTING the unmodified reference.

Run in the build container (where /root/reference exists):  ``python oracle/gen_golden.py``.
The vectors are committed; the GPU box has no reference tree, so the GPU parity tests and the
oracle self-tests compare against these files.

Every array is produced by the reference's own code (through oracle/ref_loader.py); inputs are
seeded with np.random.default_rng so the files are reproducible.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader as R  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def cartpole_states(rng, n, x_thr):
    """SURVEY.md 8(d) C2 distribution + a slice at the terminal thresholds."""
    s = rng.uniform(-1, 1, size=(n, 4)) * np.array([4.0, 5.0, np.pi, 8.0])
    k = n // 8
    s[:k, 0] = np.sign(s[:k, 0]) * rng.uniform(x_thr - 0.02, x_thr + 0.02, size=k)  # |x| near threshold
    s[k : 2 * k, 2] = rng.uniform(-0.25, 0.25, size=k)  # theta near the 12 deg threshold / upright
    s[2 * k : 3 * k, 2] *= 40.0  # large unwrapped angles (swing-up theta is never wrapped)
    s[3 * k, :] = [x_thr, 0.0, 0.0, 0.0]
    s[3 * k + 1, :] = [-x_thr, 0.0, 12 * 2 * np.pi / 360, 0.0]
    return s


def gen_cartpole():
    out = {}
    for kind in ("balancing", "swingup", "continuous_balancing", "continuous_swingup"):
        for fr in (1, 4):
            rng = np.random.default_rng(1000 + 10 * ["balancing", "swingup", "continuous_balancing", "continuous_swingup"].index(kind) + fr)
            env = R.make_cartpole(kind, freq_rate=fr, real_time_scale=0.02)
            n = 256
            states = cartpole_states(rng, n, float(env.x_threshold))
            if kind.startswith("continuous"):
                actions = rng.uniform(-1, 1, size=(n, 1)).astype(np.float32)
            else:
                actions = rng.integers(0, 2, size=n)
            nobs = np.zeros((n, 4))
            rew = np.zeros((n, 1))
            done = np.zeros((n, 1), dtype=bool)
            for i in range(n):
                env.state = states[i].copy()
                a = actions[i] if kind.startswith("continuous") else int(actions[i])
                o, r, t, tr, info = env.step(a)
                assert tr is False and info == {}
                nobs[i], rew[i, 0], done[i, 0] = o, r, t
            tag = f"{kind}_fr{fr}"
            out[f"{tag}_state"] = states
            out[f"{tag}_action"] = actions
            out[f"{tag}_next"] = nobs
            out[f"{tag}_reward"] = rew
            out[f"{tag}_done"] = done
    # free-running trajectory (not teacher forced): 8 envs x 200 steps, swingup fr=4, from reset(seed)
    traj = []
    acts = np.random.default_rng(77).integers(0, 2, size=(8, 200))
    inits = []
    for e in range(8):
        env = R.make_cartpole("swingup", freq_rate=4)
        o, _ = env.reset(seed=100 + e)
        inits.append(o)
        row = []
        for t in range(200):
            o, r, d, _, _ = env.step(int(acts[e, t]))
            row.append(np.concatenate([o, [r, float(d)]]))
        traj.append(row)
    out["traj_swingup_fr4_init"] = np.array(inits)
    out["traj_swingup_fr4_action"] = acts
    out["traj_swingup_fr4"] = np.array(traj)  # [8,200,6] = obs(4), reward, done
    # init-state distribution samples (only moments are compared)
    env = R.make_cartpole("swingup")
    env.reset(seed=5)
    out["init_swingup_seed5"] = env.get_batch_init_state(4096)
    env = R.make_cartpole("balancing")
    env.reset(seed=5)
    out["init_balancing_seed5"] = env.get_batch_init_state(4096)
    np.savez_compressed(os.path.join(OUT, "cartpole.npz"), **out)


def poison(rng, a, frac=0.02):
    n = a.shape[0]
    idx = rng.choice(n, size=max(3, int(frac * n)), replace=False)
    vals = [np.nan, np.inf, -np.inf]
    for j, i in enumerate(idx):
        a[i, rng.integers(0, a.shape[1])] = vals[j % 3]
    return a


def gen_scoring():
    out = {}
    n = 512
    # ---------------- Hopper (hopper.py:79-106)
    for T in (True, False):
        rng = np.random.default_rng(1003 + int(T))
        env = R.make_mujoco_shell("hopper", terminate_when_unhealthy=T)
        obs = np.array([0, 1.25] + [0] * 10, dtype=np.float64) + rng.standard_normal((n, 12)) * np.array(
            [1, 0.4, 0.15] + [1] * 9
        )
        obs[: n // 8, 2:] *= 60.0  # push some rows outside the +-100 healthy_state_range
        obs[n // 8, 3] = 100.0  # exactly on the (exclusive) bound
        obs[n // 8 + 1, 1] = 0.7  # exactly on the z bound
        obs = poison(rng, obs)
        pre = obs.copy()
        pre[:, 0] -= rng.standard_normal(n) * 0.01
        act = rng.uniform(-1, 1, size=(n, 3))
        tag = f"hopper_T{int(T)}"
        out[f"{tag}_obs"], out[f"{tag}_pre_obs"], out[f"{tag}_action"] = obs, pre, act
        out[f"{tag}_reward"] = env.get_batch_reward(obs, pre, act)
        out[f"{tag}_done"] = env.get_batch_terminal(obs, pre, act)
        out[f"{tag}_healthy"] = env.is_healthy(obs)
        out[f"{tag}_dt"] = np.array(env.dt)
    # reference's own known-answer test (test/test_envs/test_mujoco/test_hopper.py:6-25)
    env = R.make_mujoco_shell("hopper")
    out["hopper_kat_ones_healthy"] = env.is_healthy(np.ones([128, 12]))
    out["hopper_kat_101_healthy"] = env.is_healthy(np.ones([128, 12]) * 101)
    out["hopper_kat_reward"] = env.get_batch_reward(obs=np.ones([128, 12]), pre_obs=np.ones([128, 12]), action=np.ones([128, 3]))
    out["hopper_kat_done"] = env.get_batch_terminal(obs=np.ones([128, 12]))
    # zoo config dt (zoo/conf/task/hopper.yaml:3-5: freq_rate 10? use ctor kwargs) -- custom weights
    env = R.make_mujoco_shell(
        "hopper", freq_rate=2, real_time_scale=0.01, forward_reward_weight=1.5, ctrl_cost_weight=2e-3,
        healthy_reward=0.5, terminate_when_unhealthy=False, healthy_state_range=(-50.0, 60.0), healthy_z_range=(0.8, 2.0),
    )
    rng = np.random.default_rng(2003)
    obs = np.array([0, 1.25] + [0] * 10, dtype=np.float64) + rng.standard_normal((n, 12)) * np.array([1, 0.6, 0.15] + [30] * 9)
    pre = obs + rng.standard_normal((n, 12)) * 0.01
    act = rng.uniform(-1, 1, size=(n, 3))
    out["hopper_custom_obs"], out["hopper_custom_pre_obs"], out["hopper_custom_action"] = obs, pre, act
    out["hopper_custom_reward"] = env.get_batch_reward(obs, pre, act)
    out["hopper_custom_done"] = env.get_batch_terminal(obs, pre, act)
    out["hopper_custom_dt"] = np.array(env.dt)
    # ---------------- HalfCheetah (half_cheetah.py:59-67)
    rng = np.random.default_rng(1005)
    env = R.make_mujoco_shell("half_cheetah")
    obs = poison(rng, rng.standard_normal((n, 18)))
    pre = obs + rng.standard_normal((n, 18)) * 0.01
    act = rng.uniform(-1, 1, size=(n, 6))
    out["halfcheetah_obs"], out["halfcheetah_pre_obs"], out["halfcheetah_action"] = obs, pre, act
    out["halfcheetah_reward"] = env.get_batch_reward(obs, pre, act)
    out["halfcheetah_done"] = env.get_batch_terminal(obs, pre, act)
    out["halfcheetah_dt"] = np.array(env.dt)
    # ---------------- IP x4 (inverted_pendulum.py:73-183)
    for kind in ("ip_rebound_balancing", "ip_boundary_balancing", "ip_rebound_swingup", "ip_boundary_swingup"):
        rng = np.random.default_rng(1010 + len(kind))
        env = R.make_mujoco_shell(kind)
        obs = rng.uniform(-1, 1, size=(n, 4)) * np.array([2.2, np.pi, 5, 8])
        obs[0, 0], obs[1, 0], obs[2, 1], obs[3, 1] = 2.0, -2.0, np.pi / 2, np.arccos(0.9)
        obs = poison(rng, obs)
        out[f"{kind}_obs"] = obs
        out[f"{kind}_reward"] = env.get_batch_reward(obs)
        out[f"{kind}_done"] = env.get_batch_terminal(obs)
    env = R.make_mujoco_shell("ip_boundary_swingup")
    for k in (1, 2, 3, 5):
        out[f"ip_graph_k{k}"] = env.get_transition_graph(k)
    out["ip_env_params_name"] = np.array(env.env_params_name)
    # angle wrap rule (inverted_pendulum.py:45-49) evaluated by the reference expression itself
    th = np.random.default_rng(9).uniform(-40, 40, size=2048)
    th[:4] = [np.pi, -np.pi, 3 * np.pi, 0.0]

    class _SV:
        def __init__(s, v):
            s.v = v

        def state_vector(s):
            return s.v

    from emei.envs.mujoco.inverted_pendulum import BaseInvertedPendulumEnv

    wrapped = np.array([BaseInvertedPendulumEnv.current_obs.fget(_SV(np.array([0.0, t, 0.0, 0.0])))[1] for t in th])
    out["ip_wrap_in"], out["ip_wrap_out"] = th, wrapped
    # ---------------- I2P x4 (inverted_double_pendulum.py:84-196)
    for kind in ("i2p_rebound_balancing", "i2p_boundary_balancing", "i2p_rebound_swingup", "i2p_boundary_swingup"):
        rng = np.random.default_rng(1020 + len(kind))
        env = R.make_mujoco_shell(kind)
        obs = rng.uniform(-1, 1, size=(n, 6)) * np.array([3.3, np.pi, np.pi, 5, 8, 8])
        obs[0, 0], obs[1, 0] = 3.0, -3.0
        obs[: n // 4, 1:3] *= 0.2
        obs = poison(rng, obs)
        out[f"{kind}_obs"] = obs
        out[f"{kind}_reward"] = env.get_batch_reward(obs)
        out[f"{kind}_done"] = env.get_batch_terminal(obs)
    np.savez_compressed(os.path.join(OUT, "scoring.npz"), **out)


def gen_charged_ball():
    """Drive the reference helpers (charged_ball.py:54-82) on hand-built objects (the class is
    not constructible, SURVEY.md 0.7).  24 envs x 256 steps per config, full state trajectories, of which the first
    KEEP_STEPS steps of every third env are stored (a small file; envs 3 and 15 among them start fast)."""
    KEEP_STEPS, KEEP_ENVS = 160, slice(0, 24, 3)
    out = {}
    for continuous in (False, True):
        for fr in (1, 3):
            rng = np.random.default_rng(1004 + fr + 10 * int(continuous))
            n, T = 24, 256
            if continuous:
                actions = rng.uniform(-1, 1, size=(T, n, 1)).astype(np.float32)
            else:
                # sticky random actions so the ball gains enough energy to leave the ring
                flips = rng.random((T, n)) < 0.08
                actions = (np.cumsum(flips, axis=0) + rng.integers(0, 2, size=n)[None]) % 2
            on = np.zeros((T + 1, n), dtype=bool)
            circle = np.zeros((T + 1, n, 2))
            free = np.zeros((T + 1, n, 4))
            for e in range(n):
                env = R.make_charged_ball(continuous=continuous, freq_rate=fr)
                env.np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(500 + e)))
                env.state = env._get_initial_state()
                if e % 4 == 3:  # start some envs fast so they fly off near the top
                    env.state["circle_state"][1] = rng.uniform(3.0, 6.5) * rng.choice([-1, 1])
                    env.state["free_state"] = env.circle_to_free(env.state["circle_state"])
                on[0, e], circle[0, e], free[0, e] = env.state["on_circle"], env.state["circle_state"], env.state["free_state"]
                for t in range(T):
                    a = actions[t, e] if continuous else int(actions[t, e])
                    o32 = R.charged_ball_step(env, a)
                    assert o32.dtype == np.float32 and np.array_equal(o32, np.asarray(env.state['free_state'], dtype=np.float32))
                    on[t + 1, e] = env.state["on_circle"]
                    circle[t + 1, e] = env.state["circle_state"]
                    free[t + 1, e] = env.state["free_state"]
            tag = f"{'cont' if continuous else 'disc'}_fr{fr}"
            out[f"{tag}_action"] = actions[:KEEP_STEPS, KEEP_ENVS]
            on, circle, free = on[: KEEP_STEPS + 1, KEEP_ENVS], circle[: KEEP_STEPS + 1, KEEP_ENVS], free[: KEEP_STEPS + 1, KEEP_ENVS]
            out[f"{tag}_on"] = on
            out[f"{tag}_circle"] = circle
            out[f"{tag}_free"] = free
            print(tag, "fraction of (env,step) in free flight:", 1 - on.mean(), "landings:", int((on[1:] & ~on[:-1]).sum()))
    # scalar reward rule (charged_ball.py:158-160) on the float64 free state
    env = R.make_charged_ball()
    fs = out["disc_fr1_free"][1:40].reshape(-1, 4)
    out["reward_free"] = fs
    out["reward"] = np.array([env.get_batch_reward(f) for f in fs])
    np.savez_compressed(os.path.join(OUT, "charged_ball.npz"), **out)


def gen_core():
    """core.py:56-58 env_params_name; test/test_core.py:9-14 known answers."""
    emei = R.load_reference()
    out = {}
    e = emei.EmeiEnv(env_params={"a": 3, "b": 5, "d": 0.33, "c": "c"})
    out["name_abcd"] = np.array(e.env_params_name)
    e = R.make_cartpole("swingup", freq_rate=4, real_time_scale=0.01)
    out["name_cartpole"] = np.array(e.env_params_name)
    np.savez_compressed(os.path.join(OUT, "core.npz"), **out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    gen_core()
    gen_cartpole()
    gen_scoring()
    gen_charged_ball()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
