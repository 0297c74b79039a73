"""CPU-side checks: the C-ABI library loads and exports every symbol include/emei_b200.h declares,
argument validation returns the documented codes (no compute without a GPU), and the host-side
mirror of the reference API behaves like emei/core.py + test/test_core.py."""
import ctypes
import os
import re

import numpy as np
import pytest

import emei_b200 as E
from emei_b200 import _lib
from emei_b200.core import EmeiEnv
from emei_b200.dist import shard_range

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "emei_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(emei_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    syms = header_symbols()
    assert len(syms) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/emei_b200.h but not exported"
    assert sorted(_lib.exported_symbols()) == syms  # the ctypes binding covers the whole header
    assert _lib.lib.emei_version() == 100


def test_struct_layouts_match_header():
    # sizes the C side compiles to (doubles then int32s, natural alignment)
    assert ctypes.sizeof(_lib.CartPoleParams) == 13 * 8 + 4 * 4
    assert ctypes.sizeof(_lib.ChargedBallParams) == 5 * 8 + 2 * 4
    assert ctypes.sizeof(_lib.ScoringParams) == 2 * 4 + 13 * 8
    assert ctypes.sizeof(_lib.I2PParams) == 12 * 8 + 3 * 4 + 4  # padded to a multiple of 8
    assert ctypes.sizeof(_lib.NoiseParams) == 6 * 8 + 3 * 8


def test_noisy_step_validation_codes():
    """emei_ip_step_noisy_* / emei_i2p_step_noisy_*: IP variants only, a noise struct is required, sigmas >= 0."""
    lib = _lib.lib
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 1, 0.02, _lib.IP_BOUNDARY_SWINGUP, 3
    z = _lib.NoiseParams()
    for f in (lib.emei_ip_step_noisy_f32, lib.emei_ip_step_noisy_f64):
        assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), None, None) == -1
        assert f(None, None, None, None, None, None, None, 0, ctypes.byref(p), ctypes.byref(z), None) == 0
        assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), ctypes.byref(z), None) == -1  # null state
        p.variant = _lib.CARTPOLE_SWINGUP  # the classic-control family has no obs_noise_params (base_control.py:14-16)
        assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), ctypes.byref(z), None) == -2
        p.variant = _lib.IP_BOUNDARY_SWINGUP
        z.sigma[2] = -1.0
        assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), ctypes.byref(z), None) == -6
        z.sigma[2] = 0.0
    q = _lib.I2PParams()
    q.freq_rate, q.dt, q.variant, q.action_kind = 1, 0.02, _lib.I2P_BOUNDARY_SWINGUP, 3
    q.mass_cart = q.mass_pole0 = q.mass_pole1 = q.length0 = q.length1 = 1.0
    for f in (lib.emei_i2p_step_noisy_f32, lib.emei_i2p_step_noisy_f64):
        assert f(None, None, None, None, None, None, None, 8, ctypes.byref(q), None, None) == -1
        z.sigma[5] = float("nan")
        assert f(None, None, None, None, None, None, None, 8, ctypes.byref(q), ctypes.byref(z), None) == -6
        z.sigma[5] = 0.0
        assert f(None, None, None, None, None, None, None, 0, ctypes.byref(q), ctypes.byref(z), None) == 0


def test_argument_validation_codes():
    lib = _lib.lib
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 1, 0.02, _lib.CARTPOLE_SWINGUP, 0
    f = lib.emei_cartpole_step_f32
    assert f(None, None, None, None, None, None, None, -1, ctypes.byref(p), None) == -4
    assert f(None, None, None, None, None, None, None, 0, ctypes.byref(p), None) == 0  # empty batch: no-op
    assert f(None, None, None, None, None, None, None, 8, None, None) == -1
    assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), None) == -1  # null state
    p.variant = 99
    assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), None) == -2
    p.variant, p.action_kind = _lib.CARTPOLE_SWINGUP, 7
    assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), None) == -3
    p.action_kind, p.freq_rate = 0, 0
    assert f(None, None, None, None, None, None, None, 8, ctypes.byref(p), None) == -6
    p.freq_rate = 1
    buf = (ctypes.c_float * 64)()
    addr = ctypes.addressof(buf)
    mis = addr + 4 if addr % 16 == 0 else addr  # a deliberately misaligned (host) address: rejected before any launch
    if mis % 16 != 0:
        assert f(mis, mis, None, addr, addr, addr, None, 8, ctypes.byref(p), None) == -5
    s = _lib.ScoringParams()
    s.family = 42
    assert lib.emei_reward_terminal_f64(None, None, None, None, None, None, 4, ctypes.byref(s), None) == -2
    s.family, s.dt = _lib.HOPPER, 0.0
    assert lib.emei_reward_terminal_f64(None, None, None, None, None, None, 4, ctypes.byref(s), None) == -6
    assert lib.emei_snapshot_copy(None, None, -3, None) == -4
    assert lib.emei_snapshot_copy(None, None, 0, None) == 0
    assert b"16-byte" in lib.emei_error_string(-5)
    assert [lib.emei_family_obs_dim(k) for k in (_lib.HOPPER, _lib.HALFCHEETAH, _lib.I2P_BOUNDARY_SWINGUP, _lib.CHARGED_BALL, 77)] == [12, 18, 6, 4, -1]
    assert [lib.emei_family_action_dim(k) for k in (_lib.HOPPER, _lib.HALFCHEETAH, _lib.CARTPOLE_SWINGUP)] == [3, 6, 1]


# Malformed inputs x every rollout entry point: the code each one returns.  The packed entries (float32) check the batch,
# parameters and horizon, return early for empty work, then check state, episode buffers, actions and records (with the
# 16-byte alignment of the observation records); the reference-arithmetic entries check the episode buffers, horizon,
# actions and records (no alignment) before the early return and the state.  Every row is rejected before any launch:
# the reference entries always get a null state, the packed ones an aligned host state only where a later check fails.
# Columns: packed cart-pole, packed charged ball, reference cart-pole, I2P, reference charged ball (both precisions).
_ROLLOUT_ROWS = [
    # name,                     n,  horizon, init_kind, episode buffers, records,      packed state, codes
    ("empty batch",             0,  8,       0,         False,           None,         False, (0, 0, -1, -1, -1)),
    ("negative horizon",        16, -1,      0,         False,           None,         False, (-6, -6, -1, -1, -1)),
    ("negative horizon, bufs",  16, -1,      0,         True,            None,         False, (-6, -6, -6, -6, -6)),
    ("partial records",         16, 8,       0,         True,            "partial",    True, (-1, -1, -1, -1, -1)),
    ("misaligned obs records",  16, 8,       0,         True,            "misaligned", True, (-5, -5, -1, -1, -1)),
    ("bad init_kind",           16, 8,       5,         True,            None,         False, (-6, -1, -1, -1, -1)),
]


def _check_rollout_validation_table():
    lib = _lib.lib
    buf = (ctypes.c_char * 4096)()
    base = (ctypes.addressof(buf) + 15) & ~15
    aligned = [base + 256 * j for j in range(14)]  # distinct 16-byte-aligned host addresses (never dereferenced)
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 1, 0.02, _lib.CARTPOLE_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    q = _lib.I2PParams()
    q.gravity, q.mass_cart, q.mass_pole0, q.mass_pole1, q.length0, q.length1, q.dt = 9.81, 10.0, 4.0, 4.0, 0.3, 0.3, 0.02
    q.freq_rate, q.variant, q.action_kind = 1, _lib.I2P_BOUNDARY_SWINGUP, _lib.ACTION_CONTINUOUS_F32
    c = _lib.ChargedBallParams()
    c.gravity_acc, c.mass_ball, c.radius, c.charge, c.time_step, c.freq_rate, c.action_kind = 9.8, 1.0, 1.0, 10.0, 0.02, 1, 0
    table = (ctypes.c_double * 6)()
    for name, n, horizon, init_kind, bufs, records, packed_state, codes in _ROLLOUT_ROWS:
        r = _lib.RolloutParams()
        r.horizon, r.random_policy, r.init_kind = horizon, 1, init_kind
        episode = aligned[3:6] if bufs else [None] * 3
        rec = [None] * 6
        if records == "partial":
            rec[0] = aligned[6]
        elif records == "misaligned":
            rec = [aligned[6] + 4] + aligned[7:12]
        tail = [None] + rec + [None]  # actions (random policy), records, stats
        entries = [
            (0, lib.emei_cartpole_rollout_f32, 1, (ctypes.byref(p), ctypes.byref(r))),
            (1, lib.emei_charged_ball_rollout_f32, 3, (ctypes.byref(c), ctypes.byref(r))),
        ]
        for sfx in ("_f32", "_f64"):
            entries += [
                (2, getattr(lib, "emei_cartpole_rollout_ref" + sfx), 1, (ctypes.byref(p), ctypes.byref(r), None)),
                (3, getattr(lib, "emei_i2p_rollout" + sfx), 1, (ctypes.byref(q), ctypes.byref(r), table, table, None)),
                (4, getattr(lib, "emei_charged_ball_rollout_ref" + sfx), 3, (ctypes.byref(c), ctypes.byref(r))),
            ]
        for col, f, n_state, params in entries:
            state = aligned[:n_state] if (packed_state and col < 2) else [None] * n_state
            got = f(*state, *episode, *tail, n, *params, None)
            assert got == codes[col], f"{name}: {f.__name__} returned {got}, expected {codes[col]}"


def test_rollout_and_transpose_validation_codes():
    lib = _lib.lib
    assert ctypes.sizeof(_lib.RolloutParams) == 6 * 4 + 4 * 8 + 2 * 8 + 8 * 8 + 2 * 8
    p = _lib.CartPoleParams()
    p.freq_rate, p.dt, p.variant, p.action_kind = 4, 0.02, _lib.CARTPOLE_SWINGUP, 3
    r = _lib.RolloutParams()
    r.horizon, r.random_policy = 8, 1
    f = lib.emei_cartpole_rollout_f32
    nul = [None] * 12
    assert f(*nul, -1, ctypes.byref(p), ctypes.byref(r), None) == -4
    assert f(*nul, 0, ctypes.byref(p), ctypes.byref(r), None) == 0       # empty batch: no-op
    assert f(*nul, 16, ctypes.byref(p), None, None) == -1
    assert f(*nul, 16, ctypes.byref(p), ctypes.byref(r), None) == -1     # null state
    r.init_kind = 5
    assert f(*nul, 16, ctypes.byref(p), ctypes.byref(r), None) == -6
    r.init_kind, r.horizon = 0, 0
    assert f(*nul, 16, ctypes.byref(p), ctypes.byref(r), None) == 0      # zero steps: no-op
    c = _lib.ChargedBallParams()
    c.gravity_acc, c.mass_ball, c.radius, c.charge, c.time_step, c.freq_rate, c.action_kind = 9.8, 1.0, 1.0, 10.0, 0.02, 1, 0
    g = lib.emei_charged_ball_rollout_f32
    r.horizon = 4
    assert g(*([None] * 14), 16, ctypes.byref(c), ctypes.byref(r), None) == -1
    c.radius = 0.0
    assert g(*([None] * 14), 16, ctypes.byref(c), ctypes.byref(r), None) == -6
    q = _lib.I2PParams()
    q.gravity, q.mass_cart, q.mass_pole0, q.mass_pole1, q.length0, q.length1, q.dt = 9.81, 10.0, 4.0, 4.0, 0.3, 0.3, 0.02
    q.freq_rate, q.variant, q.action_kind = 1, _lib.I2P_BOUNDARY_SWINGUP, 3
    h = lib.emei_i2p_step_f64
    assert h(None, None, None, None, None, None, None, 0, ctypes.byref(q), None) == 0
    assert h(None, None, None, None, None, None, None, 4, ctypes.byref(q), None) == -1
    q.variant = _lib.HOPPER
    assert h(None, None, None, None, None, None, None, 4, ctypes.byref(q), None) == -2
    q.variant, q.length1 = _lib.I2P_REBOUND_BALANCING, 0.0
    assert h(None, None, None, None, None, None, None, 4, ctypes.byref(q), None) == -6
    _check_rollout_validation_table()
    t = lib.emei_records_transpose
    assert t(None, None, 4, -1, 4, None) == -4
    assert t(None, None, 4, 8, 3, None) == -6          # element sizes: 1, 4, 8, 16, 24, 32, 48
    for bad in (3, 12, 20, 64):
        assert t(None, None, 4, 8, bad, None) == -6, bad
    assert t(None, None, 0, 8, 4, None) == 0
    assert t(None, None, 4, 8, 4, None) == -1
    # the wide observation rows (6 x float32, 4 x float64, 6 x float64): null pointers, then the alignment of the words
    # they move in (8 bytes for 24, 16 for 32 and 48).  A misaligned address is refused before anything is launched, so
    # these calls need no device; every call here has a null or a misaligned pointer and never launches.
    base = 1 << 20
    for eb in (24, 32, 48):
        assert t(None, None, 0, 8, eb, None) == 0
        assert t(None, None, 3, 5, eb, None) == -1, eb
        assert t(base, None, 3, 5, eb, None) == -1, eb
        assert t(None, base, 3, 5, eb, None) == -1, eb
    for eb, off in ((24, 4), (24, 12), (32, 8), (32, 4), (48, 8), (48, 4)):
        assert t(base + off, base, 3, 5, eb, None) == -5, (eb, off)
        assert t(base, base + off, 3, 5, eb, None) == -5, (eb, off)
    assert t(base + 8, base + 4, 3, 5, 24, None) == -5  # 8 bytes suffice for in, not 4 for out


def test_offline_dataset_files_roundtrip(tmp_path, monkeypatch):
    """zoo/util.py:108-111 + core.py:61-81,109-128: flat files with the six keys, the reference's key checks, and
    the cache layout DATASET_PATH/<env_name>/<env_params_name>/<file> behind dataset_names / get_dataset."""
    from emei_b200 import offline

    rng = np.random.default_rng(0)
    n = 37
    ds = dict(observations=rng.normal(size=(n, 4)).astype(np.float32), next_observations=rng.normal(size=(n, 4)).astype(np.float32),
              actions=rng.integers(0, 2, n), rewards=rng.normal(size=n).astype(np.float32),
              dones=(rng.random(n) < 0.1).astype(np.float32), timeouts=np.zeros(n, np.float32))
    monkeypatch.setattr(offline, "DATASET_PATH", tmp_path)
    env = E.make("CartPoleSwingUp-v0", freq_rate=2)
    assert env.dataset_names == []
    path = offline.save_dataset(ds, offline.dataset_path(env, "random.npz"))
    assert path == tmp_path / "CartPoleSwingUp" / "freq_rate=2&integrator=euler&real_time_scale=0.02" / "random.npz"
    assert env.dataset_names == ["random.npz"]
    back = env.get_dataset("random.npz")
    assert sorted(back) == sorted(ds) and all(np.array_equal(back[k], ds[k]) for k in ds)
    with pytest.raises(FileNotFoundError):
        env.get_dataset("expert.h5")
    bad = dict(ds)
    del bad["timeouts"]
    with pytest.raises(AssertionError, match="missing key timeouts"):
        offline.check_dataset(bad)
    bad = dict(ds, rewards=ds["rewards"][:-1])
    with pytest.raises(AssertionError):
        offline.check_dataset(bad)
    try:
        import h5py  # noqa: F401
    except ImportError:
        with pytest.raises(ImportError):
            offline.save_dataset(ds, tmp_path / "x.h5")
    # float64 rows (the reference-exact mode) and 6-wide rows (the inverted double pendulum, Box actions [N, 1]) keep
    # their dtypes, shapes and bits through the file
    for env_id, dim, dt in (("CartPoleSwingUp-v0", 4, np.float64), ("BoundaryInvertedDoublePendulumSwingUp-v0", 6, np.float32),
                            ("ReboundInvertedDoublePendulumBalancing-v0", 6, np.float64)):
        wide = dict(observations=rng.normal(size=(n, dim)).astype(dt), next_observations=rng.normal(size=(n, dim)).astype(dt),
                    actions=(rng.integers(0, 2, n) if dim == 4 else rng.uniform(-1, 1, (n, 1)).astype(np.float32)),
                    rewards=rng.normal(size=n).astype(dt), dones=(rng.random(n) < 0.1).astype(np.float32),
                    timeouts=(rng.random(n) < 0.05).astype(np.float32))
        env = E.make(env_id)
        path = offline.save_dataset(wide, offline.dataset_path(env, "wide"))
        assert path.suffix == ".npz" and env.dataset_names == ["wide.npz"]
        back = env.get_dataset("wide.npz")
        assert sorted(back) == sorted(wide)
        for k in wide:
            assert back[k].dtype == wide[k].dtype and back[k].shape == wide[k].shape and np.array_equal(back[k], wide[k]), (env_id, k)


def test_env_params_name(golden):
    """test/test_core.py:9-14."""
    env = EmeiEnv(env_params={"a": 3, "b": 5, "d": 0.33, "c": "c"})
    assert env.env_params_name == "a=3&b=5&c=c&d=0.33" == str(golden("core")["name_abcd"])
    env = EmeiEnv(env_params=dict(freq_rate=1, real_time_scale=0.02))
    assert env.env_params_name == "freq_rate=1&real_time_scale=0.02"
    env = E.make("CartPoleSwingUp-v0", freq_rate=4, real_time_scale=0.01)
    assert env.env_params_name == str(golden("core")["name_cartpole"])
    assert E.make("BoundaryInvertedPendulumSwingUp-v0").env_params_name == str(golden("scoring")["ip_env_params_name"])


def test_freeze_flag():
    """test/test_core.py:17-23 on the bare base class, incl. the asserts of core.py:28,36."""
    env = EmeiEnv(env_params=dict(freq_rate=1, time_step=0.02))
    env.freeze()
    assert env.frozen
    with pytest.raises(AssertionError):
        env.freeze()
    env.unfreeze()
    assert not env.frozen
    with pytest.raises(AssertionError):
        env.unfreeze()


def test_abstract_methods_raise():
    """core.py:175-193; test/test_envs/test_classic_control/test_cartpole.py:4-11."""
    from emei_b200.envs.classic_control.cartpole import BaseCartPoleEnv

    env = EmeiEnv(env_params={})
    for fn in (lambda: env.get_batch_init_state(2), lambda: env.get_batch_reward(None), lambda: env.get_batch_terminal(None)):
        with pytest.raises(NotImplementedError):
            fn()
    with pytest.raises(AssertionError):
        env.get_batch_next_obs(None)  # not frozen
    with pytest.raises(NotImplementedError):
        BaseCartPoleEnv().reset()
    with pytest.raises(NotImplementedError):
        E.make("HopperRunning-v0").rollout(3)  # scoring-only env: no fused rollout kernel


def test_registry_ids_and_spaces():
    ids = set(E.registry)
    for must in (
        "CartPoleBalancing-v0", "CartPoleSwingUp-v0", "ContinuousCartPoleBalancing-v0", "ContinuousCartPoleSwingUp-v0",
        "ChargedBallCentering-v0", "ContinuousChargedBallCentering-v0", "BoundaryInvertedPendulumSwingUp-v0",
        "ReboundInvertedPendulumBalancing-v0", "BoundaryInvertedDoublePendulumSwingUp-v0", "HopperRunning-v0",
        "HalfCheetahRunning-v0",
    ):
        assert must in ids
    assert E.spec("CartPoleBalancing-v0")["max_episode_steps"] == 500
    env = E.make("CartPoleSwingUp-v0", num_envs=3)
    assert env.max_episode_steps == 1000 and env.action_space.n == 2 and env.observation_space.shape == (4,)
    assert env.x_threshold == 5 and env.action_space.contains(1) and not env.action_space.contains(2)
    env = E.make("ContinuousCartPoleSwingUp-v0")
    assert env.action_space.shape == (1,) and env.action_space.contains(np.array([0.5], dtype=np.float32))
    assert not env.action_space.contains(np.array([1.5], dtype=np.float32))
    env = E.make("HopperRunning-v0")
    assert env.observation_space.shape == (12,) and env.action_space.shape == (3,) and env.dt == 0.002 * 4
    env = E.make("HalfCheetahRunning-v0", freq_rate=10, real_time_scale=0.002)
    assert env.observation_space.shape == (18,) and env.action_space.shape == (6,) and abs(env.dt - 0.02) < 1e-15
    env = E.make("ChargedBallCentering-v0", freq_rate=2)
    assert env.env_params_name == "freq_rate=2&time_step=0.02" and env.time_step == 0.02
    with pytest.raises(KeyError):
        E.make("Walker2dRunning-v0")  # registered by the reference but its class does not exist there either
    with pytest.raises(NotImplementedError):
        E.make("HopperRunning-v0").step(np.zeros(3))  # MuJoCo dynamics are out of scope


def test_transition_graphs(golden):
    g = golden("scoring")
    env = E.make("BoundaryInvertedPendulumSwingUp-v0")
    for k in (1, 2, 3, 5):
        assert np.array_equal(env.get_transition_graph(k), g[f"ip_graph_k{k}"])
    assert env.get_reward_mech_graph() is None and env.get_termination_mech_graph() is None
    with pytest.raises(AttributeError):
        E.make("CartPoleSwingUp-v0").get_transition_graph()  # the reference has none (None.copy())
    i2p = E.make("BoundaryInvertedDoublePendulumSwingUp-v0")
    assert i2p.get_transition_graph().shape == (7, 6)


def test_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    env = E.make("CartPoleSwingUp-v0", num_envs=4)
    with pytest.raises(_lib.EmeiB200Error):
        env.reset()
    with pytest.raises(_lib.EmeiB200Error):
        E.make("HopperRunning-v0").get_batch_terminal(np.ones((4, 12)))


def test_shard_range_partitions_exactly():
    for total in (0, 1, 7, 1 << 20, (1 << 26) + 5):
        for w in (1, 2, 3, 4, 8):
            parts = [shard_range(total, r, w) for r in range(w)]
            assert parts[0][0] == 0 and parts[-1][1] == total
            assert all(parts[i][1] == parts[i + 1][0] for i in range(w - 1))
            sizes = [e - b for b, e in parts]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 3, 2)


def test_rollout_reset_sampler_mirror_is_uniform():
    """The lean in-rollout reset sampler (oracle mirror of rollout_f32.cuh: one Philox block, 24-bit uniforms) draws
    U(-0.05, 0.05) per coordinate (cartpole.py:131-132), + pi on the swing-up angle (cartpole.py:153-156); streams of
    different envs / episodes are distinct."""
    from scipy import stats

    from oracle import rollout_oracle as RO

    m = 4000
    ids = np.arange(m)
    s = RO.reset_sample_uniform(ids, np.ones(m, np.int64), 1234, pi_column=2)
    assert s.dtype == np.float32 and s.shape == (m, 4)
    s64 = s.astype(np.float64)
    s64[:, 2] -= np.pi
    assert np.all(s64 >= -0.05 - 1e-7) and np.all(s64 < 0.05 + 1e-7)
    for c in range(4):
        assert stats.kstest((s64[:, c] + 0.05) / 0.1, "uniform").pvalue > 1e-3
    assert abs(np.corrcoef(s64[:, 0], s64[:, 1])[0, 1]) < 0.06
    s2 = RO.reset_sample_uniform(ids, np.full(m, 2, np.int64), 1234, pi_column=2)
    assert not np.array_equal(s, s2) and len(np.unique(s[:, 0])) > m * 0.99


def test_obs_noise_mirror_is_gaussian_and_step_keyed():
    """oracle/philox.py obs_noise (mirror of kernels.cuh add_state_noise): N(0, sigma) per coordinate, a fresh draw
    per (env, env step, sub-step), independent of how the batch is sharded."""
    from scipy import stats

    from oracle import philox as P

    n, sig = 20000, np.array([0.01, 0.02, 0.0, 0.5])
    z = P.obs_noise(n, 4, sig, 99, 3, 2)
    assert z.shape == (2, n, 4) and np.all(z[:, :, 2] == 0.0)
    for c in (0, 1, 3):
        assert abs(z[0, :, c].std() / sig[c] - 1) < 0.03
        assert stats.kstest(z[1, :, c] / sig[c], "norm").pvalue > 1e-3
    assert abs(np.corrcoef(z[0, :, 0], z[0, :, 1])[0, 1]) < 0.03 and abs(np.corrcoef(z[0, :, 0], z[1, :, 0])[0, 1]) < 0.03
    assert not np.array_equal(z, P.obs_noise(n, 4, sig, 99, 4, 2))
    assert np.array_equal(z[:, 5000:], P.obs_noise(n - 5000, 4, sig, 99, 3, 2, env_offset=5000))


def test_step_host_ranges_are_aligned_partitions():
    """HostStaging cuts the batch into ranges whose interior edges sit on 16-env boundaries (every per-range pointer,
    uint8 flags included, stays 16-byte aligned for the C ABI) and that tile [0, n) exactly."""
    from emei_b200.engine import HostStaging

    class _Space:
        shape = (1,)

    class _Env:
        def __init__(self, n):
            self.num_envs, self.action_space = n, _Space()

    for n in (1, 4096, 300_000, 1_100_003, (1 << 23), (1 << 23) + 7, (1 << 26) + 1):
        for chunks, fractions in ((None, None), (3, None), (None, [0.1, 0.3, 0.6])):
            r = HostStaging.plan_ranges(n, chunks, fractions)
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(r, r[1:])) and all(hi > lo for lo, hi in r)
            assert all(lo % 16 == 0 for lo, _ in r)


def test_numa_binding_helpers_are_safe_without_topology():
    """emei_b200.dist.bind_to_gpu_numa: parses sysfs CPU lists, and changes nothing where there is no GPU / no
    per-GPU locality (this container)."""
    import os

    from emei_b200 import dist as D

    assert sorted(D._parse_cpulist("0-3,8,10-11")) == [0, 1, 2, 3, 8, 10, 11]
    assert D._parse_cpulist("") == set()
    before = os.sched_getaffinity(0)
    assert D.bind_to_gpu_numa(0) is None or isinstance(D.bind_to_gpu_numa(0), list)
    if not __import__("torch").cuda.is_available():
        assert D.gpu_numa_info(0) == {"pci": None, "numa_node": None, "local_cpulist": None}
        assert os.sched_getaffinity(0) == before


def test_round2_entry_points_validate_arguments_without_a_gpu():
    """The entry points added in round 2 reject bad arguments with EMEI_ERR_* codes before any CUDA call, and treat
    empty work as a valid no-op (include/emei_b200.h conventions)."""
    import ctypes

    from emei_b200 import _lib

    L = _lib.lib
    sp = _lib.ScoringParams()
    sp.family, sp.dt = _lib.HOPPER, 0.008
    for sfx in ("_f32", "_f64"):
        seq = getattr(L, "emei_reward_terminal_seq" + sfx)
        assert seq(None, None, None, None, None, 0, 5, ctypes.byref(sp), None) == 0          # no envs
        assert seq(None, None, None, None, None, 7, 0, ctypes.byref(sp), None) == 0          # no steps
        assert seq(None, None, None, None, None, -1, 5, ctypes.byref(sp), None) == -4        # EMEI_ERR_BAD_SIZE
        assert seq(None, None, None, None, None, 8, 5, None, None) == -1                     # EMEI_ERR_NULL_POINTER (params)
        assert seq(None, None, None, None, None, 8, 5, ctypes.byref(sp), None) == -1         # obs_seq missing
        bad = _lib.ScoringParams()
        bad.family = 99
        assert seq(None, None, None, None, None, 8, 5, ctypes.byref(bad), None) == -2        # EMEI_ERR_BAD_VARIANT
        cp, rp, z = _lib.CartPoleParams(), _lib.RolloutParams(), _lib.NoiseParams()
        cp.freq_rate, cp.dt, cp.variant = 1, 0.02, _lib.CARTPOLE_SWINGUP
        ro = getattr(L, "emei_cartpole_rollout_ref" + sfx)
        args = [None] * 12
        assert ro(*args, 0, ctypes.byref(cp), ctypes.byref(rp), None, None) == -1            # episode buffers missing
        assert ro(*args, -3, ctypes.byref(cp), ctypes.byref(rp), None, None) == -4
        assert ro(*args, 4, ctypes.byref(cp), ctypes.byref(rp), ctypes.byref(z), None) == -2  # noise exists for the IP variants only
        ip = _lib.I2PParams()
        i2 = getattr(L, "emei_i2p_rollout" + sfx)
        Arr = ctypes.c_double * 6
        assert i2(*args, 4, ctypes.byref(ip), ctypes.byref(rp), Arr(), Arr(), None, None) == -2   # variant 0 is not an I2P variant
        assert i2(*args, 4, ctypes.byref(ip), ctypes.byref(rp), None, None, None, None) == -1
        cb = _lib.ChargedBallParams()
        cr = getattr(L, "emei_charged_ball_rollout_ref" + sfx)
        assert cr(*([None] * 14), 4, ctypes.byref(cb), ctypes.byref(rp), None) == -6         # EMEI_ERR_BAD_PARAM (freq_rate 0)


def test_plan_rollout_pieces():
    """core.EmeiEnv.plan_rollout_pieces: how a teacher-forced rollout with HOST actions is cut for upload / kernel overlap."""
    from emei_b200.core import EmeiEnv

    plan = EmeiEnv.plan_rollout_pieces
    mb = 1 << 20
    # C4's end-to-end leg: 25 steps of 2^26 uint8 actions (64 MB per step): 8-step pieces, a ragged last one
    assert plan(25, 64 * mb, 32 * mb, 8) == [(0, 8), (8, 16), (16, 24), (24, 25)]
    # cart-pole: 100 steps of 2^20 float32 actions (4 MB per step): 32 MB = 8 steps per piece
    p = plan(100, 4 * mb, 32 * mb, 8)
    assert p[0] == (0, 8) and p[-1] == (96, 100) and len(p) == 13
    assert all(a[1] == b[0] for a, b in zip(p, p[1:]))  # a tiling
    # small rollouts stay one upload + one launch
    assert plan(15, 64 * mb, 32 * mb, 8) is None        # fewer than two pieces
    assert plan(100, 4096, 32 * mb, 8) is None          # 400 KB in total
    assert plan(40, 3000, 9000, 1) == [(lo, min(40, lo + 3)) for lo in range(0, 40, 3)]  # the GPU test's shape
    assert plan(0, 4 * mb, 32 * mb, 8) is None
