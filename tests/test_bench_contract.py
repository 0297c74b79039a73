"""bench.py's contract: the reference arm prints exactly ONE JSON line on stdout with the agreed keys, for the default
workload and a scoring workload; --dump-outputs writes what the last timed step returned, reproducibly."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("workload", (None, "c3_hopper"))
def test_reference_arm_prints_one_json_line(workload):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"]
    if workload:
        cmd += ["--workload", workload]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["higher_is_better"] is True
    assert d["metric"] in ("env_steps_per_sec", "transitions_per_sec") and d["unit"].endswith("/s") and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "oracle" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("extra", (["--impl", "reference"], ["--workload", "c4"], ["--workload", "rollout"], ["--launch", "stream"]),
                         ids=("reference", "c4", "rollout", "stream"))
def test_dump_outputs_refuses_what_it_cannot_reproduce(extra, tmp_path):
    """The CPU arm is not the timed GPU path; c4, the rollouts and stream-launched steps start their timed steps from a state
    the time-boxed warm-up advanced: refused before any work, nothing written."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--dump-outputs", str(tmp_path / "d")] + extra,
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and out.stdout == ""
    assert not (tmp_path / "d").exists()


def test_dump_outputs_writes_floats_within_64_mb(tmp_path):
    import torch

    B = _bench_module()
    small = {"obs": torch.randn(300, 4), "reward": torch.randn(300, 1, dtype=torch.float64), "terminated": torch.rand(300, 1) > 0.5}
    B.dump_outputs(small, str(tmp_path / "small"))
    for k, v in small.items():
        a = np.load(tmp_path / "small" / f"{k}.npy")
        assert a.dtype == (np.float64 if v.dtype == torch.float64 else np.float32) and np.array_equal(a, v.numpy().astype(a.dtype))
    # 128 MB of outputs as float32: one seeded sample of half the rows, the same rows of both arrays, identical from call to call
    n = 1 << 24
    big = {"reward": torch.arange(n, dtype=torch.float32).reshape(n, 1), "terminated": (torch.arange(n) % 3 == 0).reshape(n, 1)}
    B.dump_outputs(big, str(tmp_path / "a"))
    B.dump_outputs(big, str(tmp_path / "b"))
    r, t = np.load(tmp_path / "a" / "reward.npy"), np.load(tmp_path / "a" / "terminated.npy")
    assert r.nbytes + t.nbytes == B.DUMP_BYTES and r.shape == t.shape == (n // 2, 1)
    assert np.all(np.diff(r[:, 0]) > 0) and np.array_equal(t[:, 0], (r[:, 0] % 3 == 0).astype(np.float32))
    assert np.array_equal(r, np.load(tmp_path / "b" / "reward.npy"))


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """Default workload (c2): the 3 warm-up steps advance envs 0-2 of the ring, so the last of 4 timed steps is env 3's first
    step from bench.py's seeded synthetic state; its dumped outputs agree with the CPU oracle at the float32 bar of
    tests/test_gpu_parity.py."""
    from oracle import emei_oracle as O

    d = tmp_path / "out"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", "4", "--warmup", "3",
                          "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout)["steps"] == 4
    assert sorted(os.listdir(d)) == ["obs.npy", "reward.npy", "terminated.npy"]
    obs, rew, term = (np.load(d / f"{k}.npy") for k in ("obs", "reward", "terminated"))
    n = 1 << 20
    assert obs.shape == (n, 4) and rew.shape == (n, 1) and term.shape == (n, 1) and obs.dtype == rew.dtype == term.dtype == np.float32
    st, act = _bench_module().synth_cartpole(n, 1002)
    st, act = np.roll(st, 3 * 4099, axis=0)[::16], np.roll(act, 3 * 4099, axis=0)[::16]
    p = O.cartpole_params("continuous_swingup")
    ref = O.cartpole_step_f64ref(st.astype(np.float64), O.cartpole_force(act, True, p), 0.02, 4, p)
    assert (np.abs(obs[::16] - ref) <= 1e-6 + 1e-5 * np.abs(ref)).all()
    r_ref = O.cartpole_reward("swingup", ref)
    assert (np.abs(rew[::16] - r_ref) <= 1e-6 + 1e-5 * np.abs(r_ref)).all()
    far = np.abs(np.abs(ref[:, 0]) - p.x_threshold) > 1e-4
    assert np.array_equal(term[::16][far] == 1, O.cartpole_terminal("swingup", ref, p)[far])
