#!/usr/bin/env python
"""bench.py -- benchmark of the emei_b200 hot path (contract: see the task statement / DESIGN.md 6).

Default workload = BASELINE.json configs[1] ("c2"): ContinuousCartPoleSwingUp batched step, 2^20 envs
per GPU, freq_rate=4 forward-Euler sub-steps, float32.  A "step" is one pass of the hot path over
one batch.  The other BASELINE configs are selectable with --workload (they are parity-test sizes
and secondary bench lines, committed under profiles/):

  c1            BoundaryInvertedPendulumSwingUp step, 4096 envs, freq_rate=1   (launch-latency bound)
  c2 (default)  ContinuousCartPoleSwingUp step, 2^20 envs/GPU, freq_rate=4
  c3_hopper     Hopper get_batch_reward+get_batch_terminal, 2^24 transitions/GPU (terminate_when_unhealthy=False)
  c3_halfcheetah  HalfCheetah same, 2^24 transitions/GPU
  c4            ChargedBallCentering step, 2^26 envs TOTAL sharded over the ranks (strong scaling)
  c5            scoring 2^26 transitions/GPU (half Hopper, half HalfCheetah) + freeze/unfreeze of a
                2^26-env cart-pole state buffer per sweep

  c3_*_seq      the same scoring on a trajectory tensor obs_seq[T+1, n, D] (T = 16, n = 2^20): every row read once
  c2_f64 etc.   --dtype f64 runs c1 / c2 / c3_* / c4 in the float64 reference-exact mode

  python bench.py [--gpus N --steps K --warmup W] [--workload W]          # our arm (torchrun for N>1)
  python bench.py --impl reference [--steps K --warmup W] [--workload W]  # CPU arm: the oracle port on host cores

One JSON line on stdout (rank 0).  With the default workload the line also carries `secondary`: one compact record
(value, ms_per_step, roofline, e2e, clocks) per other BASELINE config, measured in the same process under a time box
(N = 1: c1, c2 in float64, c3 Hopper / HalfCheetah in both layouts, c4, c4 as fused rollouts, c5; N > 1: c4 strong,
c4 rollouts strong, c5 weak), so that the driver's BENCH / SCALE files see every config.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DT = 0.02


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ==================================================================================================
# synthetic inputs (SURVEY.md 8d): generated on the host, seeded, identical bits for CPU and GPU arms
# ==================================================================================================
def synth_cartpole(n, seed=1002):
    """C2: [x, x', th, th'] = U(-1,1)*[4,5,pi,8] (+1% slice with |x| at the terminal threshold), action U(-1,1)."""
    rng = np.random.default_rng(seed)
    st = (rng.uniform(-1, 1, size=(n, 4)) * np.array([4.0, 5.0, np.pi, 8.0])).astype(np.float32)
    k = n // 100
    st[:k, 0] = np.sign(st[:k, 0]) * rng.uniform(4.99, 5.01, size=k).astype(np.float32)
    act = rng.uniform(-1, 1, size=(n, 1)).astype(np.float32)
    return st, act


def synth_ip(n, seed=1001):
    """C1: [x, th, v, w] = U(-1,1)*[1.9, pi, 5, 8], ctrl U(-3,3)."""
    rng = np.random.default_rng(seed)
    st = (rng.uniform(-1, 1, size=(n, 4)) * np.array([1.9, np.pi, 5.0, 8.0])).astype(np.float32)
    act = rng.uniform(-3, 3, size=(n, 1)).astype(np.float32)
    return st, act


def synth_i2p(n, seed=1006):
    """I2P: [x, th0, th1, v, w0, w1] = U(-1,1)*[2.9, pi, pi, 4, 8, 10], ctrl U(-1,1) (tests/test_gpu_parity.py i2p_inputs)."""
    rng = np.random.default_rng(seed)
    st = (rng.uniform(-1, 1, size=(n, 6)) * np.array([2.9, np.pi, np.pi, 4.0, 8.0, 10.0])).astype(np.float32)
    act = rng.uniform(-1, 1, size=(n, 1)).astype(np.float32)
    return st, act


def synth_scoring(n, family, seed=1003):
    """C3: Hopper obs = [0,1.25,0..] + N(0,1)*[1,.4,.15,1..]; HalfCheetah obs N(0,1)[n,18]; pre_obs = obs with
    column 0 shifted by N(0, 0.01); action U(-1,1); 0.1% rows poisoned with NaN/Inf."""
    rng = np.random.default_rng(seed + (0 if family == "hopper" else 1))
    d, da = (12, 3) if family == "hopper" else (18, 6)
    obs = rng.standard_normal((n, d), dtype=np.float32)
    if family == "hopper":
        obs *= np.array([1, 0.4, 0.15] + [1] * 9, dtype=np.float32)
        obs[:, 1] += 1.25
    pre = obs.copy()
    pre[:, 0] -= 0.01 * rng.standard_normal(n, dtype=np.float32)
    act = rng.uniform(-1, 1, size=(n, da)).astype(np.float32)
    bad = rng.integers(0, n, size=max(1, n // 1000))
    obs[bad, rng.integers(0, d, size=bad.shape[0])] = rng.choice(np.array([np.nan, np.inf, -np.inf], dtype=np.float32), size=bad.shape[0])
    return obs, pre, act


# ==================================================================================================
# CPU arm: the oracle port (numpy restatement of the reference) on the host cores.  bench.py's
# cpu_baseline / --impl reference are the ONLY product-side users of oracle/ (as the thing timed
# beside the GPU path, never inside it).
# ==================================================================================================
def cpu_port_name():
    """Which restatement the CPU legs time: the plain-C one (oracle/emei_oracle_c.c, built by build()) where it covers
    the workload and its library is present, else the numpy one."""
    try:
        from oracle import c_oracle as C

        return "C" if C.available() else "numpy"
    except Exception:
        return "numpy"


def cpu_port_desc(kind):
    if cpu_port_name() == "C" and kind in ("c2", "c1", "i2p", "c3_hopper", "c3_halfcheetah", "c4"):
        return f"plain-C oracle port (oracle/emei_oracle_c.c, kind={kind})"
    return f"numpy oracle port (oracle/emei_oracle.py, kind={kind})"


def _cpu_worker(args):
    kind, arrays, reps = args
    from oracle import emei_oracle as O

    C = None
    if cpu_port_name() == "C":
        from oracle import c_oracle as C

    t0 = time.perf_counter()
    for _ in range(reps):
        if kind == "c2":
            st, act = arrays
            p = O.cartpole_params("continuous_swingup")
            if C is not None:
                nxt = C.cartpole_step_f64ref(st, O.cartpole_force(act, True, p), DT, 4, p)
                C.cartpole_reward_terminal("continuous_swingup", nxt, p)
                continue
            nxt = O.cartpole_step_f64ref(st, O.cartpole_force(act, True, p), DT, 4, p, libm=False)
            O.cartpole_reward("continuous_swingup", nxt)
            O.cartpole_terminal("continuous_swingup", nxt, p)
        elif kind == "c1":
            st, act = arrays
            p = O.InvertedPendulumParams()
            if C is not None:
                nxt, obs = C.ip_step(st, np.clip(act[:, 0].astype(np.float64), p.ctrl_low, p.ctrl_high), DT, 1, True, p)
            else:
                nxt, obs = O.ip_step(st, act[:, 0].astype(np.float64), DT, 1, True, p)
            O.ip_reward("ip_boundary_swingup", obs)
            O.ip_terminal("ip_boundary_swingup", obs, p)
        elif kind == "i2p":
            st, act = arrays
            p = O.I2PParams()
            if C is not None:
                nxt, obs = C.i2p_step(st, act[:, 0].astype(np.float64), DT, 1, True, p)
            else:
                nxt, obs = O.i2p_step(st, act[:, 0].astype(np.float64), DT, 1, True, p)
            O.i2p_reward("i2p_boundary_swingup", obs)
            O.i2p_terminal("i2p_boundary_swingup", obs)
        elif kind == "c3_hopper":
            obs, pre, act = arrays
            p = O.HopperParams(terminate_when_unhealthy=False)
            if C is not None:
                C.hopper_reward_terminal(obs, pre, act, p)
                continue
            O.hopper_reward(obs, pre, act, p)
            O.hopper_terminal(obs, p)
        elif kind == "c3_halfcheetah":
            obs, pre, act = arrays
            p = O.HalfCheetahParams()
            if C is not None:
                C.halfcheetah_reward_terminal(obs, pre, act, p)
                continue
            O.halfcheetah_reward(obs, pre, act, p)
            O.halfcheetah_terminal(obs)
        elif kind == "c4":
            on, ci, fr, act = arrays
            p = O.ChargedBallParams()
            if C is not None:
                on, ci, fr = C.charged_ball_step(on, ci, fr, O.charged_ball_force(act, False, p), 1, p)
                C.charged_ball_reward(fr, p)
                continue
            on, ci, fr = O.charged_ball_step(on, ci, fr, O.charged_ball_force(act, False, p), 1, p)
            O.charged_ball_reward(fr, p)
        else:
            raise ValueError(kind)
    return time.perf_counter() - t0


def _cpu_inputs(kind, n):
    if kind == "c2":
        st, act = synth_cartpole(n)
        return [st.astype(np.float64), act]
    if kind == "c1":
        st, act = synth_ip(n)
        return [st.astype(np.float64), act]
    if kind == "i2p":
        st, act = synth_i2p(n)
        return [st.astype(np.float64), act]
    if kind in ("c3_hopper", "c3_halfcheetah"):
        obs, pre, act = synth_scoring(n, kind[3:])
        return [obs.astype(np.float64), pre.astype(np.float64), act.astype(np.float64)]
    if kind == "c4":
        from oracle import emei_oracle as O

        rng = np.random.default_rng(1004)
        on, ci, fr = O.charged_ball_init_state(n, rng, O.ChargedBallParams())
        return [on, ci, fr, rng.integers(0, 2, size=n)]
    raise ValueError(kind)


_CPU_CHUNKS = None


def _cpu_worker_indexed(i):
    return _cpu_worker(_CPU_CHUNKS[i])


def _cpu_worker_warm(i):
    kind, arrays, _ = _CPU_CHUNKS[i]
    return _cpu_worker((kind, [a[:256] for a in arrays], 1))


def cpu_rate(kind, sample_units, reps, cores):
    """units/s of the oracle port: `cores` processes, each owning sample_units/cores units."""
    import multiprocessing as mp

    global _CPU_CHUNKS
    arrays = _cpu_inputs(kind, sample_units)
    chunks = [(kind, [a[i::cores].copy() for a in arrays], reps) for i in range(cores)]
    with np.errstate(all="ignore"):
        if cores == 1:
            t0 = time.perf_counter()
            _cpu_worker(chunks[0])
            wall = time.perf_counter() - t0
        else:
            # the workers are forked AFTER the inputs exist and inherit them (copy-on-write): the timed map ships only
            # an index, not gigabytes of pickled arrays, so the CPU arm is timed on its arithmetic
            _CPU_CHUNKS = chunks
            with mp.get_context("fork").Pool(cores) as pool:
                pool.map(_cpu_worker_warm, range(cores))  # spin the workers up, touch the inherited pages
                t0 = time.perf_counter()
                pool.map(_cpu_worker_indexed, range(cores))
                wall = time.perf_counter() - t0
            _CPU_CHUNKS = None
    return sample_units * reps / wall, wall


# ==================================================================================================
# workloads
# ==================================================================================================
def _tdtype(args):
    import torch

    return torch.float64 if args.dtype == "f64" else torch.float32


class Workload:
    key = name = metric = unit = ""
    scaling = "weak"
    use_graph = True  # launch-bound steps: the K launches may be captured in one CUDA graph
    bound = "hbm"  # which roofline bounds the dominant kernel: "hbm" | "math" (no per-unit HBM traffic to speak of)
    alg_bytes = 0  # algorithmic bytes per unit (SURVEY.md 8d / DESIGN.md 4), float32
    alg_bytes_f64 = 0
    kernel = kernel_f64 = ""
    # algorithmic math per unit (SURVEY.md 8d): FP operations (an add, a multiply, an FMA or a divide is ONE op) and
    # special-function evaluations (sin, cos, rcp/div, sqrt, asin: one MUFU-class op each); None = trivial / not stated
    alg_fp_ops = alg_sfu_ops = alg_fp64_ops = None
    inst_per_unit = None  # thread-level SASS instructions per unit from ncu (issue utilisation, reported beside the roofline)
    cpu_kind = None  # which oracle routine is the CPU baseline
    cpu_sample = 1 << 20
    supports_f64 = False
    e2e_api = None
    units = 0  # units processed by THIS rank in one step
    stateful = False  # a step advances a state that the next step reads

    @classmethod
    def reproducible(cls, args):
        """Whether the timed steps start from the same inputs in every run with the same arguments.  The untimed warm-up
        before them runs until the clock sampler has delivered samples, a run-dependent number of steps: a stateful step
        is reproducible only when launched as a graph, whose input buffers restore_inputs() resets after that warm-up."""
        return not cls.stateful or (cls.use_graph and args.launch != "stream" and hasattr(cls, "restore_inputs"))

    def outputs(self):
        """name -> device tensor: what a caller of the timed path received from the last step."""
        raise NotImplementedError

    def __init__(self, args, rank, world, dev):
        self.args, self.rank, self.world, self.dev = args, rank, world, dev
        self.f64 = args.dtype == "f64"
        if self.f64 and not self.supports_f64:
            raise SystemExit(f"bench.py: workload {self.key} has no float64 mode (the fused rollouts are float32)")

    def setup(self):
        raise NotImplementedError

    def step(self, i):
        raise NotImplementedError

    def setup_e2e(self):
        self.h2d = self.d2h = 0
        self.e2e_api = None

    def step_e2e(self, i):
        raise NotImplementedError

    def teardown(self):
        """drop every device / pinned buffer (the next workload of a `secondary` sweep needs the memory)"""
        for k in list(self.__dict__):
            if k not in ("args", "rank", "world", "dev", "f64"):
                delattr(self, k)

    # ---- config: a pure function of (class, args, world) so that the CPU reference arm prints the SAME dict
    @classmethod
    def config(cls, args, world):
        return {}

    @classmethod
    def units_per_step_total(cls, args, world):
        """units of one step over all ranks (what the reference arm processes per step)"""
        raise NotImplementedError

    def bytes_per_unit(self):
        return self.alg_bytes_f64 if self.f64 else self.alg_bytes

    def kernel_name(self):
        return self.kernel_f64 if self.f64 else self.kernel


class CartPoleStep(Workload):
    """C2 (and, with the IP env, C1): ring of independent batches larger than L2, rotated every launch."""

    key, metric, unit = "c2", "env_steps_per_sec", "env-steps/s"
    title = "ContinuousCartPoleSwingUp batched step, 2^20 envs/GPU, freq_rate=4 (BASELINE configs[1])"
    kernel = "emei::cartpole_step_f32_tma_kernel<IP=0, AK=f32, FR=4, HAS_OBS=0>"
    kernel_f64 = "emei::cartpole_step_kernel<double, IP=0> (reference-exact mixed arithmetic, -fmad=false)"
    env_id, n_envs, freq_rate, ring = "ContinuousCartPoleSwingUp-v0", 1 << 20, 4, 8
    alg_bytes = 41  # state 16 + action 4 + next 16 + reward 4 + done 1
    alg_bytes_f64 = 77  # state 32 + action 4 + next 32 + reward 8 + done 1
    # cartpole.py:48-60 per sub-step: 26 FP ops of which 4 divides, 1 sin + 1 cos; + reward cos and 2 ops, terminal 2 ops
    alg_fp_ops = 4 * 26 + 4
    alg_sfu_ops = 4 * (2 + 4) + 1
    alg_fp64_ops = 4 * (22 + 4 * 10 + 2 * 20) + 20 + 4  # float64: 22 plain ops + 4 divides + sin + cos per sub-step; reward cos
    cpu_kind = "c2"
    supports_f64 = True
    inst_per_unit = 165.8  # 32 x smsp__inst_executed / envs, packed f32x2 (ncu, profiles/r02_ncu_full_c2.txt: 5 432 964 warp instructions per 2^20-env launch)
    stateful = True

    def synth(self, seed):
        return synth_cartpole(self.n_envs, seed)

    def setup(self):
        import torch

        import emei_b200 as E

        self.units = self.n_envs
        ring = self.args.ring or self.ring
        st, act = self.synth(1002 + self.rank)
        self.envs, self.acts = [], []
        for j in range(ring):
            env = E.make(self.env_id, freq_rate=self.freq_rate, real_time_scale=DT, num_envs=self.n_envs, dtype=_tdtype(self.args),
                         device=self.dev, env_offset=(self.rank * ring + j) * self.n_envs, copy_outputs=False)
            env.state = np.roll(st, j * 4099, axis=0)
            env._stats = self.envs[0].stats if self.envs else env.stats  # one shared statistics buffer
            self.envs.append(env)
            self.acts.append(torch.as_tensor(np.roll(act, j * 4099, axis=0)).to(self.dev).reshape(self.n_envs))
        self.envs[0].reset_stats()
        self.stats = self.envs[0].stats
        self._act_host = act

    def step(self, i):
        j = i % len(self.envs)
        self.out = self.envs[j].step(self.acts[j])

    def outputs(self):
        obs, reward, terminated = self.out[:3]
        return {"obs": obs, "reward": reward, "terminated": terminated}

    def restore_inputs(self):
        """Put the synthetic states of SURVEY 8(d) back into the buffers the first timed step of every env reads (outside the
        timed region).  The step kernels never reset, and the warm-up replays advance every env by hundreds of steps under
        constant actions: poles spin up beyond the integrator's guard (|theta_dot| > 39 rad/s) and the timed steps would
        measure the cold redo path instead of the workload's state distribution."""
        if getattr(self, "_restore", None) is None:  # first call (before capture): remember the buffers and their contents
            self._restore = [(e._engine._bufs[e._engine._cur], e._engine._bufs[e._engine._cur].clone()) for e in self.envs]
        for buf, init in self._restore:
            buf.copy_(init)

    def setup_e2e(self):
        import torch

        a = self._act_host
        self.act_host = [torch.as_tensor(np.roll(a, j * 4099, axis=0).reshape(self.n_envs)).pin_memory() for j in range(4)]
        self.env0 = self.envs[0]
        self.env0.step_host(self.act_host[0])
        self.h2d, self.d2h = self.env0._staging.h2d_bytes, self.env0._staging.d2h_bytes
        self.e2e_api = ("env.step_host(action_host) -> numpy obs/reward/terminated (pinned staging; >= 2^17 envs: chunked copy/compute overlap through the "
                        "copy engines; <= 2^16 envs: the kernel loads / stores the pinned host arrays itself)")

    e2e_warmup = 24  # 4 pinned action buffers x 2 ping-pong sides, each seen eagerly, captured, replayed

    def step_e2e(self, i):
        self.env0.step_host(self.act_host[i % len(self.act_host)])

    # the same host step for a caller that consumes reward and done only (evaluation of a policy's return): the
    # observation stays on the device -- 5 bytes per env come back instead of 21
    e2e_light_api = "env.step_host(action_host, outputs=('reward', 'done')) -> numpy reward/terminated; obs stays on the device"

    def step_e2e_light(self, i):
        self.env0.step_host(self.act_host[i % len(self.act_host)], outputs=("reward", "done"))

    @classmethod
    def config(cls, args, world):
        ring = args.ring or cls.ring
        bpu = cls.alg_bytes_f64 if args.dtype == "f64" else cls.alg_bytes
        mb = ring * cls.n_envs * bpu / 1e6
        return {
            "envs_per_gpu": cls.n_envs, "freq_rate": cls.freq_rate, "real_time_scale": DT,
            "l2_policy": f"inputs larger than L2: ring of {ring} independent {cls.n_envs}-env batches ({mb:.0f} MB of step traffic) rotated every launch; "
                         "L2 flushed before the timed region (256 MB written, then 64 MB read: half of the L2 is left dirty, as in the steady state)",
        }

    @classmethod
    def units_per_step_total(cls, args, world):
        return cls.n_envs * world


class IPStep(CartPoleStep):
    key = "c1"
    title = "BoundaryInvertedPendulumSwingUp batched step, 4096 envs, freq_rate=1 (BASELINE configs[0])"
    kernel = "emei::cartpole_step_f32_small_kernel<IP=1, AK=f32, FR=1, HAS_OBS=1>"
    kernel_f64 = "emei::cartpole_step_kernel<double, IP=1>"
    env_id, n_envs, freq_rate, ring = "BoundaryInvertedPendulumSwingUp-v0", 4096, 1, 1024
    alg_bytes = 57  # state 16 + action 4 + next state 16 + wrapped obs 16 + reward 4 + done 1
    alg_bytes_f64 = 109
    alg_fp_ops, alg_sfu_ops = 26 + 4 + 3, (2 + 4) + 1
    alg_fp64_ops = (22 + 4 * 10 + 2 * 20) + 20 + 4 + 10  # + the observation's floored modulo
    cpu_kind, cpu_sample = "c1", 1 << 20
    inst_per_unit = 202.5  # one env per thread, 128-thread CTAs: profiles/r01_launches_bench_c1.csv

    def synth(self, seed):
        return synth_ip(self.n_envs, seed)


class CartPoleStepLarge(CartPoleStep):
    """The C2 step at 2^24 envs per GPU: launch ramp and drain amortised, the kernel's steady state (recycled TMA ring)."""

    key = "c2_large"
    title = "ContinuousCartPoleSwingUp batched step, 2^24 envs/GPU, freq_rate=4 (C2's kernel at 16x the batch)"
    n_envs, ring = 1 << 24, 2
    use_graph = False


class I2PStep(CartPoleStep):
    """SURVEY 8f rank 3: the analytic inverted double pendulum step (dynamics + observation + reward/terminal in one
    launch), same protocol as C2."""

    key = "i2p"
    title = "BoundaryInvertedDoublePendulumSwingUp batched step, 2^20 envs/GPU, freq_rate=1 (SURVEY 8f rank 3)"
    kernel = "emei::i2p_step_kernel<float>"
    kernel_f64 = "emei::i2p_step_kernel<double>"
    env_id, n_envs, freq_rate, ring = "BoundaryInvertedDoublePendulumSwingUp-v0", 1 << 20, 1, 8
    alg_bytes = 81  # state 24 + action 4 + next state 24 + observation 24 + reward 4 + done 1
    alg_bytes_f64 = 157
    alg_fp_ops = alg_sfu_ops = None  # SURVEY 8d states no operation count for the 3x3 Lagrangian solve
    cpu_kind, cpu_sample = "i2p", 1 << 18
    inst_per_unit = 334.6  # 32 x smsp__inst_executed / envs (ncu, profiles/r02_ncu_full_i2p.txt: 10 963 240 warp instructions per 2^20-env launch)

    def synth(self, seed):
        return synth_i2p(self.n_envs, seed)


class Scoring(Workload):
    """C3: get_batch_reward + get_batch_terminal over n transitions resident in HBM (>> L2), through the reference's
    one-shot signature (obs, pre_obs, action) with pre_obs a SEPARATE array."""

    metric, unit = "transitions_per_sec", "transitions/s"
    use_graph = False
    family, n = "hopper", 1 << 24
    env_kwargs = {}
    supports_f64 = True

    def setup(self):
        import torch

        import emei_b200 as E

        self.units = self.n
        self.env = E.make(self.env_id, dtype=_tdtype(self.args), device=self.dev, **self.env_kwargs)
        obs, pre, act = synth_scoring(self.n, self.family, 1003 + 17 * self.rank)
        self._host = (obs, pre, act)
        self.obs, self.pre, self.act = (torch.as_tensor(a).to(self.dev).to(_tdtype(self.args)) for a in (obs, pre, act))
        self.stats = self.env.stats

    def step(self, i):
        self.out = self.env.get_batch_reward_terminal(self.obs, self.pre, self.act)

    def outputs(self):
        return {"reward": self.out[0], "terminated": self.out[1]}

    def setup_e2e(self):
        import torch

        dt = _tdtype(self.args)
        self.h_in = [torch.as_tensor(a).to(dt).pin_memory() for a in self._host]
        self.h_r = torch.empty((self.n, 1), dtype=dt).pin_memory()
        self.h_d = torch.empty((self.n, 1), dtype=torch.bool).pin_memory()
        self.h2d = sum(t.numel() * t.element_size() for t in self.h_in)
        self.d2h = self.h_r.numel() * self.h_r.element_size() + self.h_d.numel()
        self.e2e_api = "env.get_batch_reward_terminal(obs, pre_obs, action) with pinned HOST tensors -> reward/terminal copied back to pinned host"

    def step_e2e(self, i):
        import torch

        r, d = self.env.get_batch_reward_terminal(*self.h_in)
        self.h_r.copy_(r, non_blocking=True)
        self.h_d.copy_(d, non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()

    @classmethod
    def config(cls, args, world):
        bpu = cls.alg_bytes_f64 if args.dtype == "f64" else cls.alg_bytes
        return {"transitions_per_gpu": cls.n, "l2_policy": f"inputs larger than L2 ({cls.n * bpu / 1e6:.0f} MB per sweep)",
                "note": "step = emei_sumsq (batch-wide control cost, 1 launch) + fused emei_reward_terminal (1 launch); the roofline counts the WHOLE step"}

    @classmethod
    def units_per_step_total(cls, args, world):
        return cls.n * world


class HopperScoring(Scoring):
    key, family, env_id = "c3_hopper", "hopper", "HopperRunning-v0"
    title = "Hopper get_batch_reward+get_batch_terminal, 2^24 transitions/GPU, terminate_when_unhealthy=False (BASELINE configs[2])"
    kernel = "emei::sumsq_kernel<float> + emei::reward_terminal_kernel<float, HOPPER>"
    kernel_f64 = "emei::sumsq_kernel<double> + emei::reward_terminal_kernel<double, HOPPER>"
    env_kwargs = {"terminate_when_unhealthy": False}
    alg_bytes = 69  # obs 48 + pre_obs[:,0] 4 + action 12 + reward 4 + done 1
    alg_bytes_f64 = 137
    cpu_kind, cpu_sample = "c3_hopper", 1 << 22


class HalfCheetahScoring(Scoring):
    key, family, env_id = "c3_halfcheetah", "halfcheetah", "HalfCheetahRunning-v0"
    title = "HalfCheetah get_batch_reward+get_batch_terminal, 2^24 transitions/GPU (BASELINE configs[2])"
    kernel = "emei::sumsq_kernel<float> + emei::reward_terminal_kernel<float, HALFCHEETAH>"
    kernel_f64 = "emei::sumsq_kernel<double> + emei::reward_terminal_kernel<double, HALFCHEETAH>"
    alg_bytes = 105  # obs 72 + pre_obs[:,0] 4 + action 24 + reward 4 + done 1
    alg_bytes_f64 = 209
    cpu_kind, cpu_sample = "c3_halfcheetah", 1 << 22


class SeqScoring(Scoring):
    """C3 on the layout an MBRL scorer holds its imagined rollouts in: obs_seq [T+1, n, D], action [T, n, A]
    (T = 16, n = 2^20: the same 2^24 transitions).  pre_obs of step t IS obs of step t-1, so a thread that walks the
    time steps of its env reads every observation row once: no pre_obs traffic at all."""

    T, n_env = 16, 1 << 20

    def setup(self):
        import torch

        import emei_b200 as E

        self.units = self.n = self.T * self.n_env
        dt = _tdtype(self.args)
        self.env = E.make(self.env_id, dtype=dt, device=self.dev, **self.env_kwargs)
        g = torch.Generator(device=self.dev)
        g.manual_seed(1003 + 17 * self.rank)
        d, da = (12, 3) if self.family == "hopper" else (18, 6)
        seq = torch.randn((self.T + 1, self.n_env, d), device=self.dev, dtype=torch.float32, generator=g)
        if self.family == "hopper":
            seq *= torch.tensor([1, 0.4, 0.15] + [1] * 9, device=self.dev)
            seq[:, :, 1] += 1.25
        bad = torch.randint(0, seq.numel(), (max(1, seq.numel() // 12000),), device=self.dev, generator=g)
        seq.view(-1)[bad] = float("nan")  # poisoned rows (SURVEY 8d): 0.1 % of the transitions
        self.seq = seq.to(dt)
        self.act = (torch.rand((self.T, self.n_env, da), device=self.dev, generator=g) * 2 - 1).to(dt)
        self.stats = self.env.stats

    def step(self, i):
        self.out = self.env.get_batch_reward_terminal_seq(self.seq, self.act)

    def setup_e2e(self):
        import torch

        self.h_in = [self.seq.cpu().pin_memory(), self.act.cpu().pin_memory()]
        self.h_r = torch.empty((self.T, self.n_env, 1), dtype=self.seq.dtype).pin_memory()
        self.h_d = torch.empty((self.T, self.n_env, 1), dtype=torch.bool).pin_memory()
        self.h2d = sum(t.numel() * t.element_size() for t in self.h_in)
        self.d2h = self.h_r.numel() * self.h_r.element_size() + self.h_d.numel()
        self.e2e_api = "env.get_batch_reward_terminal_seq(obs_seq, action) with pinned HOST tensors -> reward/terminal copied back to pinned host"

    def step_e2e(self, i):
        import torch

        r, d = self.env.get_batch_reward_terminal_seq(*self.h_in)
        self.h_r.copy_(r, non_blocking=True)
        self.h_d.copy_(d, non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()

    @classmethod
    def config(cls, args, world):
        bpu = cls.alg_bytes_f64 if args.dtype == "f64" else cls.alg_bytes
        return {"transitions_per_gpu": cls.T * cls.n_env, "layout": f"obs_seq [T+1={cls.T + 1}, n={cls.n_env}, D], action [T, n, A]",
                "l2_policy": f"inputs larger than L2 ({cls.T * cls.n_env * bpu / 1e6:.0f} MB per sweep)",
                "note": "step = emei_sumsq (1 launch) + emei_reward_terminal_seq (1 launch); the roofline counts the WHOLE step"}

    @classmethod
    def units_per_step_total(cls, args, world):
        return cls.T * cls.n_env * world


class HopperSeqScoring(SeqScoring):
    key, family, env_id = "c3_hopper_seq", "hopper", "HopperRunning-v0"
    title = "Hopper reward+terminal of imagined rollouts obs_seq[17, 2^20, 12] = 2^24 transitions/GPU, terminate_when_unhealthy=False (BASELINE configs[2], trajectory layout)"
    kernel = "emei::sumsq_kernel<float> + emei::reward_terminal_seq_kernel<float, HOPPER>"
    kernel_f64 = "emei::sumsq_kernel<double> + emei::reward_terminal_seq_kernel<double, HOPPER>"
    env_kwargs = {"terminate_when_unhealthy": False}
    alg_bytes = 65 + 48 / 16  # obs 48 + action 12 + reward 4 + done 1, + the t = 0 row once per 16 steps
    alg_bytes_f64 = 129 + 96 / 16
    cpu_kind, cpu_sample = "c3_hopper", 1 << 22


class HalfCheetahSeqScoring(SeqScoring):
    key, family, env_id = "c3_halfcheetah_seq", "halfcheetah", "HalfCheetahRunning-v0"
    title = "HalfCheetah reward+terminal of imagined rollouts obs_seq[17, 2^20, 18] = 2^24 transitions/GPU (BASELINE configs[2], trajectory layout)"
    kernel = "emei::sumsq_kernel<float> + emei::reward_terminal_seq_kernel<float, HALFCHEETAH>"
    kernel_f64 = "emei::sumsq_kernel<double> + emei::reward_terminal_seq_kernel<double, HALFCHEETAH>"
    alg_bytes = 101 + 72 / 16
    alg_bytes_f64 = 201 + 144 / 16
    cpu_kind, cpu_sample = "c3_halfcheetah", 1 << 22


class ChargedBall(Workload):
    """C4: 2^26 envs in total, sharded contiguously over the ranks (strong scaling); state updated in place."""

    key, metric, unit = "c4", "env_steps_per_sec", "env-steps/s"
    title = "ChargedBallCentering batched step, 2^26 envs total sharded over the ranks, freq_rate=1 (BASELINE configs[3])"
    kernel = "emei::charged_ball_step_f32_kernel<AK=u8>"
    kernel_f64 = "emei::charged_ball_step_kernel<double, F32FORCE=0>"
    scaling, use_graph = "strong", False
    total = 1 << 26
    alg_bytes = 56  # state in 25 + action 1 (uint8) + state out 25 + reward 4 + done 1
    alg_bytes_f64 = 108  # state 49 + 1 + 49 + 8 + 1
    # charged_ball.py:68-82 on the ring: sin, cos of theta before and after the update (4), 1 divide, ~20 FP ops;
    # reward: 1 sqrt + 1 divide (:158-160)
    alg_fp_ops, alg_sfu_ops = 22, 4 + 1 + 2
    alg_fp64_ops = 20 + 4 * 20 + 10 + 2 * 10
    cpu_kind, cpu_sample = "c4", 1 << 20
    supports_f64 = True
    stateful = True

    @classmethod
    def _total(cls, args):
        return 1 << args.total_log2 if args.total_log2 else cls.total

    def setup(self):
        import torch

        import emei_b200 as E
        from emei_b200.dist import shard_range

        self.total = self._total(self.args)
        b, e = shard_range(self.total, self.rank, self.world)
        self.units = e - b
        self.env = E.make("ChargedBallCentering-v0", num_envs=self.units, dtype=_tdtype(self.args), device=self.dev, env_offset=b,
                          copy_outputs=False)
        self.env.reset(seed=1004)
        g = torch.Generator(device=self.dev)
        g.manual_seed(1004 + self.rank)
        self.acts = [torch.randint(0, 2, (self.units,), device=self.dev, dtype=torch.uint8, generator=g) for _ in range(4)]
        self.env.reset_stats()
        self.stats = self.env.stats

    def step(self, i):
        self.env.step(self.acts[i % 4])

    def setup_e2e(self):
        self.act_host = [a.cpu().pin_memory() for a in self.acts]
        self.env.step_host(self.act_host[0])
        self.h2d, self.d2h = self.env._staging.h2d_bytes, self.env._staging.d2h_bytes
        self.e2e_api = "env.step_host(action_host) -> numpy obs/reward/terminated (pinned staging)"

    e2e_warmup = 8  # 4 pinned action buffers, each seen eagerly once, then captured

    def step_e2e(self, i):
        self.env.step_host(self.act_host[i % 4])

    @classmethod
    def config(cls, args, world):
        tot = cls._total(args)
        bpu = cls.alg_bytes_f64 if args.dtype == "f64" else cls.alg_bytes
        return {"envs_total": tot, "envs_per_gpu": tot // world, "freq_rate": 1,
                "l2_policy": f"inputs larger than L2 ({tot // world * bpu / 1e6:.0f} MB per step per GPU)"}

    @classmethod
    def units_per_step_total(cls, args, world):
        return cls._total(args)


class ScoringSweep(Workload):
    """C5: one imagined-rollout scoring sweep per step = freeze() of a 2^26-env cart-pole state buffer,
    Hopper + HalfCheetah reward/terminal over 2^25 transitions each, unfreeze()."""

    key, metric, unit = "c5", "transitions_per_sec", "transitions/s"
    title = "MBRL scoring sweep: 2^26 transitions/GPU (half Hopper, half HalfCheetah) reward+terminal + freeze/unfreeze of a 2^26-env cart-pole buffer (BASELINE configs[4])"
    kernel = "emei::reward_terminal_kernel<float, HALFCHEETAH> (dominant), HOPPER, sumsq, snapshot_copy"
    use_graph = False
    n_half, n_env = 1 << 25, 1 << 26
    # per transition: (69 + 105)/2 scoring + 2 x (16 read + 16 write) snapshot bytes per env over n_env == 2*n_half transitions
    alg_bytes = (69 + 105) / 2 + 64
    cpu_kind, cpu_sample = "c3_hopper", 1 << 22
    e2e_half = 1 << 22  # transitions per family of the host-buffer sample

    def setup(self):
        import torch

        import emei_b200 as E

        self.units = 2 * self.n_half
        self.hop = E.make("HopperRunning-v0", terminate_when_unhealthy=False, dtype=torch.float32, device=self.dev)
        self.chee = E.make("HalfCheetahRunning-v0", dtype=torch.float32, device=self.dev)
        self.cp = E.make("CartPoleSwingUp-v0", num_envs=self.n_env, dtype=torch.float32, device=self.dev, copy_outputs=False)
        self.cp.reset(seed=1005)
        self.data = []
        for fam in ("hopper", "halfcheetah"):
            obs, pre, act = synth_scoring(self.n_half, fam, 1005 + 31 * self.rank)
            self.data.append(tuple(torch.as_tensor(a).to(self.dev) for a in (obs, pre, act)))
        self.stats = self.hop.stats

    def step(self, i):
        self.cp.freeze()
        self.o1 = self.hop.get_batch_reward_terminal(*self.data[0])
        self.o2 = self.chee.get_batch_reward_terminal(*self.data[1])
        self.cp.unfreeze()

    def outputs(self):
        return {"hopper_reward": self.o1[0], "hopper_terminated": self.o1[1],
                "halfcheetah_reward": self.o2[0], "halfcheetah_terminated": self.o2[1]}

    def setup_e2e(self):
        import torch

        m = self.e2e_half
        self.h_in = [[t[:m].cpu().pin_memory() for t in fam] for fam in self.data]
        self.h_out = [(torch.empty((m, 1), dtype=torch.float32).pin_memory(), torch.empty((m, 1), dtype=torch.bool).pin_memory()) for _ in range(2)]
        self.h2d = sum(t.numel() * t.element_size() for fam in self.h_in for t in fam)
        self.d2h = 2 * m * 5
        self.e2e_units = 2 * m
        self.e2e_api = (f"freeze(); hopper / halfcheetah get_batch_reward_terminal on pinned HOST tensors ({m} transitions each: a bounded "
                        "sample of the sweep, the rate is per transition) -> results copied back to pinned host; unfreeze()")

    def step_e2e(self, i):
        import torch

        self.cp.freeze()
        for env, h_in, (h_r, h_d) in zip((self.hop, self.chee), self.h_in, self.h_out):
            r, d = env.get_batch_reward_terminal(*h_in)
            h_r.copy_(r, non_blocking=True)
            h_d.copy_(d, non_blocking=True)
        self.cp.unfreeze()
        torch.cuda.current_stream(self.dev).synchronize()

    @classmethod
    def config(cls, args, world):
        return {"transitions_per_gpu": 2 * cls.n_half, "snapshot_envs_per_gpu": cls.n_env,
                "l2_policy": "inputs larger than L2 (10 GB per sweep)"}

    @classmethod
    def units_per_step_total(cls, args, world):
        return 2 * cls.n_half * world


class ScoringSweepSeq(ScoringSweep):
    """C5 with the imagined rollouts held as trajectory tensors obs_seq [17, 2^21, D] per family (the layout an MBRL
    scorer produces them in): get_batch_reward_terminal_seq reads every observation row once."""

    key = "c5_seq"
    title = ScoringSweep.title.replace("reward+terminal", "reward+terminal on trajectory tensors obs_seq[17, 2^21, D]")
    kernel = "emei::reward_terminal_seq_kernel<float, HALFCHEETAH> (dominant), HOPPER, sumsq, snapshot_copy"
    T, n_traj = 16, 1 << 21
    alg_bytes = ((65 + 48 / 16) + (101 + 72 / 16)) / 2 + 64

    def setup(self):
        import torch

        import emei_b200 as E

        self.units = 2 * self.n_half
        assert self.T * self.n_traj == self.n_half
        self.hop = E.make("HopperRunning-v0", terminate_when_unhealthy=False, dtype=torch.float32, device=self.dev)
        self.chee = E.make("HalfCheetahRunning-v0", dtype=torch.float32, device=self.dev)
        self.cp = E.make("CartPoleSwingUp-v0", num_envs=self.n_env, dtype=torch.float32, device=self.dev, copy_outputs=False)
        self.cp.reset(seed=1005)
        g = torch.Generator(device=self.dev)
        g.manual_seed(1005 + 31 * self.rank)
        self.data = []
        for d, da in ((12, 3), (18, 6)):
            seq = torch.randn((self.T + 1, self.n_traj, d), device=self.dev, generator=g)
            if d == 12:
                seq[:, :, 1] += 1.25
            self.data.append((seq, torch.rand((self.T, self.n_traj, da), device=self.dev, generator=g) * 2 - 1))
        self.stats = self.hop.stats

    def step(self, i):
        self.cp.freeze()
        self.o1 = self.hop.get_batch_reward_terminal_seq(*self.data[0])
        self.o2 = self.chee.get_batch_reward_terminal_seq(*self.data[1])
        self.cp.unfreeze()

    def setup_e2e(self):
        import torch

        m_traj = self.e2e_half // self.T  # trajectories per family of the host-buffer sample
        self.h_in = [[seq[:, :m_traj].contiguous().cpu().pin_memory(), act[:, :m_traj].contiguous().cpu().pin_memory()] for seq, act in self.data]
        m = m_traj * self.T
        self.h_out = [(torch.empty((m, 1), dtype=torch.float32).pin_memory(), torch.empty((m, 1), dtype=torch.bool).pin_memory()) for _ in range(2)]
        self.h2d = sum(t.numel() * t.element_size() for fam in self.h_in for t in fam)
        self.d2h = 2 * m * 5
        self.e2e_units = 2 * m
        self.e2e_api = (f"freeze(); hopper / halfcheetah get_batch_reward_terminal_seq on pinned HOST trajectory tensors ({m_traj} trajectories x {self.T} steps "
                        "each: a bounded sample of the sweep, the rate is per transition) -> results copied back to pinned host; unfreeze()")

    def step_e2e(self, i):
        import torch

        self.cp.freeze()
        for env, h_in, (h_r, h_d) in zip((self.hop, self.chee), self.h_in, self.h_out):
            r, d = env.get_batch_reward_terminal_seq(*h_in)
            h_r.copy_(r.reshape(-1, 1), non_blocking=True)
            h_d.copy_(d.reshape(-1, 1), non_blocking=True)
        self.cp.unfreeze()
        torch.cuda.current_stream(self.dev).synchronize()

    @classmethod
    def config(cls, args, world):
        c = ScoringSweep.config.__func__(cls, args, world)
        c["layout"] = f"obs_seq [T+1={cls.T + 1}, n={cls.n_traj}, D], action [T, n, A] per family"
        c["l2_policy"] = "inputs larger than L2 (8 GB per sweep)"
        return c


class CartPoleRollout(Workload):
    """SURVEY 8f rank 1: the collection loop (zoo/util.py:33-93) as ONE launch per `horizon` env-steps: state,
    TimeLimit counter and episode return in registers, in-kernel auto-reset and uniform random policy.  No
    per-step HBM traffic (24 B per env per launch), so the bound is math."""

    key, metric, unit = "rollout", "env_steps_per_sec", "env-steps/s"
    title = "ContinuousCartPoleSwingUp fused rollout, 2^20 envs/GPU x horizon steps per launch, freq_rate=4, in-kernel random policy + TimeLimit(1000) + auto-reset (SURVEY 8f rank 1)"
    kernel = "emei::rollout_f32_kernel<CartPoleDyn<IP=0, AK=f32, FR=4>, RECORD=0>"
    kernel_f64 = "emei::rollout_ref_kernel<RefCartPole<double, IP=0>> (the float64 step's own arithmetic, one env per thread)"
    env_id, n_envs, freq_rate = "ContinuousCartPoleSwingUp-v0", 1 << 20, 4
    use_graph, bound = False, "math"
    record = False
    supports_f64 = True
    state_bytes = 16
    alg_fp_ops, alg_sfu_ops, alg_fp64_ops = CartPoleStep.alg_fp_ops, CartPoleStep.alg_sfu_ops, CartPoleStep.alg_fp64_ops
    inst_per_unit = 185.8  # thread-level SASS instructions per env-step incl. in-kernel resets (ncu, profiles/r02_launches_rollout.csv; 247.1 before the spare reset samples)
    cpu_kind = "c2"
    e2e_max_steps = 5
    stateful = True

    @classmethod
    def _horizon(cls, args):
        return args.horizon if args.horizon_set else (32 if cls.record else 100)

    def setup(self):
        import torch

        import emei_b200 as E

        self.T = self._horizon(self.args)
        self.units = self.n_envs * self.T
        self.env = E.make(self.env_id, freq_rate=self.freq_rate, real_time_scale=DT, num_envs=self.n_envs,
                          dtype=_tdtype(self.args), device=self.dev, env_offset=self.rank * self.n_envs)
        self.env.reset(seed=1006)
        self.stats = self.env.stats
        # state + 3 counters 12, read and written once per launch; records (if any) per env-step
        sb = self.state_bytes * (2 if self.f64 else 1)
        self.alg_bytes = self.alg_bytes_f64 = 2 * (sb + 12) / self.T + (42 if self.record else 0)

    def step(self, i):
        self.out = self.env.rollout(self.T, record=self.record)

    def setup_e2e(self):
        import torch

        if self.record:
            return Workload.setup_e2e(self)
        rng = np.random.default_rng(1006 + self.rank)
        self.act_host = [torch.as_tensor(rng.uniform(-1, 1, size=(self.T, self.n_envs)).astype(np.float32)).pin_memory() for _ in range(2)]
        self.h2d = self.act_host[0].numel() * 4
        self.d2h = 48
        self.e2e_api = "env.rollout(horizon, actions=pinned HOST [T,n] float32) -> env.rollout_info(stats) read on the host (the horizon is cut into pieces whose uploads run one piece ahead of the kernels)"

    def step_e2e(self, i):
        out = self.env.rollout(self.T, actions=self.act_host[i % 2])
        self.info = self.env.rollout_info(out["stats"])

    @classmethod
    def config(cls, args, world):
        T = cls._horizon(args)
        return {"envs_per_gpu": cls.n_envs, "horizon": T, "freq_rate": cls.freq_rate, "max_episode_steps": 1000,
                "records": cls.record,
                "l2_policy": "no reuse to defeat: every env's state is read once and written once per launch"
                             + (f"; records are {cls.n_envs * T * 42 / 1e6:.0f} MB of fresh writes per launch" if cls.record else "")}

    @classmethod
    def units_per_step_total(cls, args, world):
        return cls.n_envs * cls._horizon(args) * world


class I2PRollout(CartPoleRollout):
    """The four inverted-double-pendulum tasks of zoo/conf/task/BI2P*.yaml through the collection loop, one launch
    (emei_i2p_rollout_*): the step kernel's arithmetic, one env per thread."""

    key = "i2p_rollout"
    title = "BoundaryInvertedDoublePendulumSwingUp fused rollout, 2^20 envs/GPU x horizon steps per launch, freq_rate=1, in-kernel random policy + TimeLimit + auto-reset (SURVEY 8f ranks 1+3)"
    kernel = "emei::rollout_ref_kernel<RefI2P<float>>"
    kernel_f64 = "emei::rollout_ref_kernel<RefI2P<double>>"
    env_id, freq_rate = "BoundaryInvertedDoublePendulumSwingUp-v0", 1
    state_bytes = 24
    alg_fp_ops = alg_sfu_ops = alg_fp64_ops = None
    bound = "hbm"  # no stated operation count for the 3x3 solve: reported against the (tiny) HBM traffic + issue utilisation only
    inst_per_unit = None
    cpu_kind = "i2p"

    def setup_e2e(self):
        return Workload.setup_e2e(self)


class CartPoleRolloutRecord(CartPoleRollout):
    """Same launch, additionally writing every transition in the reference's dataset layout (zoo/util.py:62-67):
    observations/next_observations [T,n,4], actions/rewards [T,n], dones/timeouts u8[T,n] = 42 B per env-step."""

    key = "rollout_rec"
    title = CartPoleRollout.title.replace("fused rollout", "fused rollout + transition records (dataset layout)")
    kernel = "emei::rollout_f32_kernel<CartPoleDyn<IP=0, AK=f32, FR=4>, RECORD=1>"
    record = True
    inst_per_unit = 223.8  # ncu, profiles/r02_launches_rollout_rec.csv (289.9 before the spare reset samples)


class ChargedBallRollout(Workload):
    """C4 as BASELINE words it ("rollouts, 64M envs x 200 steps"): ONE launch advances every env of the shard by
    `horizon` steps with the state in registers (emei_charged_ball_rollout_f32), in-kernel Bernoulli(1/2) policy,
    TimeLimit(500) + auto-reset.  HBM is touched once per env per launch, so the bound is math."""

    key, metric, unit = "c4_rollout", "env_steps_per_sec", "env-steps/s"
    title = "ChargedBallCentering fused rollouts, 2^26 envs total sharded over the ranks x 200 steps per launch, freq_rate=1 (BASELINE configs[3])"
    kernel = "emei::rollout_f32_kernel<ChargedBallDyn<u8>, RECORD=0>"
    scaling, use_graph, bound = "strong", False, "math"
    total = 1 << 26
    alg_fp_ops, alg_sfu_ops = ChargedBall.alg_fp_ops, ChargedBall.alg_sfu_ops
    inst_per_unit = 139.7  # warp-level SASS instructions per env-step, all three divergent paths issued (ncu, profiles/r02_launches_c4_rollout.csv: mean of two consecutive 200-step launches, 128.1 from the reset state and 151.3 after it; 166.0 in round 1)
    cpu_kind, cpu_sample = "c4", 1 << 20
    e2e_max_steps = 5
    stateful = True

    @classmethod
    def _total(cls, args):
        return 1 << args.total_log2 if args.total_log2 else cls.total

    @classmethod
    def _horizon(cls, args):
        return args.horizon if args.horizon_set else 200

    def setup(self):
        import torch

        import emei_b200 as E
        from emei_b200.dist import shard_range

        self.total = self._total(self.args)
        self.T = self._horizon(self.args)
        b, e = shard_range(self.total, self.rank, self.world)
        self.n = e - b
        self.units = self.n * self.T
        self.env = E.make("ChargedBallCentering-v0", num_envs=self.n, dtype=torch.float32, device=self.dev, env_offset=b)
        self.env.reset(seed=1004)
        self.stats = self.env.stats
        self.alg_bytes = 2 * (25 + 12) / self.T  # state 25 + 3 episode counters 12, read + written once per launch

    def step(self, i):
        self.out = self.env.rollout(self.T)

    def setup_e2e(self):
        import torch

        # teacher-forced policy from the host: uint8 [T, n] actions in pinned memory, statistics read back
        self.Te = min(self.T, 25)
        g = torch.Generator()
        g.manual_seed(1004 + self.rank)
        self.act_host = [torch.randint(0, 2, (self.Te, self.n), dtype=torch.uint8, generator=g).pin_memory() for _ in range(2)]
        self.h2d, self.d2h = self.Te * self.n, 48
        self.e2e_units = self.n * self.Te
        self.e2e_api = f"env.rollout({self.Te}, actions=pinned HOST uint8[{self.Te}, n]) -> env.rollout_info(stats) read on the host (the horizon is cut into pieces whose uploads run one piece ahead of the kernels)"

    def step_e2e(self, i):
        out = self.env.rollout(self.Te, actions=self.act_host[i % 2])
        self.info = self.env.rollout_info(out["stats"])

    @classmethod
    def config(cls, args, world):
        tot = cls._total(args)
        return {"envs_total": tot, "envs_per_gpu": tot // world, "horizon": cls._horizon(args), "freq_rate": 1, "max_episode_steps": 500,
                "l2_policy": f"no reuse to defeat: {tot // world * 37 / 1e6:.0f} MB of state read once and written once per launch"}

    @classmethod
    def units_per_step_total(cls, args, world):
        return cls._total(args) * cls._horizon(args)


WORKLOADS = {w.key: w for w in (IPStep, CartPoleStep, CartPoleStepLarge, I2PStep, HopperScoring, HalfCheetahScoring, HopperSeqScoring,
                                HalfCheetahSeqScoring, ChargedBall, ScoringSweep, ScoringSweepSeq, CartPoleRollout, CartPoleRolloutRecord,
                                I2PRollout, ChargedBallRollout)}


def workload_name(W, args):
    return W.title + (", float64 reference-exact mode" if args.dtype == "f64" else ", float32")


def full_config(W, args, world):
    cfg = {"workload": workload_name(W, args)}
    cfg.update(W.config(args, world))
    return cfg


# ==================================================================================================
# reference arm
# ==================================================================================================
def cpu_literal(workload):
    """The reference-literal CPU number (BASELINE.md 5.1): the unmodified reference's scalar env.step loop, timed in
    the BUILD container by scripts/time_reference_literal.py (the GPU box has no reference tree), carried as a constant."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "cpu_literal.json")))
        w = d["workloads"].get({"c1": "c1_cartpole_counterpart", "c3_hopper_seq": "c3_hopper", "c3_halfcheetah_seq": "c3_halfcheetah"}.get(workload, workload))
        if w is None:
            return None
        return {"one_core": w["one_core"], "all_cores": w["all_cores"], "processes": w["processes"],
                "unit": d["unit"] if "freq_rate" in w else d.get("unit_scoring", "transitions/s"),
                "env": w["env"], "freq_rate": w.get("freq_rate"), "kind": "reference-literal, measured in the build container (NOT on this box)",
                "provenance": f"{d['script']} on {d['cpu']} ({d['cores_available']} cores), {d['when']}: {d['what']}"}
    except Exception:
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    W = WORKLOADS[args.workload]
    cores = host_cores()
    kind = W.cpu_kind
    # every step processes the units the GPU arm's step processes (all ranks), unless that exceeds the time box of
    # ~100 s for the whole run: then a bounded sample of it, stated in cpu_baseline.sample
    rate1, _ = cpu_rate(kind, 1 << 14, 1, 1)
    total_steps = args.steps + args.warmup
    want = W.units_per_step_total(args, world)
    cap = int(max(1 << 12, rate1 * cores * 0.6 * 100.0 / total_steps))
    sample = int(min(want, cap, W.cpu_sample * 16))
    sample -= sample % cores
    if args.warmup:
        cpu_rate(kind, sample, args.warmup, cores)
    rate, wall = cpu_rate(kind, sample, args.steps, cores)
    desc = (f"{sample} units/step ({'the whole step' if sample >= want - cores else f'a bounded sample of the {want}-unit step'}) x {args.steps} "
            f"steps of the {cpu_port_desc(kind)}, {cores} processes")
    line = {
        "impl": "reference", "metric": W.metric, "value": rate, "unit": W.unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": W.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": full_config(W, args, world),
        "cpu_baseline": {"value": rate, "unit": W.unit, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": rate, "unit": W.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    lit = cpu_literal(args.workload)
    if lit is not None:
        line["cpu_baseline_literal"] = lit
    emit_json_line(line)


# ==================================================================================================
# GPU arm
# ==================================================================================================
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled for the whole run (B200_PROFILING.md); a workload's record is the
    slice of samples taken while its timed regions ran."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.proc = None
        try:  # started here rather than in run(), so that finish() always finds the process it has to stop
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
        except Exception:
            pass

    def run(self):
        if self.proc is None:
            return
        try:
            for ln in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append((time.monotonic(), [c.strip() for c in ln.split(",")]))
        except Exception:
            pass

    def count(self):
        return len(self.rows)

    def summary(self, t0=None, t1=None):
        sm, mx, reasons = [], 0, set()
        for ts, r in list(self.rows):
            if (t0 is not None and ts < t0) or (t1 is not None and ts > t1):
                continue
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}

    def finish(self):
        """Stop nvidia-smi and reap it: a child left unreaped when bench.py exits stays behind as a zombie.  Safe to call
        more than once (run_ours also registers it with atexit, for runs that end in an error)."""
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=10)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(d.get("sm_max_mhz", 1965.0))
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def measured_math_peaks():
    """FP32 / FP64 FMA and MUFU peaks measured on the box by tools/f2bench (SURVEY 8d asks for them beside hbm_gbs)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "math_peaks.json")))
    except Exception:
        return None


def measured_traffic(workload, f64):
    """dram bytes per launch of the step from the committed ncu captures (profiles/traffic.json, written by
    scripts/make_traffic_json.py); None when there is no capture for this workload."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload + ("_f64" if f64 else ""))
    except Exception:
        return None


class Ctx:
    def __init__(self, rank, world, local, dev, sampler):
        self.rank, self.world, self.local, self.dev, self.sampler = rank, world, local, dev, sampler


def math_model(wl, units, seconds, sm_mhz, peak_gbs):
    """The north star's second bound from ALGORITHMIC operation counts (SURVEY 8d), not from the kernel's own
    instruction count: t_fp32 = FP ops / (148 SMs x 128 lanes x clock), t_sfu = special-function evaluations /
    (148 x 16 x clock) -- for float64: the measured FP64 peak.  Issue utilisation (the kernel's own instructions against
    the issue peak) is reported beside it as a utilisation, not as a roofline."""
    if wl.alg_fp_ops is None:
        return None
    mp = measured_math_peaks() or {}
    clock = sm_mhz * 1e6
    if wl.f64:
        fp_peak = float(mp.get("fp64_tflops", 37.0)) * 1e12 / 2.0  # FMA-class FP64 operations per second
        # float64 has no special-function unit: a divide or square root is ~10 FMA-class operations (Newton iterations),
        # a sin or cos ~20 (reduction + a degree-13 polynomial); the kernel's SASS holds 142 FP64 instructions per
        # sub-step iteration + epilogue, ~440 executed per C2 env-step, against 432 by this count
        fp_ops = wl.alg_fp64_ops if wl.alg_fp64_ops is not None else wl.alg_fp_ops + 15.0 * (wl.alg_sfu_ops or 0)
        t_fp, t_sfu = fp_ops * units / fp_peak, 0.0
        peaks = {"fp64_ops_per_s": fp_peak, "source": "profiles/math_peaks.json fp64_tflops / 2 (tools/f2bench on the B200 box)",
                 "fp64_ops_per_unit": fp_ops, "note": "plain FP ops + 10 per divide / sqrt + 20 per sin / cos (no FP64 special-function unit)"}
    else:
        fp_peak, sfu_peak = 148 * 128 * clock, 148 * 16 * clock
        t_fp, t_sfu = wl.alg_fp_ops * units / fp_peak, (wl.alg_sfu_ops or 0) * units / sfu_peak
        peaks = {"fp32_lane_ops_per_s": fp_peak, "sfu_ops_per_s": sfu_peak, "source": f"148 SMs x 128 FP32 lanes (16 SFU lanes) x {sm_mhz:.0f} MHz",
                 "measured": {k: mp[k] for k in ("fp32_tflops", "mufu_rcp_per_s", "mufu_sin_per_s") if k in mp}}
    t_hbm = wl.bytes_per_unit() * units / (peak_gbs * 1e9)
    t_math = max(t_fp, t_sfu)
    out = {
        "fp_ops_per_unit": wl.alg_fp_ops, "sfu_ops_per_unit": wl.alg_sfu_ops, "t_fp_us": t_fp * 1e6, "t_sfu_us": t_sfu * 1e6,
        "t_math_us": t_math * 1e6, "t_hbm_us": t_hbm * 1e6, "slower_bound": "math" if t_math > t_hbm else "hbm",
        "frac_of_slower_bound": max(t_math, t_hbm) / seconds, "peaks": peaks,
        "source": "operation counts of SURVEY.md 8(d): the reference's arithmetic as written (cartpole.py:48-60, charged_ball.py:68-82), not this kernel's instruction stream",
    }
    if wl.inst_per_unit and not wl.f64:
        issue_peak = 148 * 4 * clock
        out["issue_utilisation"] = {"thread_inst_per_unit": wl.inst_per_unit, "value": wl.inst_per_unit * units / 32.0 / seconds / issue_peak,
                                    "note": "this kernel's own warp instructions (ncu smsp__inst_executed, profiles/) / (148 SMs x 4 schedulers x clock): a utilisation, not a roofline"}
    return out


def measure(wl, ctx, K, W, args, want_e2e=True, keep_outputs=False):
    """One workload: W warm-up steps, exactly K timed steps (barrier + synchronize on both sides, CUDA events on the
    launching stream, max over ranks), the dominant-kernel roofline, the end-to-end leg.  Returns the record.
    keep_outputs: copy the last timed step's outputs to the host as wl.last_outputs."""
    import torch
    import torch.distributed as dist

    from emei_b200 import _lib

    rank, world, dev, sampler = ctx.rank, ctx.world, ctx.dev, ctx.sampler
    wl.setup()
    for i in range(W):
        wl.step(i)
    torch.cuda.synchronize()
    launch_mode = args.launch
    if launch_mode == "auto":
        # measured (profiles/r02_kbench_c2_variants.txt): at K = 20 the graph runs 9.9 us per step, 20 plain stream
        # launches queued behind a spinning kernel 10.5 us
        launch_mode = "graph" if wl.use_graph else "stream"
    if not wl.use_graph:
        launch_mode = "stream"
    launches0 = _lib.launch_count
    restore = getattr(wl, "restore_inputs", None)
    if restore is not None:
        restore()
        torch.cuda.synchronize()
    graph = None
    ev_in = None
    if launch_mode == "graph":  # launch-bound steps: K launches captured once, replayed as one graph
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(dev)
        # the timing events are NODES of the graph (cudaEventRecordExternal), immediately before the first step kernel
        # and after the last: they bracket exactly the K steps on the device.  Events recorded around graph.replay()
        # additionally contain the graph's own launch (a one-off of ~5-10 us, 3-5 % of a 20-step region, nothing at
        # K = 2000); that figure is reported beside it (protocol.ms_per_step_including_graph_launch).
        try:
            ev_in = (torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
        except TypeError:
            ev_in = None
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                if ev_in is not None:
                    ev_in[0].record()
                for i in range(K):
                    wl.step(i)
                if ev_in is not None:
                    ev_in[1].record()
        launches = _lib.launch_count - launches0
    # warm the instantiated graph / the step, and keep the GPU under load until nvidia-smi has delivered samples
    # (it needs a few hundred ms to start; a 0.2 ms region would otherwise end before the first one)
    t_clock0 = time.monotonic()
    n0 = sampler.count() if sampler is not None else 0
    t_warm = time.perf_counter()
    while True:
        if graph is not None:
            graph.replay()
        else:
            for i in range(min(K, 8)):
                wl.step(i)
        torch.cuda.synchronize()
        stop = sampler is None or sampler.count() - n0 >= 3 or time.perf_counter() - t_warm > 1.5
        if world > 1:  # a step may contain a collective (the batch-wide control cost): every rank runs the same number
            flag = torch.tensor([1.0 if (stop or rank != 0) else 0.0], device=dev)
            dist.broadcast(flag, 0)
            stop = flag.item() > 0
        if stop:
            break
    _lib.call("emei_stats_reset", wl.stats.data_ptr(), torch.cuda.current_stream(dev).cuda_stream, launches=0)
    if restore is not None and graph is not None:  # the graph reads the buffers remembered before its capture
        restore()
    if wl.use_graph:
        # a 20-step region touches only the first batches of the ring (C1: 20 of 1024), which the warm-up replays left in
        # L2: write 256 MB (> the 126 MB L2) so that every timed step reads its inputs from HBM
        # The writes alone would leave the L2 holding 126 MB of DIRTY flush lines, whose write-back the first timed steps
        # would pay for (measured: 9.28-9.38 us per step at K = 20 against 9.15 with a clean L2).  In the steady state of
        # this workload about half of the L2 is dirty (22 of every 43 MB a step moves are stores), so 64 MB are read
        # from another buffer after the writes: half the flush lines are written back before the region, half stay dirty.
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        flush.zero_()
        if args.flush_read_mb > 0:
            other = torch.empty(args.flush_read_mb << 20, dtype=torch.uint8, device=dev)
            other.view(torch.int32).sum()
            del other
        del flush
    launches0 = _lib.launch_count
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if wl.use_graph:
        # launch-bound steps: keep the device busy while the host submits the work, so that the events bracket the K
        # steps and not the host's submission latency (graph: ~30 us; K direct step() calls: ~25 us each)
        cyc = args.presleep if args.presleep >= 0 else (200_000 if graph is not None else 400_000 + 80_000 * K)
        if cyc > 0:
            torch.cuda._sleep(int(cyc))
    ev0.record()
    if graph is not None:
        graph.replay()
    else:
        for i in range(K):
            wl.step(i)
    ev1.record()
    if world > 1:
        dist.all_reduce(wl.stats)  # end-of-rollout statistics: 2 doubles over NCCL/NVLink
    torch.cuda.synchronize()
    if graph is None:
        launches = _lib.launch_count - launches0
    if keep_outputs:  # before the e2e leg below steps the same envs again
        wl.last_outputs = {k: v.cpu() for k, v in wl.outputs().items()}
    if world > 1:
        dist.barrier()
    ms_outer = ev0.elapsed_time(ev1)
    ms_region = ms_outer
    if graph is not None and ev_in is not None:
        try:
            ms_inner = ev_in[0].elapsed_time(ev_in[1])
            if 0.0 < ms_inner <= ms_outer:
                ms_region = ms_inner
        except RuntimeError:
            pass
    t = torch.tensor([ms_region, ms_outer], dtype=torch.float64, device=dev)
    units = torch.tensor([float(wl.units)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(units)
    ms_total, ms_outer = float(t[0].item()), float(t[1].item())
    ms_per_step = ms_total / K
    value = float(units.item()) * K / (ms_total * 1e-3)
    graph = None

    # ---------------- e2e: host inputs in, host results out, every step, through the public API
    e2e = None
    if want_e2e:
        wl.setup_e2e()
    if want_e2e and wl.e2e_api is not None:
        e2e_steps = max(3, min(K, args.e2e_steps))
        e2e_steps = min(e2e_steps, getattr(wl, "e2e_max_steps", e2e_steps))
        for i in range(getattr(wl, "e2e_warmup", 2)):  # untimed: first-use work (step_host captures one CUDA graph per
            wl.step_e2e(i)                               # action buffer and ping-pong side the third time it sees the pair)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(e2e_steps):
            wl.step_e2e(i)
        e1.record()
        torch.cuda.synchronize()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        te = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_units = float(units.item()) * getattr(wl, "e2e_units", wl.units) / wl.units
        e2e = {
            "value": e2e_units * e2e_steps / (float(te.item()) * 1e-3), "unit": wl.unit,
            "h2d_bytes_per_step": wl.h2d, "d2h_bytes_per_step": wl.d2h, "steps": e2e_steps, "api": wl.e2e_api,
        }
    e2e_light = None
    if e2e is not None and hasattr(wl, "step_e2e_light"):
        for i in range(getattr(wl, "e2e_warmup", 2)):
            wl.step_e2e_light(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(e2e["steps"]):
            wl.step_e2e_light(i)
        e1.record()
        torch.cuda.synchronize()
        te = torch.tensor([max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        st = wl.env0._staging
        e2e_light = {"value": float(units.item()) * e2e["steps"] / (float(te.item()) * 1e-3), "unit": wl.unit, "h2d_bytes_per_step": st.h2d_bytes,
                     "d2h_bytes_per_step": st.d2h_bytes, "steps": e2e["steps"], "api": wl.e2e_light_api}
    t_clock1 = time.monotonic()
    if rank != 0:
        return None

    peak, peak_src, sm_mhz = measured_peaks()
    step_s = ms_per_step * 1e-3
    bpu = wl.bytes_per_unit()
    achieved = bpu * wl.units / step_s / 1e9
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
        "peak_source": peak_src, "frac_of_datasheet_8tbs": achieved / 8000.0,  # SURVEY 8(d): also against the 8 TB/s datasheet figure
        "algorithmic_bytes_per_unit": bpu, "kernel": wl.kernel_name(),
        "kernel_ms_per_launch": ms_per_step,
        "note": "duration = CUDA-event time of ONE WHOLE STEP (timed region / steps: every kernel of the step and the gaps between launches included)",
    }
    mm = math_model(wl, wl.units, step_s, sm_mhz, peak)
    # the north star's roofline is the SLOWER of the two bounds: workloads with no per-unit HBM traffic to speak of (rollouts), and
    # float64 steps whose algorithmic FP64 work outlasts their bytes (C2 in reference-exact mode: 25 us of FP64 against 12 us of HBM)
    if mm is not None and (wl.bound == "math" or mm["slower_bound"] == "math"):
        if wl.f64:
            binding, ops, pk = "fp64", mm["peaks"]["fp64_ops_per_unit"], mm["peaks"]["fp64_ops_per_s"]
        else:
            binding = "sfu" if mm["t_sfu_us"] >= mm["t_fp_us"] else "fp32"
            ops = wl.alg_sfu_ops if binding == "sfu" else wl.alg_fp_ops
            pk = mm["peaks"]["sfu_ops_per_s" if binding == "sfu" else "fp32_lane_ops_per_s"]
        roofline = {
            "bound": "math", "achieved": ops * wl.units / step_s / 1e12, "peak": pk / 1e12, "unit": f"T {binding} op/s (algorithmic)",
            "frac": mm["frac_of_slower_bound"], "traffic": None, "kernel": wl.kernel_name(), "kernel_ms_per_launch": ms_per_step,
            "frac_of_math_bound": mm["t_math_us"] * 1e-6 / step_s,
            "binding_unit": binding, "math": mm,
            "hbm": {"algorithmic_bytes_per_unit": bpu, "achieved_gbs": achieved, "frac_of_hbm_peak": achieved / peak},
            "note": "duration = CUDA-event time per launch; operations = SURVEY 8(d)'s algorithmic counts per env-step x env-steps",
        }
    elif mm is not None:
        roofline["math"] = mm
    tr = measured_traffic(wl.key, wl.f64)
    if tr is not None:
        roofline["traffic"] = tr["bytes_per_launch"]
        roofline["traffic_source"] = tr.get("note") or f"{tr['source']}: dram__bytes_read.sum + dram__bytes_write.sum per step (ncu)"
        roofline["algorithmic_bytes_per_launch"] = bpu * wl.units
    cfg = full_config(type(wl), args, world)
    protocol = {
        "launch": (f"K={K} steps captured in one CUDA graph (programmatic dependent launches), replayed once; the two timing events are nodes "
                   "of that graph, directly before the first step kernel and after the last" if launch_mode == "graph"
                   else f"K={K} step() calls launched back to back on one stream" + (" behind a spinning kernel (the device never waits for the host)" if wl.use_graph else ""))
                  + "; CUDA events on the launching stream",
        "parallelism": f"batch sharded over {world} rank(s), no data-path collective; NCCL all-reduce of the 2-double statistics at the end",
    }
    if world > 1:
        hb = getattr(args, "host_binding", None)
        protocol["host_binding"] = (f"rank 0 bound to {len(hb)} CPUs local to its GPU's NUMA node" if hb else
                                    "none: the host exposes one NUMA node / no per-GPU CPU locality")
    if restore is not None and launch_mode == "graph":
        protocol["inputs"] = ("the synthetic states of SURVEY 8(d) are copied back into every env's input buffer after the warm-up replays, outside "
                              "the timed region (the step kernels never reset: warm-up alone would spin the poles beyond the integrator's guard); "
                              "then 256 MB are written to flush the 126 MB L2 and 64 MB read from another buffer (the L2 starts half dirty, as in the steady state of "
                              "a step that stores 22 of every 43 MB it moves), so every timed step reads from HBM")
    if launch_mode == "graph":
        protocol["ms_per_step_including_graph_launch"] = ms_outer / K
        protocol["note"] = ("events recorded around graph.replay() also contain the graph's launch, a one-off per replay: "
                            f"{(ms_outer - ms_total) * 1e3:.1f} us here")
    rec = {
        "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None,
        "dtype": "f64" if wl.f64 else "f32", "data": "synthetic", "config": cfg, "protocol": protocol, "roofline": roofline,
        "e2e": e2e, "gpu_launches": launches,
        "clocks": sampler.summary(t_clock0, t_clock1) if sampler is not None else None,
    }
    if e2e_light is not None:
        rec["e2e_reward_done"] = e2e_light
    return rec


DUMP_BYTES = 64 << 20


def dump_outputs(outs, directory):
    """--dump-outputs: every output as <directory>/<name>.npy, float64 where the path computed float64, else float32 (flags
    as 0 / 1).  Above DUMP_BYTES in all, the arrays are cut to one fixed, seeded sample of rows (the same rows of every array
    with the same row count), so that runs with the same arguments can be compared output for output."""
    arrays = {k: v.numpy() for k, v in outs.items()}
    arrays = {k: a.astype(np.float64 if a.dtype == np.float64 else np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        rows = {}
        for k, a in arrays.items():
            n = a.shape[0]
            if n not in rows:
                rows[n] = np.sort(np.random.default_rng(0).choice(n, n * DUMP_BYTES // total, replace=False))
            arrays[k] = a[rows[n]]
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)


SECONDARY_N1 = [("c1", "f32"), ("c2_f64", "f64"), ("c3_hopper", "f32"), ("c3_halfcheetah", "f32"), ("c3_hopper_seq", "f32"),
                ("c3_halfcheetah_seq", "f32"), ("c4", "f32"), ("c4_rollout", "f32"), ("c5", "f32"), ("c5_seq", "f32")]
SECONDARY_MULTI = [("c4", "f32"), ("c4_rollout", "f32"), ("c5", "f32"), ("c5_seq", "f32")]


def run_ours(args):
    import copy
    import gc

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; emei_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's banner must not share stdout with the JSON line
        import datetime

        # a collective that cannot complete (a rank died) fails after two minutes instead of NCCL's ten
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    # several ranks on one host: pin each to the CPUs next to its GPU before any pinned staging buffer is allocated
    # (first touch places the pages on that NUMA node); a no-op where the host exposes a single node
    from emei_b200.dist import bind_to_gpu_numa

    args.host_binding = bind_to_gpu_numa(local) if world > 1 else None
    t_start = time.monotonic()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler is not None:
        sampler.start()
        atexit.register(sampler.finish)
        time.sleep(0.3)
    ctx = Ctx(rank, world, local, dev, sampler)
    K, W = args.steps, max(args.warmup, 3)
    wl = WORKLOADS[args.workload](args, rank, world, dev)
    line = measure(wl, ctx, K, W, args, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(wl.last_outputs, args.dump_outputs)
    # ---------------- CPU baseline on this box's host cores (bounded sample; oracle = the thing timed beside us)
    if rank == 0 and world == 1 and not args.no_cpu:
        n_s = wl.cpu_sample
        _, wall0 = cpu_rate(wl.cpu_kind, n_s, 1, 1)  # calibrate with one pass, then size the pass count for ~10 s of one core
        reps = int(max(2, min(200, round(10.0 / max(wall0, 1e-3)))))
        rate1, wall1 = cpu_rate(wl.cpu_kind, n_s, reps, 1)
        line["cpu_baseline"] = {
            "value": rate1, "unit": wl.unit, "cores": 1, "kind": "port",
            "sample": f"{n_s} units x {reps} passes of the {cpu_port_desc(wl.cpu_kind)}, {wall1:.1f} s",
        }
    if rank == 0:
        lit = cpu_literal(args.workload)
        if lit is not None:
            line["cpu_baseline_literal"] = lit
    wl.teardown()
    del wl
    # ---------------- the other BASELINE configs, same process, compact records, time-boxed
    if args.secondary:
        sec = {}
        plan = SECONDARY_N1 if world == 1 else SECONDARY_MULTI
        for name, dtype in plan:
            gc.collect()
            torch.cuda.empty_cache()
            elapsed = time.monotonic() - t_start
            flag = torch.tensor([1.0 if elapsed > args.secondary_budget else 0.0], device=dev)
            if world > 1:
                dist.broadcast(flag, 0)  # every rank takes the same decision
            if flag.item() > 0:
                if rank == 0:
                    sec[name] = {"skipped": f"time box: {elapsed:.0f} s elapsed > {args.secondary_budget:.0f} s"}
                continue
            a2 = copy.copy(args)
            a2.dtype, a2.ring, a2.total_log2, a2.horizon_set = dtype, 0, 0, False
            key = name[:-4] if name.endswith("_f64") else name
            Wc = WORKLOADS[key]
            k2 = max(3, min(K, 20 if Wc.use_graph else (3 if key == "c4_rollout" else 10)))
            w2 = Wc(a2, rank, world, dev)
            try:
                rec = measure(w2, ctx, k2, 3, a2)
            except Exception as e:  # a secondary must never cost the primary line
                rec = {"error": f"{type(e).__name__}: {e}"[:300]}
                if world > 1:
                    raise
            w2.teardown()
            del w2
            if rank == 0 and rec is not None and "error" not in rec:
                lit = cpu_literal(key)
                if lit is not None:
                    rec["cpu_baseline_literal"] = lit
            if rank == 0 and rec is not None:
                sec[name] = {k: rec[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "config", "roofline",
                                                 "e2e", "e2e_reward_done", "gpu_launches", "clocks", "cpu_baseline_literal") if k in rec} if "error" not in rec else rec
        if rank == 0:
            line["secondary"] = sec
    if rank == 0:
        sampler.finish()
        emit_json_line(line)
    if world > 1:
        dist.destroy_process_group()


# The contract is ONE JSON line on stdout.  Libraries write to the process's stdout on their own (NCCL prints its
# version banner there with printf when NCCL_DEBUG is set in the environment), so file descriptor 1 is pointed at
# stderr for the whole run and the JSON line alone goes to the real stdout.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json_line(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.buffer.write(data)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    capture_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"], help="f64 = the float64 reference-exact mode (c1, c2, i2p, c3_*, c4)")
    ap.add_argument("--launch", default="auto", choices=["auto", "graph", "stream"],
                    help="launch-bound workloads (c1, c2, i2p): K steps as one CUDA graph (auto), or K step() calls queued behind a spinning kernel")
    ap.add_argument("--presleep", type=int, default=-1, help="development knob: cycles of the spinning kernel queued before the timed region of launch-bound workloads (-1 = default)")
    ap.add_argument("--no-secondary", action="store_true", help="default workload only: skip the `secondary` records of the other BASELINE configs")
    ap.add_argument("--flush-read-mb", type=int, default=64, help="graph workloads: MB read from a second buffer after the 256 MB L2 flush writes (0: leave the L2 full of dirty flush lines)")
    ap.add_argument("--secondary-budget", type=float, default=240.0, help="seconds after which remaining secondary workloads are skipped")
    ap.add_argument("--ring", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--total-log2", type=int, default=0, help="c4 only: log2 of the total env count (default 26)")
    ap.add_argument("--horizon", type=int, default=None, help="rollout workloads: env-steps per launch (default 100; 32 with records)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them returned (rank 0's shard) as DIR/<name>.npy, "
                         "at most 64 MB in all (a fixed, seeded sample of rows beyond that)")
    args = ap.parse_args()
    args.horizon_set = args.horizon is not None
    if args.horizon is None:
        args.horizon = 100
    args.secondary = args.workload is None and not args.no_secondary and args.impl == "ours" and args.dtype == "f32"
    if args.workload is None:
        args.workload = "c2"
    if args.dump_outputs:
        if args.impl != "ours":
            raise SystemExit("bench.py: --dump-outputs writes what the GPU path computed (--impl ours)")
        if not WORKLOADS[args.workload].reproducible(args):
            raise SystemExit(f"bench.py: --dump-outputs: the timed steps of {args.workload} (launched this way) start from a state the "
                             "untimed warm-up advanced by a run-dependent number of steps, so their outputs would differ from run to run")
    if args.steps is None:
        args.steps = 2000 if WORKLOADS[args.workload].use_graph else 20
        if args.impl == "reference":
            args.steps = 20
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
