"""ctypes binding of ``libemei_b200.so`` (the C ABI declared in ``include/emei_b200.h``).

There is NO fallback: if the shared library is missing or fails to load, importing this module
raises, and every op raises ``EmeiB200Error`` on a non-zero return code.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libemei_b200.so")

# ---- constants mirrored from include/emei_b200.h ---------------------------------------------
ACTION_DISCRETE_U8, ACTION_DISCRETE_I32, ACTION_DISCRETE_I64, ACTION_CONTINUOUS_F32, ACTION_CONTINUOUS_F64 = range(5)
(
    CARTPOLE_BALANCING,
    CARTPOLE_SWINGUP,
    IP_REBOUND_BALANCING,
    IP_BOUNDARY_BALANCING,
    IP_REBOUND_SWINGUP,
    IP_BOUNDARY_SWINGUP,
    I2P_REBOUND_BALANCING,
    I2P_BOUNDARY_BALANCING,
    I2P_REBOUND_SWINGUP,
    I2P_BOUNDARY_SWINGUP,
    HOPPER,
    HALFCHEETAH,
    CHARGED_BALL,
) = range(13)


SUMSQ_WORKSPACE_BYTES = (148 * 8 + 1) * 8  # EMEI_SUMSQ_WORKSPACE_BYTES


class EmeiB200Error(RuntimeError):
    pass


class CartPoleParams(Structure):
    _fields_ = [
        ("gravity", c_double),
        ("mass_pole", c_double),
        ("total_mass", c_double),
        ("length", c_double),
        ("pole_mass_length", c_double),
        ("force_mag", c_double),
        ("x_threshold", c_double),
        ("theta_threshold", c_double),
        ("x_left", c_double),
        ("x_right", c_double),
        ("ctrl_low", c_double),
        ("ctrl_high", c_double),
        ("dt", c_double),
        ("freq_rate", c_int32),
        ("variant", c_int32),
        ("action_kind", c_int32),
        ("reserved", c_int32),
    ]


class ChargedBallParams(Structure):
    _fields_ = [
        ("gravity_acc", c_double),
        ("mass_ball", c_double),
        ("radius", c_double),
        ("charge", c_double),
        ("time_step", c_double),
        ("freq_rate", c_int32),
        ("action_kind", c_int32),
    ]


class ScoringParams(Structure):
    _fields_ = [
        ("family", c_int32),
        ("terminate_when_unhealthy", c_int32),
        ("forward_reward_weight", c_double),
        ("ctrl_cost_weight", c_double),
        ("healthy_reward", c_double),
        ("healthy_state_lo", c_double),
        ("healthy_state_hi", c_double),
        ("healthy_z_lo", c_double),
        ("healthy_z_hi", c_double),
        ("dt", c_double),
        ("x_threshold", c_double),
        ("theta_threshold", c_double),
        ("x_left", c_double),
        ("x_right", c_double),
        ("radius", c_double),
    ]


class I2PParams(Structure):
    _fields_ = [
        ("gravity", c_double), ("mass_cart", c_double), ("mass_pole0", c_double), ("mass_pole1", c_double),
        ("length0", c_double), ("length1", c_double), ("gear", c_double), ("ctrl_low", c_double), ("ctrl_high", c_double),
        ("x_left", c_double), ("x_right", c_double), ("dt", c_double),
        ("freq_rate", c_int32), ("variant", c_int32), ("action_kind", c_int32),
    ]


class NoiseParams(Structure):
    _fields_ = [("sigma", c_double * 6), ("seed", c_uint64), ("env_offset", c_uint64), ("step", c_uint64)]


class RolloutParams(Structure):
    _fields_ = [
        ("horizon", c_int32),
        ("max_episode_steps", c_int32),
        ("auto_reset", c_int32),
        ("random_policy", c_int32),
        ("init_kind", c_int32),
        ("init_pi_column", c_int32),
        ("seed_reset", c_uint64),
        ("seed_action", c_uint64),
        ("env_offset", c_uint64),
        ("t0", c_uint64),
        ("init_low", c_double),
        ("init_high", c_double),
        ("init_mean", c_double * 4),
        ("init_sigma", c_double * 4),
        ("action_low", c_double),
        ("action_high", c_double),
    ]


_P = c_void_p
_PROTOTYPES = {
    # name: (restype, argtypes)
    "emei_cartpole_step": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(CartPoleParams), _P]),
    "emei_charged_ball_step": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(ChargedBallParams), _P]),
    "emei_i2p_step": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(I2PParams), _P]),
    "emei_cartpole_step_jacobian": (c_int, [_P, _P, _P, _P, c_int64, POINTER(CartPoleParams), _P]),
    "emei_cartpole_step_vjp": (c_int, [_P] * 7 + [c_int64, POINTER(CartPoleParams), _P]),
    "emei_i2p_step_jacobian": (c_int, [_P, _P, _P, _P, c_int64, POINTER(I2PParams), _P]),
    "emei_i2p_step_vjp": (c_int, [_P] * 7 + [c_int64, POINTER(I2PParams), _P]),
    "emei_cartpole_trajectory": (c_int, [_P] * 6 + [c_int64, c_int64, POINTER(CartPoleParams), _P]),
    "emei_cartpole_trajectory_vjp": (c_int, [_P] * 7 + [c_int64, c_int64, POINTER(CartPoleParams), _P]),
    "emei_i2p_trajectory": (c_int, [_P] * 6 + [c_int64, c_int64, POINTER(I2PParams), _P]),
    "emei_i2p_trajectory_vjp": (c_int, [_P] * 7 + [c_int64, c_int64, POINTER(I2PParams), _P]),
    "emei_ip_step_noisy": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(CartPoleParams), POINTER(NoiseParams), _P]),
    "emei_i2p_step_noisy": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(I2PParams), POINTER(NoiseParams), _P]),
    "emei_cartpole_rollout_ref": (c_int, [_P] * 12 + [c_int64, POINTER(CartPoleParams), POINTER(RolloutParams), POINTER(NoiseParams), _P]),
    "emei_i2p_rollout": (c_int, [_P] * 12 + [c_int64, POINTER(I2PParams), POINTER(RolloutParams), POINTER(c_double), POINTER(c_double),
                                  POINTER(NoiseParams), _P]),
    "emei_charged_ball_rollout_ref": (c_int, [_P] * 14 + [c_int64, POINTER(ChargedBallParams), POINTER(RolloutParams), _P]),
    "emei_reward_terminal": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, POINTER(ScoringParams), _P]),
    "emei_reward_terminal_seq": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int64, POINTER(ScoringParams), _P]),
    "emei_sumsq": (c_int, [_P, c_int64, _P, _P, _P]),
    "emei_sum": (c_int, [_P, c_int64, _P, _P, _P]),
    "emei_reward_vjp": (c_int, [_P] * 7 + [c_int64, POINTER(ScoringParams), _P]),
    "emei_reward_seq_vjp": (c_int, [_P] * 6 + [c_int64, c_int64, POINTER(ScoringParams), _P]),
    "emei_init_uniform": (c_int, [_P, c_int64, c_int32, c_double, c_double, c_int32, c_uint64, c_uint64, _P]),
    "emei_init_gaussian": (c_int, [_P, c_int64, c_int32, POINTER(c_double), POINTER(c_double), c_uint64, c_uint64, _P]),
    "emei_init_charged_ball": (c_int, [_P, _P, _P, c_int64, c_double, c_uint64, c_uint64, _P]),
}
_PLAIN = {
    "emei_cartpole_rollout_f32": (c_int, [_P] * 12 + [c_int64, POINTER(CartPoleParams), POINTER(RolloutParams), _P]),
    "emei_charged_ball_rollout_f32": (c_int, [_P] * 14 + [c_int64, POINTER(ChargedBallParams), POINTER(RolloutParams), _P]),
    "emei_snapshot_copy": (c_int, [_P, _P, c_int64, _P]),
    "emei_records_transpose": (c_int, [_P, _P, c_int64, c_int64, c_int32, _P]),
    "emei_stats_reset": (c_int, [_P, _P]),
    "emei_version": (c_int, []),
    "emei_error_string": (c_char_p, [c_int]),
    "emei_family_obs_dim": (c_int, [c_int]),
    "emei_family_action_dim": (c_int, [c_int]),
}


def exported_symbols():
    """Every symbol include/emei_b200.h declares."""
    names = []
    for base in _PROTOTYPES:
        names += [base + "_f32", base + "_f64"]
    return names + list(_PLAIN)


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"emei_b200: native library not found at {LIB_PATH}. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C emei_b200/csrc`). "
            "There is no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for base, (res, args) in _PROTOTYPES.items():
        for suffix in ("_f32", "_f64"):
            fn = getattr(lib, base + suffix)
            fn.restype, fn.argtypes = res, args
    for name, (res, args) in _PLAIN.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


lib = _load()

# number of kernel launches issued through this binding (bench.py reports it as gpu_launches)
launch_count = 0


def check(code: int, what: str):
    if code != 0:
        msg = lib.emei_error_string(code).decode()
        raise EmeiB200Error(f"{what} failed: [{code}] {msg}")


def call(name: str, *args, launches: int = 1):
    """Invoke a C-ABI function, raise on error, count launches."""
    global launch_count
    code = getattr(lib, name)(*args)
    check(code, name)
    launch_count += launches
