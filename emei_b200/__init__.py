"""emei_b200 -- B200-native batched environment engine behind polixir/emei's EmeiEnv API.

One data-parallel hot path (BASELINE.json north_star): the analytic classic-control step
(cart-pole / inverted-pendulum swing-up, charged-ball centering, freq_rate forward-Euler sub-steps)
and the model-based scoring interface (get_batch_reward / get_batch_terminal / batched init-obs /
freeze / unfreeze).  Python holds torch CUDA tensors and calls hand-written sm_100a kernels through
the C ABI in ``include/emei_b200.h``.  There is no CPU fallback.
"""
__version__ = "0.1.0"

from . import _lib  # noqa: F401  (loads libemei_b200.so; raises if it is missing)
from .core import EmeiEnv, Freezable, PlanResult, PolicySearchResult, plan_iteration_seed, policy_starts_seed  # noqa: F401
from .envs import register_env  # noqa: F401
from .envs.register_env import make, registry, spec  # noqa: F401
