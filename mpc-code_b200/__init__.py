"""Batched MPC step solver for B200 (sm_100a) behind the CPCLAB-UNIPI/MPC-code user API.

Host side (this package): symbolic tracer for the user's ``Ex_*.py`` files, code generator,
mirrors of the reference builders (``opt_dyn``, ``opt_ss``, ``defEstimator``) and the batched
closed loop.  Device side: ``csrc/`` CUDA kernels behind the C-ABI declared in ``include/mpcb.h``.
"""
__version__ = "0.1.0"

from .loader import load_example  # noqa: F401
from .problem import build_problem, make_specs  # noqa: F401
from .sensitivity import OcpLayer, OcpSensitivity, params_of, theta_of, with_params, with_theta  # noqa: F401
from .sensitivity import TargetLayer, TargetSensitivity, theta_ss_of, with_theta_ss  # noqa: F401


def compile_problem(*args, **kwargs):
    from .mpc_loop import compile_problem as _cp
    return _cp(*args, **kwargs)
