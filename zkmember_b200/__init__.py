"""zkmember_b200 -- B200-native MSM / NTT backend for zkMember's Groth16 and Marlin provers.

Only the hot path lives here: `csrc/` (hand-written CUDA for sm_100a + the C ABI of
include/zkm_b200.h) and the host-side mirrors of the two arkworks interfaces it replaces:

    from zkmember_b200 import VariableBaseMSM, FixedBaseMSM, Radix2EvaluationDomain
"""
import os as _os

# Hardware work queues: a proof keeps six streams busy (the witness map + five MSM lanes) and several proofs are in flight;
# with the default of 8 queues streams share a queue and wait behind one another's kernels (measured on B200, Groth16
# proxy: 389 -> 454 proofs/s with 32).  Read by the CUDA runtime when it initialises, so it is set at import time (the C
# library does the same in zkm_init* for callers that are not Python); an explicit setting of the user wins.
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from ._lib import ZkmError, DomainError, init, shutdown, set_option, launch_count, load  # noqa: F401
from .msm import VariableBaseMSM, FixedBaseMSM, RegisteredBases, AffinePoint, msm_window_bits  # noqa: F401
from .domain import Radix2EvaluationDomain, GeneralEvaluationDomain  # noqa: F401

__all__ = [
    "VariableBaseMSM", "FixedBaseMSM", "RegisteredBases", "AffinePoint", "Radix2EvaluationDomain", "GeneralEvaluationDomain",
    "ZkmError", "DomainError", "init", "shutdown", "set_option", "launch_count", "load", "msm_window_bits",
]
