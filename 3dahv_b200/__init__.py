"""3dahv_b200 — B200-native hypothesis-and-verification path of 3DAHV.

The directory name starts with a digit, so import it with
`importlib.import_module("3dahv_b200")` or through the alias module `ahv_b200`
at the repository root.
"""
from ._lib import LIB_PATH, MATH_FP32, MATH_TC, MATH_TC_F16GATHER, VOL_BF16, VOL_F32  # noqa: F401
from . import ops, so3, dist, refcompat, training, evaluate  # noqa: F401
from .verify import GraphedRefiner, GraphedTail, GraphedVerifier, HypothesisVerifier, Posterior, VerifyResult  # noqa: F401

__version__ = "0.2.0"
