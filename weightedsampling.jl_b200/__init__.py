"""wsb200 — B200-native particle hot path behind WeightedSampling.jl's API.

The package keeps the reference's public names for the path (``src/WeightedSampling.jl:11-26``):
``SMCState, WeightedKernel, run (run!), exp_norm, RW, autoRW, default_proposals, default_kernels,
importance_kernel, expectation, E (@E), sample, log_evidence, model (@model)`` plus the transformer
types.  All particle work runs in ``lib/libwsb200.so`` (hand-written sm_100a CUDA behind the C ABI of
``include/wsb200.h``); there is no CPU fallback.
"""
from ._lib import LIB_PATH, UnsupportedModelError, WsError, load  # noqa: F401
from .expr import (abs2, atan, col, cos, exp, expm1, floor, lgamma, log, log1p, maximum, minimum, randexp, randn,  # noqa: F401
                   randu, sin, sqrt, table, tan, tanh, where)
from .core import *  # noqa: F401,F403
from .core import NormalDist  # noqa: F401
from .analysis import (E, describe, ess_perc, exp_norm, expectation, icdf, log_evidence, logsumexp,  # noqa: F401
                       resample_indices, sample, to_dataframe)
from .model import model  # noqa: F401
