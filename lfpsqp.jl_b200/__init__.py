"""lfpsqp.jl_b200 -- B200-native hot path of LFPSQP.jl behind the reference's `optimize` API.

Host-side mirror of src/optimize.jl's public method family (:13, :83, :88, :107, :112) over the C ABI of
include/lfpsqp_b200.h.  All numerics run in hand-written sm_100a CUDA kernels; there is no CPU fallback.
"""
from . import families
from ._lib import Context, MultiContext, LFPSQPError, default_context, load
from .large import LargeProblem, ineq_op, make_diagquad, linesearch, aug_hess_vec, optimize_large
from .host import optimize_explicit, optimize_slack
from .api import (LFPSQPParams, TerminationCondition, TerminationInfo, optimize, optimize_batched, armijo, exact,
                  off, iter_)

__all__ = ["optimize", "optimize_large", "optimize_explicit", "optimize_slack", "optimize_batched", "LFPSQPParams", "TerminationInfo", "TerminationCondition", "families",
           "LargeProblem", "ineq_op", "linesearch", "aug_hess_vec", "make_diagquad", "Context", "MultiContext", "LFPSQPError", "default_context", "load", "armijo", "exact", "off", "iter_"]
