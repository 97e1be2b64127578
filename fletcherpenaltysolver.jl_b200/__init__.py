"""fps-b200: B200-native two-right-hand-side quasi-definite solves behind
FletcherPenaltySolver.jl's plugin surface (QDSolver / solve_two_*).

`import fpsb200` (repo-root alias) loads this package.  All arithmetic runs in
libfpsb200.so (hand-written CUDA for sm_100a, C ABI in include/fpsb.h).
"""
from . import _lib
from ._lib import FPSB_DEVICE, FPSB_HOST, ExtrasOpts, FpsbError, IterOpts, KrylovStats, LdltOpts
from .qdsolver import (B200Handle, IterativeSolver, LDLtSolver, QDSolver, batch_solve_two, qdsolver_correspondence,
                       solve_two_extras, solve_two_extras_batch, solve_two_least_squares, solve_two_least_squares_batch,
                       solve_two_mixed, solve_two_mixed_batch)
from .fletcher_nlp import FletcherPenaltyNLP
from .device_nlp import BatchFletcherPenaltyNLP, DeviceCurvedQP, DeviceFletcherPenaltyNLP, DeviceSparseQP
from .fps_solve import AlgoData, FPSSSolver, GenericExecutionStats, GNSolver, fps_solve, solve, trunk
from . import models

__all__ = ["B200Handle", "IterativeSolver", "LDLtSolver", "QDSolver", "qdsolver_correspondence",
           "solve_two_extras", "solve_two_extras_batch", "solve_two_least_squares", "solve_two_mixed", "solve_two_least_squares_batch",
           "solve_two_mixed_batch", "FletcherPenaltyNLP",
           "DeviceFletcherPenaltyNLP", "BatchFletcherPenaltyNLP", "DeviceSparseQP", "DeviceCurvedQP", "fps_solve", "FPSSSolver", "AlgoData", "GNSolver",
           "GenericExecutionStats", "solve", "trunk",
           "models", "batch_solve_two", "FPSB_HOST", "FPSB_DEVICE", "FpsbError", "IterOpts", "KrylovStats", "LdltOpts",
           "ExtrasOpts"]
