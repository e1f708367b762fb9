"""B200-native batched solver for the Apollo 11 LM ascent NLP of Launch_Optimiser.py.

Public API: :func:`optimise`, :func:`optimise_batch`, :class:`AscentParams`, :class:`Mesh`,
:class:`SolverOptions`, and :func:`fly`, which flies a solved control through the continuous dynamics.  All
numerical work runs in hand-written sm_100a CUDA kernels behind the C ABI in ``include/lmato_b200.h``; there is no CPU fallback.
"""
from .api import (AscentBatchSolution, AscentMultiSolver, AscentParams, AscentSolution, AscentSolver, FlownAscent, Mesh,
                  SolverOptions, default_fly_substeps, final_state_si, fly, multi_device_solve, optimise, optimise_batch, shard_bounds, sharded_solve)
from .dispersions import dispersed_params, nominal_params
from ._cabi import LmatoError, build_library

__all__ = ["AscentBatchSolution", "AscentMultiSolver", "AscentParams", "AscentSolution", "AscentSolver", "FlownAscent",
           "Mesh", "SolverOptions", "default_fly_substeps", "final_state_si", "fly", "multi_device_solve", "optimise", "optimise_batch", "shard_bounds", "sharded_solve",
           "dispersed_params", "nominal_params", "LmatoError", "build_library"]
