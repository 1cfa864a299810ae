"""lp_b200 -- B200-native (sm_100a) interior-point hot path of the `ripped` LP solver.

Public surface mirrors the reference's prelude (/root/reference/src/prelude.rs:3-11):
``Problem``, ``InteriorPoint``, ``EquationSolverType``, ``Solver``, ``LinearProgramError``.
Importing this package never touches CUDA; the first compute call loads liblpb200.so
(``lp_b200/_lib``) and fails loudly if it was not built or no B200 is visible.
"""
from .api import (  # noqa: F401
    BatchedResult,
    ResidentProblem,
    ShardedProblem,
    SyntheticShardedProblem,
    solve_batched,
    solve_many,
    pinned_empty,
    presolve,
    Presolved,
    release_cached_contexts,
    EquationSolverType,
    IncompatibleInputDimensions,
    Infeasible,
    InteriorPoint,
    InteriorPointBuilder,
    InvalidParameter,
    IterationLimitExceeded,
    LinearProgramError,
    NumericalProblem,
    OptimizeResult,
    Problem,
    ProblemBuilder,
    Solver,
    Unbounded,
    Unconstrained,
)

__all__ = [
    "BatchedResult", "ResidentProblem", "ShardedProblem", "SyntheticShardedProblem", "solve_batched", "solve_many", "pinned_empty", "presolve", "Presolved", "release_cached_contexts",
    "EquationSolverType", "IncompatibleInputDimensions", "Infeasible", "InteriorPoint", "InteriorPointBuilder",
    "InvalidParameter", "IterationLimitExceeded", "LinearProgramError", "NumericalProblem", "OptimizeResult",
    "Problem", "ProblemBuilder", "Solver", "Unbounded", "Unconstrained",
]
