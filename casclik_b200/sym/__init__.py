"""`cs`-compatible expression namespace: `from casclik_b200 import cs` stands in for
`import casadi as cs` in CASCLIK user code (the subset listed in SURVEY.md §8b)."""
import numpy as np  # noqa: F401  (reference code reaches NumPy through `cs.np`)

from . import dag  # noqa: F401
from .matrix import (  # noqa: F401
    GenericMatrixCommon, MX, SX, DM, Sparsity, Function,
    inf, pi,
    vertcat, horzcat, mtimes, transpose, dot, sumsqr, norm_1, norm_2, norm_fro, norm_inf,
    sum1, sum2, trace, diag, reshape, vec, cross,
    sin, cos, tan, asin, acos, atan, atan2, exp, log, sqrt, fabs, sign, floor, ceil,
    fmin, fmax, power, logic_and, logic_or, logic_not, if_else,
    jacobian, jtimes, gradient, hessian, substitute, depends_on, symvar,
    solve, inv, det, pinv,
)


def conic(name, solver_name, structure, opts=None):
    """`cs.conic(name, "qpoases", {"h": sp, "a": sp}, opts)` (reference reactive_qp.py:256-260).
    Returns a callable `solver(h=, a=, lba=, uba=[, x0=])` backed by the batched CUDA QP kernel."""
    from ..controllers.qp_solver import ConicSolver
    return ConicSolver(name, solver_name, structure, opts or {})
