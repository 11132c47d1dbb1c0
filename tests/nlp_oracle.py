"""Host-side references for the NLP controller tests: a first-order KKT certificate and an SLSQP solve of
one instance, independent of the kernel code (F, its gradient and the constraint rows are evaluated by
the expression interpreter from the lowered program, the optimiser is SciPy's)."""
import numpy as np
from scipy.optimize import minimize

from casclik_b200.sym import dag


def nlp_kkt_residuals(grad, A, lb, ub, x):
    """First-order certificate of x for  min F  s.t. lb <= A x <= ub  given grad = dF/dx at x.  Multipliers
    are recovered by least squares on the rows active at x (grad + A' lam = 0; lam >= 0 on rows at their
    upper bound, <= 0 at their lower bound, any sign on equality rows).
    -> dict(primal, stationarity, sign, lam)"""
    r = A @ x
    primal = max(0.0, float(np.max(lb - r, initial=0.0)), float(np.max(r - ub, initial=0.0)))
    tol = 1e-7 * (1.0 + np.abs(r))
    at_u = np.abs(r - ub) <= tol
    at_l = np.abs(r - lb) <= tol
    act = np.nonzero(at_u | at_l)[0]
    lam = np.zeros(A.shape[0])
    if len(act):
        sol, *_ = np.linalg.lstsq(A[act].T, -grad, rcond=None)
        lam[act] = sol
    stat = float(np.max(np.abs(grad + A.T @ lam)))
    bad = 0.0
    for i in range(A.shape[0]):
        if at_u[i] and at_l[i]:
            continue
        if at_u[i]:
            bad = max(bad, -lam[i])
        elif at_l[i]:
            bad = max(bad, lam[i])
        else:
            bad = max(bad, abs(lam[i]))
    return {"primal": primal, "stationarity": stat, "sign": float(bad), "lam": lam}


def _inputs_map(prog, inp, i=None):
    vals = {}
    pick = (lambda a: a) if i is None else (lambda a: float(a[i]))
    t = np.broadcast_to(np.asarray(inp["t"], dtype=np.float64).reshape(-1), (inp["q"].shape[1],))
    vals[prog.syms.t[0].id] = pick(t)
    for key, nodes in (("q", prog.syms.q), ("x", prog.syms.x), ("y", prog.syms.y)):
        if nodes:
            arr = inp.get(key)
            if arr is None:
                arr = np.zeros((len(nodes), inp["q"].shape[1]))
            for j, n in enumerate(nodes):
                vals[n.id] = pick(arr[j])
    return vals


def constraint_rows(prog, inp):
    """Numeric A (N, m, nx), lb, ub (N, m) of every instance."""
    N = inp["q"].shape[1]
    vals = _inputs_map(prog, inp)
    flat = [n for r in prog.A for n in r] + list(prog.lb) + list(prog.ub)
    out = [np.broadcast_to(np.asarray(v, dtype=np.float64), (N,)) for v in dag.evaluate(flat, vals)]
    k = prog.m * prog.nx
    A = np.stack(out[:k], axis=1).reshape(N, prog.m, prog.nx)
    lb = np.stack(out[k:k + prog.m], axis=1) if prog.m else np.zeros((N, 0))
    ub = np.stack(out[k + prog.m:], axis=1) if prog.m else np.zeros((N, 0))
    return A, lb, ub


class Instance(object):
    """F and its gradient of instance i as functions of the decision vector."""

    def __init__(self, prog, inp, i):
        self.prog = prog
        self.vals = _inputs_map(prog, inp, i)
        self.nodes = [prog.F] + list(prog.g)

    def fg(self, v):
        vals = dict(self.vals)
        vals.update({n.id: float(v[j]) for j, n in enumerate(self.prog.dec)})
        out = [float(a) for a in dag.evaluate(self.nodes, vals)]
        return out[0], np.array(out[1:])


def slsqp(inst, A, lb, ub, v0):
    """SciPy SLSQP from v0 (ftol 1e-14) -> (x, F, ok).  ok: converged, or stopped because no line-search
    step decreases F any further (SLSQP's status 8, reached at 1e-14 on some well-solved instances)."""
    cons = []
    eq = np.isfinite(lb) & (lb == ub)
    lo = np.isfinite(lb) & ~eq
    hi = np.isfinite(ub) & ~eq
    if eq.any():
        cons.append({"type": "eq", "fun": lambda v: A[eq] @ v - lb[eq], "jac": lambda v: A[eq]})
    if lo.any():
        cons.append({"type": "ineq", "fun": lambda v: A[lo] @ v - lb[lo], "jac": lambda v: A[lo]})
    if hi.any():
        cons.append({"type": "ineq", "fun": lambda v: ub[hi] - A[hi] @ v, "jac": lambda v: -A[hi]})
    res = minimize(inst.fg, v0, jac=True, method="SLSQP", constraints=cons,
                   options={"ftol": 1e-14, "maxiter": 1000})
    return res.x, float(res.fun), res.status in (0, 8)
