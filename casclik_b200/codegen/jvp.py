"""The tangent programs of the step's JVP and Jacobian (csrc/clik_jvp.cuh): at fixed x* and lam,

    r1 = g(x*, theta) + A(theta)' lam,   r2u = A(theta) x* - ub(theta),   r2l = A(theta) x* - lb(theta)

built from the program's own nodes (QP: g = H x with H = diag(h); NLP: g = grad F) over fresh per-instance
symbols for x* and lam, so the lb / ub choice of the working set is data, not code.  theta = (t, q, x, y) of the
skill.  The JVP program is the directional derivative of (r1, r2u, r2l) along fresh tangent symbols; the
Jacobian program is their derivative with respect to every entry of theta (dag.jacobian, which keeps the reverse
rows through kinematic-chain blocks where they are smaller)."""
from ..sym import dag


def _residuals(prog, kind):
    n, m = prog.nx, prog.m
    if kind == "qp":
        xs = [dag.symbol("xs_%d" % j) for j in range(n)]
        g = [dag.mul(prog.h[j], xs[j]) for j in range(n)]
    elif kind == "nlp":
        xs = list(prog.dec)               # the cost's own decision symbols
        g = list(prog.g)
    else:
        raise ValueError(kind)
    lam = [dag.symbol("lam_%d" % r) for r in range(m)]
    r1 = []
    for j in range(n):
        acc = g[j]
        for r in range(m):
            if prog.A[r][j] is not dag.ZERO:
                acc = dag.add(acc, dag.mul(prog.A[r][j], lam[r]))
        r1.append(acc)
    r2u, r2l = [], []
    for r in range(m):
        ax = dag.ZERO
        for j in range(n):
            if prog.A[r][j] is not dag.ZERO:
                ax = dag.add(ax, dag.mul(prog.A[r][j], xs[j]))
        r2u.append(dag.sub(ax, prog.ub[r]))
        r2l.append(dag.sub(ax, prog.lb[r]))
    names = dict(prog.syms.names)
    for arr, nodes in (("xs_", xs), ("lam_", lam)):
        for k, s in enumerate(nodes):
            names[s.id] = "%s[%d]" % (arr, k)
    return names, r1, r2u, r2l


def theta_symbols(syms):
    return list(syms.t) + list(syms.q) + list(syms.x) + list(syms.y)


class JvpProgram(object):
    """`names`: C names of every symbol the outputs read (the skill's inputs, xs_, lam_ and the tangents td_,
    qd_, xd_, yd_); `r1`, `r2u`, `r2l`: nodes of the directional derivatives along (td_, qd_, xd_, yd_)."""

    def __init__(self, prog, kind):
        names, r1, r2u, r2l = _residuals(prog, kind)
        syms = prog.syms
        seeds = {}
        for arr, nodes in (("td_", syms.t), ("qd_", syms.q), ("xd_", syms.x), ("yd_", syms.y)):
            for k, s in enumerate(nodes):
                d = dag.symbol("%s%d" % (arr, k))
                names[d.id] = arr[:-1] if arr == "td_" else "%s[%d]" % (arr, k)
                seeds[s.id] = d
        self.names = names
        n, m = len(r1), len(r2u)
        out = dag.forward(r1 + r2u + r2l, seeds)
        self.r1, self.r2u, self.r2l = out[:n], out[n:n + m], out[n + m:]


class JacProgram(object):
    """`names` as JvpProgram without the tangents; `r1`, `r2u`, `r2l`: rows of nodes, one column per entry of
    theta = (t, q, x, y)."""

    def __init__(self, prog, kind):
        self.names, r1, r2u, r2l = _residuals(prog, kind)
        n, m = len(r1), len(r2u)
        rows = dag.jacobian(r1 + r2u + r2l, theta_symbols(prog.syms))
        self.n_theta = len(theta_symbols(prog.syms))
        self.r1, self.r2u, self.r2l = rows[:n], rows[n:n + m], rows[n + m:]
