"""The gradient program of the step's VJP (csrc/clik_vjp.cuh): theta_bar = -grad_theta Phi with

    Phi = u'(g(x*, theta) + A(theta)' lam) + vu'(A(theta) x* - ub(theta)) + vl'(A(theta) x* - lb(theta))

built from the program's own nodes (QP: g = H x with H = diag(h); NLP: g = grad F) over fresh per-instance
symbols for x*, lam, u and the adjoint v split by bound (vu on rows held at ub, vl on rows held at lb), so the
lb / ub choice of the working set is data, not code.  theta = (t, q, x, y) of the skill."""
from ..sym import dag


class VjpProgram(object):
    """`names`: C names of every symbol the outputs read (the skill's inputs and the fresh symbols xs_, lam_,
    u_, vu_, vl_); `t`, `q`, `x`, `y`: nodes of -dPhi/dt, -dPhi/dq_j, -dPhi/dx_j, -dPhi/dy_j."""

    def __init__(self, prog, kind):
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
        u = [dag.symbol("u_%d" % j) for j in range(n)]
        vu = [dag.symbol("vu_%d" % r) for r in range(m)]
        vl = [dag.symbol("vl_%d" % r) for r in range(m)]
        self.names = dict(prog.syms.names)
        for arr, nodes in (("xs_", xs), ("lam_", lam), ("u_", u), ("vu_", vu), ("vl_", vl)):
            for k, s in enumerate(nodes):
                self.names[s.id] = "%s[%d]" % (arr, k)
        terms = []
        for j in range(n):
            r1 = g[j]
            for r in range(m):
                if prog.A[r][j] is not dag.ZERO:
                    r1 = dag.add(r1, dag.mul(prog.A[r][j], lam[r]))
            terms.append(dag.mul(u[j], r1))
        for r in range(m):
            ax = dag.ZERO
            for j in range(n):
                if prog.A[r][j] is not dag.ZERO:
                    ax = dag.add(ax, dag.mul(prog.A[r][j], xs[j]))
            terms.append(dag.mul(vu[r], dag.sub(ax, prog.ub[r])))
            terms.append(dag.mul(vl[r], dag.sub(ax, prog.lb[r])))
        phi = dag.ZERO
        for term in terms:
            phi = dag.add(phi, term)
        syms = prog.syms
        theta = list(syms.t) + list(syms.q) + list(syms.x) + list(syms.y)
        grad = [dag.neg(d) for d in dag.jacobian([phi], theta)[0]]
        nt, nq, nx = len(syms.t), len(syms.q), len(syms.x)
        self.t = grad[0]
        self.q = grad[nt:nt + nq]
        self.x = grad[nt + nq:nt + nq + nx]
        self.y = grad[nt + nq + nx:]
