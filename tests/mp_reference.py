"""A 50-digit referee for the controller steps, and seeded input families at kinematic singularities.
TEST INFRASTRUCTURE ONLY.

The skill's expression graph is evaluated in mpmath at 50 significant digits; fp64 inputs and graph
constants count as exact binary values.  The oracle's own algebra (oracle/clik_oracle.py) then runs
unchanged on object arrays of mpf.  Nothing here imports the kernel sources, and the only numbers this
shares with the product come from the expression graph, which test_independent_pins.py pins to sympy.  (Through
oracle_bridge it imports one lookup of the code generator, codegen.lower.kind_of, the table from constraint
class to constraint kind; no lowering or emitted code.)

Error criterion (tests/test_singular_on_host.py, tests/test_gpu_singular.py).  For an instance whose
50-digit condition number kappa satisfies kappa u < 1e-2 (u = 2^-53), a kernel result must satisfy

    |r_kernel - r_ref| <= C u kappa s + ATOL        (2-norms over the instance's vector)

where s is the size of the terms the step adds up: |v| plus |P(J_i) des_i| of every task for the pinv step
(the result of a multi-task chain can be much smaller than its terms), |(z, lam)| of the face solution for
the QP.

C = 64 comes from the sizes involved, not from observed errors: the kernels form a Gram matrix of at most
k = 9 rows from Jacobian entries that the FK chain evaluates with a relative error of a few u, factor it by
Cholesky (backward error <= (k + 1) u |G| per entry) and do two triangular solves (<= k u each) plus one
product with J (<= NS u, NS <= 7).  That adds up to 3k + NS + a few = 40 u of backward error, which the
Gram matrix amplifies by kappa; C = 64 rounds it up to the next power of two.  ATOL = 1e-12 is the
absolute floor of the north-star tolerance (BASELINE.json).  Decisions (mode flags, working-set masks) are
compared wherever their 50-digit decision margin exceeds the error bound of the quantity tested.
"""
import contextlib
import math

import mpmath as mp
import numpy as np

import oracle_bridge as ob
from oracle_bridge import orc
from casclik_b200 import cs
from casclik_b200.sym import dag

DPS = 50
U = 2.0 ** -53
C = 64.0
ATOL = 1e-12
CLAIM = 1e-2          # accuracy is claimed where kappa * u < CLAIM
RANK_BAND = 1e3       # the kernels' 1e-12 rank thresholds, widened by this factor either way


def _b(x):
    return mp.mpf(1) if x else mp.mpf(0)


_MP1 = {
    "neg": lambda a: -a, "sin": mp.sin, "cos": mp.cos, "tan": mp.tan, "asin": mp.asin, "acos": mp.acos,
    "atan": mp.atan, "exp": mp.exp, "log": mp.log, "sqrt": mp.sqrt, "fabs": abs, "sign": mp.sign,
    "floor": mp.floor, "ceil": mp.ceil, "not": lambda a: _b(a == 0),
}
_MP2 = {
    "add": lambda a, b: a + b, "sub": lambda a, b: a - b, "mul": lambda a, b: a * b,
    "div": lambda a, b: a / b, "atan2": mp.atan2, "pow": mp.power, "fmin": min, "fmax": max,
    "lt": lambda a, b: _b(a < b), "le": lambda a, b: _b(a <= b), "eq": lambda a, b: _b(a == b),
    "ne": lambda a, b: _b(a != b), "and": lambda a, b: _b(a != 0 and b != 0),
    "or": lambda a, b: _b(a != 0 or b != 0),
}
assert set(dag.OPS) == set(_MP1) | set(_MP2) | {"const", "sym", "if_else"}, "an op without a 50-digit case"


def _eval_order(order, outputs, values):
    v = {}
    for n in order:
        op = n.op
        if op == "const":
            v[n.id] = mp.mpf(n.val)
        elif op == "sym":
            v[n.id] = mp.mpf(values[n.id])
        elif op in _MP1:
            v[n.id] = _MP1[op](v[n.args[0].id])
        elif op in _MP2:
            v[n.id] = _MP2[op](v[n.args[0].id], v[n.args[1].id])
        elif op == "if_else":
            c, a, b = (v[x.id] for x in n.args)
            v[n.id] = a if c != 0 else b
        else:
            raise NotImplementedError(op)
    return [v[o.id] for o in outputs]


def mp_eval(outputs, values):
    """Evaluate DAG nodes at 50 digits.  `values`: symbol id -> float or mpf.  -> list of mpf."""
    with mp.workdps(DPS):
        return _eval_order(dag.topo(outputs), outputs, values)


def mp_num(matrix, vals, N):
    """oracle_bridge._num in mpf: cs matrix -> (N, rows, cols) object array."""
    m = matrix if isinstance(matrix, cs.GenericMatrixCommon) else cs.DM(matrix)
    r, c = m.shape
    out = np.empty((N, c * r), dtype=object)
    nodes = m.nodes() if m.numel() else []
    order = dag.topo(nodes)
    with mp.workdps(DPS):
        for i in range(N):
            vi = {k: (a[i] if np.ndim(a) else a) for k, a in vals.items()}
            out[i] = _eval_order(order, nodes, vi)
    return out.reshape(N, c, r).transpose(0, 2, 1)


@contextlib.contextmanager
def _mp_constraint_values():
    saved = ob._num
    ob._num = mp_num
    try:
        yield
    finally:
        ob._num = saved


def mp_blocks(spec, inputs):
    """The oracle Blocks of `inputs` with 50-digit entries -> (blocks, n_state)."""
    with _mp_constraint_values(), mp.workdps(DPS):
        return ob.blocks_from_skill(spec, inputs["t"], inputs["q"], inputs.get("x"), inputs.get("y"))


def take(blocks, idx):
    return [orc._take(b, np.asarray(idx)) for b in blocks]


def _f(a):
    return np.array([[float(v) for v in row] for row in np.atleast_2d(a)])


def _norm(vec):
    return math.sqrt(sum(float(x) ** 2 for x in vec))


# ----------------------------------------------------------------------------------------------
# pinv
# ----------------------------------------------------------------------------------------------

def gram_kappa(J, method="damped", lam=1e-7):
    """(sigma_max^2 + lam) / (sigma_min^2 + lam) of the Gram matrix damped_pinv factorises for J (m, n),
    at 50 digits; inf where it is singular."""
    m, n = J.shape
    wide = (n >= m) if method == "damped" else not (m >= n)
    lam = lam if method == "damped" else 0.0
    M = mp.matrix(J.tolist())
    G = M * M.T if wide else M.T * M
    for i in range(G.rows):
        G[i, i] += lam
    ev = mp.eigsy(G, eigvals_only=True)
    lo, hi = min(ev), max(ev)
    return math.inf if lo <= 0 else float(hi / lo)


def _mode_grams(bi, bits, opts):
    """The matrices damped_pinv receives in one mode: mirrors orc._mode_velocity's bookkeeping."""
    conv_last = opts.get("converge_final_set_to_max", False)
    Jl, mats, s = [], [], 0
    for b in bi:
        J = b.J[0]
        if b.kind in (orc.EQ, orc.VELEQ):
            first = not Jl
            if first:
                mats.append(J)
                if b.kind == orc.EQ:
                    Jl.append(J)
            if not first or b.kind == orc.EQ:
                mats += [np.concatenate(Jl, axis=0), J]
            Jl.append(J)
        elif b.kind == orc.SET:
            if bits[s] and conv_last and b is bi[-1]:
                mats += [np.concatenate(Jl, axis=0), J]
            if bits[s]:
                Jl.append(J)
            s += 1
    return mats


def _task_terms(bi, opts):
    """Sum over the Eq / VelEq tasks of |P(J_i) des_i| at 50 digits: the size of the terms the step adds up.
    The rounding error of a sum scales with its terms, not with the result, which cancellation between
    priority levels can make much smaller."""
    method = opts.get("pinv_method", "damped")
    lam = opts.get("damping_factor", 1e-7)
    ff = opts.get("feedforward", True)
    tot = 0.0
    for b in bi:
        if b.kind == orc.EQ:
            des = -orc._gain_times(b.gain, b.e)
        elif b.kind == orc.VELEQ:
            des = orc._bcast(b.target, 1, b.rows).astype(object)
        else:
            continue
        if ff:
            des = des - b.Jt
        tot += _norm(np.einsum("nij,nj->ni", orc.damped_pinv(b.J, method, lam), des)[0])
    return tot


def _itc_ratio(e, de, lo, hi, bnd_e, bnd_de):
    """Decision margin / error bound of orc.in_tangent_cone along its 50-digit path, and its result."""
    a = lo - e - 1e-12
    if a < 0:
        b = e - hi - 1e-12
        if b < 0:
            return min(-a / bnd_e, -b / bnd_e), True
        return min(-a / bnd_e, b / bnd_e, abs(de) / bnd_de), de < 0
    return min(a / bnd_e, abs(de) / bnd_de), de > 0


def pinv_reference(blocks, n, options=None):
    """orc.pinv_step at 50 digits, per instance.  -> dict of
      v (n, N) float64, mode (N,),
      kappa (N,): largest Gram condition number in the chosen mode,
      kappa_all (N,): the same over every mode the search tried,
      ratio (N,): smallest decision margin of the search over its error bound (< 1: either answer is right),
      scale (N,): |v| + the sizes of the task terms (_task_terms), the scale of the velocity's error bound."""
    opts = dict(options or {})
    method = opts.get("pinv_method", "damped")
    lam = opts.get("damping_factor", 1e-7)
    N = blocks[0].e.shape[0]
    n_sets = sum(1 for b in blocks if b.kind == orc.SET)
    amap = orc.activation_map(n_sets) or [[]]
    out = {"v": np.zeros((n, N)), "mode": np.zeros(N, dtype=np.int32), "kappa": np.zeros(N),
           "kappa_all": np.zeros(N), "ratio": np.full(N, np.inf), "scale": np.zeros(N)}
    with mp.workdps(DPS):
        for i in range(N):
            bi = take(blocks, [i])
            try:
                v, mode = orc.pinv_step(bi, n, opts)
                out["v"][:, i] = [float(a) for a in v[0]]
                out["mode"][i] = mode[0]
            except ZeroDivisionError:        # "standard" on an exactly singular Gram matrix
                out["v"][:, i] = np.nan
                out["mode"][i] = -9
                out["kappa"][i] = out["kappa_all"][i] = math.inf
                continue
            try:
                out["scale"][i] = _norm(v[0]) + _task_terms(bi, opts)
            except ZeroDivisionError:
                out["scale"][i] = math.inf
            last = mode[0] if mode[0] >= 0 else len(amap) - 1
            for k in range(last + 1):
                kap = max([gram_kappa(J, method, lam) for J in _mode_grams(bi, amap[k], opts)] or [1.0])
                out["kappa_all"][i] = max(out["kappa_all"][i], kap)
                if k == last:
                    out["kappa"][i] = kap
                vk, to_test = orc._mode_velocity(bi, amap[k], n, 1, opts)
                vn = _norm(vk[0])
                worst_ok, best_fail = math.inf, 0.0
                for b in to_test:
                    if b.rows != 1:
                        raise NotImplementedError("decision margins of multidim sets")
                    e, Jr, jt = b.e[0, 0], b.J[0, 0], b.Jt[0, 0]
                    de = jt + sum(Jr[j] * vk[0][j] for j in range(n))
                    lo = orc._bcast(b.set_min, 1, 1)[0, 0]
                    hi = orc._bcast(b.set_max, 1, 1)[0, 0]
                    jn = _norm(Jr)
                    bnd_e = C * U * max(1.0, abs(float(e)), abs(float(lo)), abs(float(hi)))
                    bnd_de = jn * (C * U * min(kap, 1e300) * vn + ATOL) + C * U * (abs(float(jt)) + jn * vn) + 1e-300
                    r, ok = _itc_ratio(e, de, lo, hi, bnd_e, bnd_de)
                    if ok:
                        worst_ok = min(worst_ok, float(r))
                    else:
                        best_fail = max(best_fail, float(r))
                r_mode = worst_ok if best_fail == 0.0 else best_fail
                out["ratio"][i] = min(out["ratio"][i], r_mode)
    return out


def velocity_bound(ref):
    with np.errstate(invalid="ignore"):      # kappa = inf with scale = 0: no claim is made there anyway
        return C * U * ref["kappa"] * ref["scale"] + ATOL


# ----------------------------------------------------------------------------------------------
# QP: the face of the fp64 oracle's working set, solved and certified at 50 digits
# ----------------------------------------------------------------------------------------------

def qp_mp_problem(spec, inputs, blocks=None):
    """(hdiag (nx,), A (N, m, nx), lb, ub) with 50-digit entries."""
    if blocks is None:
        blocks, _ = mp_blocks(spec, inputs)
    n_virt = spec.n_virtual_var if spec.virtual_var is not None else 0
    with mp.workdps(DPS):
        return orc.qp_matrices(blocks, spec.n_robot_var, n_virt)


def qp_face_reference(h, A, lb, ub, lam64):
    """One instance.  The working set W = {r : lam64[r] != 0} (the side from the sign) of the oracle's fp64
    solve; the face KKT system [[I, B'], [B, 0]] [z; lam_W] = [0; b_W] with B = A_W H^-1/2 is solved at 50
    digits.  -> dict(x, lam (float64), cert (bool: feasible, stationary, signs right), kappa (of the KKT
    matrix), rank_ratio (sigma_min / sigma_max of B), ratio (smallest decision margin over its bound),
    up / lo masks)."""
    m, nx = A.shape
    W = [r for r in range(m) if lam64[r] != 0.0]
    k = len(W)
    with mp.workdps(DPS):
        s = [1 / mp.sqrt(mp.mpf(float(hv))) for hv in h]
        At = [[mp.mpf(A[r, j]) * s[j] for j in range(nx)] for r in range(m)]
        bW = [mp.mpf(ub[r] if lam64[r] > 0 else lb[r]) for r in W]
        K = mp.zeros(nx + k, nx + k)
        for j in range(nx):
            K[j, j] = 1
        for a, r in enumerate(W):
            for j in range(nx):
                K[nx + a, j] = K[j, nx + a] = At[r][j]
        rhs = mp.matrix([0] * nx + bW)
        if k:
            B = mp.matrix([At[r] for r in W])
            mu = mp.eigsy(B * B.T, eigvals_only=True)
            mu_lo, mu_hi = min(mu), max(mu)
        else:
            mu_lo = mu_hi = mp.mpf(1)
        rank_ratio = float(mp.sqrt(mu_lo / mu_hi)) if mu_lo > 0 else 0.0
        if mu_lo <= 0:
            return {"x": np.full(nx, np.nan), "lam": np.full(m, np.nan), "cert": False, "kappa": math.inf,
                    "rank_ratio": 0.0, "ratio": 0.0, "up": 0, "lo": 0}
        eigs = [mp.mpf(1)] + [(1 + mp.sqrt(1 + 4 * u_)) / 2 for u_ in (mu_lo, mu_hi)] + \
               [(mp.sqrt(1 + 4 * u_) - 1) / 2 for u_ in (mu_lo, mu_hi)]
        kappa = float(max(eigs) / min(eigs))
        sol = mp.lu_solve(K, rhs)
        z = [sol[j] for j in range(nx)]
        lamW = [sol[nx + a] for a in range(k)]
        lam = [mp.mpf(0)] * m
        for a, r in enumerate(W):
            lam[r] = lamW[a]
        sn = math.sqrt(sum(float(v) ** 2 for v in list(z) + lamW))
        bnd = C * U * kappa * sn + ATOL
        tau = mp.mpf(10) ** (-30)
        cert, ratio = True, math.inf
        stat = max([abs(z[j] + sum(At[r][j] * lam[r] for r in W)) for j in range(nx)])
        cert &= stat < tau
        for r in range(m):
            row = sum(At[r][j] * z[j] for j in range(nx))
            lo_r, hi_r = mp.mpf(lb[r]), mp.mpf(ub[r])
            cert &= (row >= lo_r - tau * (1 + abs(lo_r))) and (row <= hi_r + tau * (1 + abs(hi_r)))
            if r in W:
                eq = lo_r == hi_r
                if not eq:
                    cert &= (lam[r] >= 0) if lam64[r] > 0 else (lam[r] <= 0)
                ratio = min(ratio, float(abs(lam[r])) / bnd)
            else:
                rn = math.sqrt(sum(float(a) ** 2 for a in At[r]))
                slack = min(row - lo_r, hi_r - row)
                ratio = min(ratio, float(slack) / (rn * bnd + C * U * (1 + float(max(abs(lo_r), abs(hi_r))))))
        x = np.array([float(z[j] * s[j]) for j in range(nx)])
        up = sum(1 << r for r in W if lam[r] > 0)
        lo = sum(1 << r for r in W if lam[r] < 0)
    return {"x": x, "lam": np.array([float(v) for v in lam]), "cert": bool(cert), "kappa": kappa,
            "rank_ratio": rank_ratio, "ratio": ratio, "up": up, "lo": lo, "scale": sn, "bound": bnd}


def qp_residuals(h, A, lb, ub, x, up, lo, lam=None, steps=None):
    """One instance, at 50 digits: how far a returned point x (float64) is from ending on its own working set
    (up / lo masks), as normwise backward errors.  -> the largest of
      |a_r x - b_r| over the held rows and the bound violation over all rows, over (k + 1) C u (max_r sum_j
      |a_rj x_j| + max over the held rows of |b_r|);
      with lam, |H x + A' lam|_j over (k + 1) C u (max_j |h_j x_j| + max_j sum_r |a_rj lam_r|) (stationarity).
    k is the size of the working set: each of its rows entered through one Goldfarb-Idnani step, and each step's
    full-size update of x leaves up to C u of the problem's magnitudes (the count of the module docstring) in
    the held rows.  steps = 1 replaces k + 1 for a point that one direct solve of its face produced (the
    prediction pass of the QP kernel).  Independent of kappa: whatever the conditioning, a backward-stable solver that certifies its
    face ends on it to rounding, so a working set accepted with a loose row check shows here even where x is
    still close to the reference."""
    m, nx = A.shape
    worst = 0.0
    with mp.workdps(DPS):
        xm = [mp.mpf(float(v)) for v in x]
        rows, size, bsize, devs = [], mp.mpf(0), mp.mpf(0), []
        for r in range(m):
            terms = [mp.mpf(A[r, j]) * xm[j] for j in range(nx)]
            row = sum(terms)
            size = max(size, sum(abs(t) for t in terms))
            lo_r, hi_r = mp.mpf(lb[r]), mp.mpf(ub[r])
            if (up >> r) & 1 or (lo >> r) & 1:
                b = hi_r if (up >> r) & 1 else lo_r
                bsize = max(bsize, abs(b))
                devs.append(abs(row - b))
            else:
                devs.append(max(lo_r - row, row - hi_r, 0))
        k1 = bin(up | lo).count("1") + 1 if steps is None else steps
        worst = float(max(devs) / (k1 * C * U * (size + bsize) + mp.mpf(10) ** -300))
        if lam is not None:
            lm = [mp.mpf(float(v)) for v in lam]
            g, gsize, asize = [], mp.mpf(0), mp.mpf(0)
            for j in range(nx):
                hx = mp.mpf(float(h[j])) * xm[j]
                at = [mp.mpf(A[r, j]) * lm[r] for r in range(m)]
                g.append(abs(hx + sum(at)))
                gsize, asize = max(gsize, abs(hx)), max(asize, sum(abs(t) for t in at))
            worst = max(worst, float(max(g) / (k1 * C * U * (gsize + asize) + mp.mpf(10) ** -300)))
    return worst


def face_rank_ratio(h, A, rows):
    """sigma_min / sigma_max of the rows `rows` of A H^-1/2 at 50 digits (0.0 where they are dependent): the
    quantity the multipliers' rank test looks at."""
    nx = A.shape[1]
    with mp.workdps(DPS):
        s = [1 / mp.sqrt(mp.mpf(float(hv))) for hv in h]
        B = mp.matrix([[mp.mpf(A[r, j]) * s[j] for j in range(nx)] for r in rows])
        mu = mp.eigsy(B * B.T, eigvals_only=True)
        lo, hi = min(mu), max(mu)
        return float(mp.sqrt(lo / hi)) if lo > mp.mpf(10) ** -40 * hi else 0.0


def qp_reference(spec, inputs, blocks=None):
    """qp_face_reference for every instance of a batch; the working sets come from orc.solve_qp_single on
    the fp64 problem (oracle_bridge.oracle_qp_problem).  -> list of dicts (+ 'status64')."""
    h64, A64, lb64, ub64 = ob.oracle_qp_problem(spec, inputs)
    h, A, lb, ub = qp_mp_problem(spec, inputs, blocks)
    out = []
    for i in range(A64.shape[0]):
        x64, lam64, st = orc.solve_qp_single(h64, A64[i], lb64[i], ub64[i])
        r = qp_face_reference(h, A[i], lb[i], ub[i], lam64) if st == 0 else {"cert": False}
        r["status64"] = st
        r["problem"] = (h, A[i], lb[i], ub[i])
        out.append(r)
    return out


# ----------------------------------------------------------------------------------------------
# input families at singularities (seeded, deterministic)
# ----------------------------------------------------------------------------------------------

DELTAS = [0.0] + [s * 10.0 ** -k for k in range(1, 15) for s in (1.0, -1.0)]

# The 3-row position task of the UR5 (6 joints) is rank deficient only where the arm is stretched and the
# wrist continues the line: q3 in {0, pi}, q4 = +-pi/2, q5 in {0, pi} (found by a search over the special
# values of every joint pair and triple; the elbow or the wrist alone leaves J_p of rank 3).  The two UR5
# families approach that set along q3 (elbow) and along q5 (wrist).
UR5_FAMILIES = ("elbow", "wrist")
# iiwa: q2, q4, q6 = delta alone, in pairs and all three (the straight arm).
IIWA_FAMILIES = ((1,), (3,), (5,), (1, 3), (1, 5), (3, 5), (1, 3, 5))


def singular_inputs(sc, family, draws, seed=0, reachable=True):
    """len(DELTAS) * draws instances: the scenario's own sampler for the free joints, the family's joints
    set to base + delta.  Unreachable targets are the reachable ones pushed outwards to 2.5 times their
    distance from the base, outside the workspace: an arm chasing one stretches into the singular set."""
    N = len(DELTAS) * draws
    inp = {k: (None if v is None else np.array(v)) for k, v in sc.sample(N, seed=seed).items()}
    q = inp["q"]
    rng = np.random.default_rng(seed + 1)
    d = np.repeat(np.array(DELTAS), draws)
    if family in UR5_FAMILIES:
        a = rng.choice([0.0, math.pi], N)
        b = rng.choice([0.0, math.pi], N)
        q[3] = rng.choice([0.5 * math.pi, -0.5 * math.pi], N)
        q[2], q[4] = (a + d, b) if family == "elbow" else (a, b + d)
    else:
        for j in family:
            q[j] = d
    if not reachable:
        y = inp["y"]
        if y.shape[0] == 3:
            y *= 2.5
        else:
            y[9:] *= 2.5
    inp["delta"] = d
    return inp


def family_kappa(blocks, row_block=-1):
    """Undamped 50-digit sigma_max^2 / sigma_min^2 of one constraint's Jacobian per instance (inf if singular):
    the family property, independent of the controller's damping."""
    J = blocks[row_block].J
    out = np.zeros(J.shape[0])
    with mp.workdps(DPS):
        for i in range(J.shape[0]):
            M = mp.matrix(J[i].tolist())
            G = M * M.T if J.shape[1] <= J.shape[2] else M.T * M
            ev = mp.eigsy(G, eigvals_only=True)
            out[i] = math.inf if min(ev) <= 0 else float(max(ev) / min(ev))
    return out


# ----------------------------------------------------------------------------------------------
# faces of the QP and NLP steps: solution, certificate and derivative at 50 (80) digits
# ----------------------------------------------------------------------------------------------
#
# The face problem of a working set W (masks up / lo; b_r = ub_r on an upper bit, lb_r on a lower bit):
#
#     r1 = g(x, theta) + A_W(theta)' lam_W = 0,    r2 = A_W(theta) x - b_W(theta) = 0,
#
# g = H x (QP, H = diag(h)) or grad F (NLP).  K = [[M, A_W'], [A_W, 0]] with M = H or grad^2 F(x*).
#
# Criteria of tests/test_face_reference_on_host.py and tests/test_gpu_face_reference.py, derived here.
#
# Metric and kappa.  Both kernels work in the metric of a factor L of M (QP: L = H^1/2, exact to one rounding per
# entry; NLP: the Cholesky factor of grad^2 F, whose backward error u|M| is a forward error of up to u kappa(M)
# relative), on the rows B = A_W L^-T: the scaled face matrix K' = [[I, B'], [B, 0]] has the eigenvalues 1,
# (1 +- sqrt(1 + 4 mu)) / 2 for the eigenvalues mu of B B' (as in qp_face_reference).  kappa = kappa(K') for the
# QP and kappa(K') kappa(M) for the NLP; the accuracy claim is made where kappa u < CLAIM, as for the other steps.
#
# NLP step.  x is compared in the L metric, |L'(x - x_ref)| <= C u kappa s + |L'| E_stop, s = |(L'x_ref, lam_ref)|.
# E_stop is what the two stopping rules of clik_nlp.cuh leave.  Rule 1 accepts the full step p of the subproblem
# at v with |p|_inf max(1, delta) <= tol (1 + |v|_inf); rule 2 a line-search step alpha p (alpha <= 1) with
# |p|_inf <= 100 tol (1 + |v|_inf).  Without a shift (delta = 0) p is the Newton step of the face, so the error of
# the returned point is at most |p| (alpha < 1) plus a term of second order; with a shift the iteration contracts
# by delta / (lambda + delta) per step and the error is at most |p| (1 + delta / lambda_min(M)).  Both rules
# together (where a rule runs): E_stop = 100 tol (1 + |x|_inf) sqrt(nx) (1 + delta_hat / lambda_min(M)).  delta_hat is the largest
# shift the step can have used: 0 where lambda_min(M) > 2e-12 max(1, max_j M_jj) (every Cholesky pivot is at least
# lambda_min minus (n + 1) u of the diagonal, above the step's pivot threshold 1e-12 max(1, max_j M_jj)), else the
# first shift 1e-8 max(1, max_j M_jj), which makes a positive semi-definite M factorisable.
#
# NLP backward error (every status-0 instance, whatever kappa): the stationarity residual |g(x) + A' lam|_j at the
# returned x and its multipliers.  Rule 1 leaves (H~ - H - delta) p with H~ the mean Hessian on [v, x]: at most
# tol (1 + |v|_inf) plus a term of second order; rule 2 leaves (alpha H~ - H - delta) p, at most
# (|M|_inf + delta_hat) 100 tol (1 + |x|_inf).  The rounding of the subproblem, solved in the metric of L (M = L L'),
# adds (k + 1) C u of the sizes of the terms (as qp_residuals) and (k + 1) C u |L|_2 s_L, s_L = |L'x| + |L^-1 c| +
# |L^-1 A' lam| (c = g - M x), mapped to x through L (on a row: |L^-1 a_r| s_L).
#
# Where no stopping rule runs, E_stop and both stopping terms are 0 (exact_step): the QP, and a cost quadratic in
# the decision variables without a possible shift, which the step solves by its first subproblem.  Its error is then
# arithmetic alone.  Rule 2's bound is first order in |p| (it must allow a line-search step alpha < 1), so a widened
# rule 2 can stay inside it; test_face_reference_on_host.py checks the claim of include/clik.h on the last step itself.
#
# Multipliers (NLP, metric D = I): |lam - lam_ref| <= C u kappa s + |A_W^+|_2 |g(x) - g(x_ref)|_2, the second term
# the 50-digit sensitivity of the least-squares multipliers to the kernel's own x.
#
# VJP.  theta_bar = -[u; v]' dr/dtheta with K [u; v] = [xb; 0].  The adjoint solve in the scaled metric has
# the error C u kappa |w'| (w' = [L'u; v]), which reaches u through L^-T: per theta entry k the bound is
# C u kappa (|dr1/dtheta_k|_2 |L^-1|_2 + |dr2/dtheta_k|_2) |w'|_2 + ATOL.  What the kernel's fp64 x* and lam carry
# into Phi is evaluated at 50 digits along the kernel's own point: |theta_bar_50(x_kernel, lam_50(x_kernel)) -
# theta_bar_ref|_inf is added to the bound.
#
# NaN bands (as the multipliers' rank rule): theta_bar may be NaN only where the face's sigma_min / sigma_max (in
# the kernel's metric) is below 1e-9 or, NLP only, lambda_min / max(1, lambda_max) of grad^2 F(x*) is below 1e-9
# (the kernels' 1e-12 thresholds widened by RANK_BAND), and must be NaN where either is below 1e-15.

TOL_NLP = 1e-10        # ReactiveNLPController's default options["tol"]


def exact_step(P, delta_hat):
    """True where no stopping rule runs: the QP, and an NLP whose cost is quadratic in the decision variables
    (S::NLP_QUADRATIC) with no shift possible, which clik_nlp.cuh solves by its first subproblem (`exact`).  Its
    error is then arithmetic alone, and E_stop = 0."""
    return P.qp or (P.prog.quadratic and delta_hat == 0)


class MpProblem(object):
    """One instance of a lowered program (codegen.lower.QpProgram or NlpProgram) at `dps` digits.  `vals`: symbol
    id -> float or mpf for t, q, x, y.  A (m rows of nx mpf), lb, ub; fgH(x) -> (F, g, H as an mp.matrix) of the
    cost (QP: 1/2 x' diag(h) x)."""

    def __init__(self, prog, vals, dps=DPS):
        self.prog, self.vals, self.dps = prog, dict(vals), dps
        self.qp = not hasattr(prog, "F")
        self.nx, self.m = nx, m = prog.nx, prog.m
        flat = [n for r in prog.A for n in r] + list(prog.lb) + list(prog.ub) + (list(prog.h) if self.qp else [])
        with mp.workdps(dps):
            out = _eval_order(dag.topo(flat), flat, self.vals)
        k = m * nx
        self.A = [out[r * nx:(r + 1) * nx] for r in range(m)]
        self.lb, self.ub = out[k:k + m], out[k + m:k + 2 * m]
        if self.qp:
            self.h = out[k + 2 * m:]
        else:
            self._nodes = [prog.F] + list(prog.g) + list(prog.H)
            self._order = dag.topo(self._nodes)

    def fgH(self, x):
        nx = self.nx
        with mp.workdps(self.dps):
            if self.qp:
                g = [self.h[j] * x[j] for j in range(nx)]
                return sum(g[j] * x[j] for j in range(nx)) / 2, g, mp.diag(self.h)
            vals = dict(self.vals)
            vals.update({n.id: x[j] for j, n in enumerate(self.prog.dec)})
            out = _eval_order(self._order, self._nodes, vals)
            H = mp.matrix(nx, nx)
            for i in range(nx):
                for j in range(i + 1):
                    H[i, j] = H[j, i] = out[1 + nx + i * (i + 1) // 2 + j]
            return out[0], out[1:1 + nx], H

    def rows(self, up, lo):
        """W and b_W of the masks (an upper bit selects ub, as the kernels' vjp_split_v)."""
        W = [r for r in range(self.m) if ((up | lo) >> r) & 1]
        return W, [self.ub[r] if (up >> r) & 1 else self.lb[r] for r in W]


def mp_problem(prog, inp, i, dps=DPS, theta=None):
    """MpProblem of instance i of the batch `inp` (the layout of sc.sample); theta: {symbol id: offset} added to
    the inputs at `dps` digits."""
    from nlp_oracle import _inputs_map
    vals = {k: mp.mpf(v) for k, v in _inputs_map(prog, inp, i).items()}
    with mp.workdps(dps):
        for k, d in (theta or {}).items():
            vals[k] = vals[k] + d
    return MpProblem(prog, vals, dps)


def theta_symbols(prog, rows):
    """The symbol id of each (key, row) of test_vjp_on_host.theta_rows (None where the program does not read it)."""
    syms = {"t": prog.syms.t, "q": prog.syms.q, "x": prog.syms.x, "y": prog.syms.y}
    out = []
    for key, row in rows:
        nodes = syms[key]
        j = 0 if row is None else row
        out.append(nodes[j].id if j < len(nodes) else None)
    return out


def check_derivatives(P, x, dps=120):
    """Largest |prog.g - d F| and |prog.H - d2 F| (mp.diff of prog.F, central differences with h = 1e-30 on a
    `dps`-digit evaluation: truncation ~1e-60, rounding ~1e-60) at x, relative to 1 + the largest entry: the only
    place where the NLP referee relies on the product's automatic differentiation."""
    nx = P.nx
    Q = MpProblem(P.prog, P.vals, dps)
    with mp.workdps(dps):
        step = mp.mpf(10) ** -30
        xm = [mp.mpf(v) for v in x]
        _, g, H = Q.fgH(xm)

        def F(*v):
            return Q.fgH(list(v))[0]
        worst = mp.mpf(0)
        for j in range(nx):
            d = [0] * nx
            d[j] = 1
            worst = max(worst, abs(mp.diff(F, xm, tuple(d), h=step) - g[j]) / (1 + max(abs(a) for a in g)))
            for i in range(j + 1):
                d2 = [0] * nx
                d2[i] += 1
                d2[j] += 1
                hmax = 1 + max(abs(H[a, b]) for a in range(nx) for b in range(nx))
                worst = max(worst, abs(mp.diff(F, xm, tuple(d2), h=step) - H[i, j]) / hmax)
    return float(worst)


def _face_newton(P, up, lo, x0):
    """Newton on [r1; r2] = 0 of the face from x0 until the residual is below 10^(10 - dps) (1e-40 at 50 digits).
    -> (x, lam_W, W) as mpf lists, or None where K is singular at this precision or Newton does not converge."""
    W, b = P.rows(up, lo)
    nx, k = P.nx, len(W)
    with mp.workdps(P.dps):
        tol = mp.mpf(10) ** (10 - P.dps)
        x = [mp.mpf(v) for v in x0]
        lam = [mp.mpf(0)] * k
        for _ in range(40):
            _, g, H = P.fgH(x)
            r = [g[j] + sum(P.A[W[a]][j] * lam[a] for a in range(k)) for j in range(nx)]
            r += [sum(P.A[W[a]][j] * x[j] for j in range(nx)) - b[a] for a in range(k)]
            if max(abs(v) for v in r) < tol:
                return x, lam, W
            K = mp.zeros(nx + k, nx + k)
            for i in range(nx):
                for j in range(nx):
                    K[i, j] = H[i, j]
            for a in range(k):
                for j in range(nx):
                    K[nx + a, j] = K[j, nx + a] = P.A[W[a]][j]
            try:
                d = mp.lu_solve(K, mp.matrix([-v for v in r]))
            except ZeroDivisionError:
                return None
            x = [x[j] + d[j] for j in range(nx)]
            lam = [lam[a] + d[nx + a] for a in range(k)]
    return None


def _eigs(S):
    ev = mp.eigsy(S, eigvals_only=True)
    return min(ev), max(ev)


def face_solve(P, up, lo, x0, tol=TOL_NLP):
    """The face of the working set (up, lo) at P's precision, from the kernel's x0.  -> dict of
      x, lam (m,) float64 (CasADi's signs, 0 off W), xm / lamW (mpf), W;
      kappa (the criterion's kappa), kappa_K (of K' in the kernel's metric), kappa_M (of M), rank_ratio
      (sigma_min / sigma_max of B = A_W L^-T), hess_ratio (lambda_min / max(1, lambda_max) of M), lam_min (of M);
      ratio (smallest decision margin over its bound), cert (feasible, stationary, signs right, reduced Hessian
      positive definite: for a convex F a proof of global optimality), scale s, bound (C u kappa s + ATOL), e_stop
      (the NLP's stopping error in the L metric), Lnorm / Linv (|L'|_2, |L^-1|_2)."""
    nx, m = P.nx, P.m
    W, _ = P.rows(up, lo)
    k = len(W)
    bad = {"x": np.full(nx, np.nan), "lam": np.full(m, np.nan), "cert": False, "kappa": math.inf, "kappa_K": math.inf,
           "kappa_M": math.inf, "rank_ratio": 0.0, "hess_ratio": 0.0, "ratio": 0.0, "W": W, "xm": None}
    sol = _face_newton(P, up, lo, x0)
    with mp.workdps(P.dps):
        _, _, H = P.fgH(sol[0] if sol else [mp.mpf(v) for v in x0])
        ev_lo, ev_hi = _eigs(H)
        hmax = max([mp.mpf(1)] + [abs(H[j, j]) for j in range(nx)])
        bad["hess_ratio"] = float(ev_lo / max(1, ev_hi))
        bad["lam_min"] = float(ev_lo)
        if k:
            Aw = mp.matrix([P.A[r] for r in W])
            mu0 = _eigs(Aw * Aw.T)
            bad["rank_ratio_plain"] = float(mp.sqrt(max(mu0[0], 0) / mu0[1])) if mu0[1] > 0 else 0.0
        try:                     # singular to 50 digits (an eigenvalue of rounding size) counts as singular
            L = mp.cholesky(H) if ev_lo > 0 else None
        except ValueError:
            L = None
        if L is not None:
            Bt = [mp.lu_solve(L, mp.matrix(P.A[r])) for r in W]          # rows of B = A_W L^-T
            if k:
                B = mp.matrix([[Bt[a][j] for j in range(nx)] for a in range(k)])
                mu_lo, mu_hi = _eigs(B * B.T)
            else:
                mu_lo = mu_hi = mp.mpf(1)
            bad["rank_ratio"] = rank_ratio = float(mp.sqrt(mu_lo / mu_hi)) if mu_lo > 0 else 0.0
        if sol is None or L is None:
            return bad
        x, lamW, _ = sol
        eigs = [mp.mpf(1)] + [(1 + mp.sqrt(1 + 4 * u_)) / 2 for u_ in (mu_lo, mu_hi)] + \
               [(mp.sqrt(1 + 4 * u_) - 1) / 2 for u_ in (mu_lo, mu_hi)]
        kappa_K = float(max(eigs) / min(eigs)) if mu_lo > 0 else math.inf
        kappa_M = 1.0 if P.qp else float(ev_hi / ev_lo)
        kappa = kappa_K * kappa_M
        z = L.T * mp.matrix(x)
        sn = math.sqrt(sum(float(v) ** 2 for v in list(z) + lamW))
        bnd = C * U * kappa * sn + ATOL
        delta_hat = 0.0 if ev_lo > 2e-12 * hmax else 1e-8 * float(hmax)
        xinf = max(float(abs(v)) for v in x)
        e_stop = 0.0 if exact_step(P, delta_hat) else \
            100 * tol * (1 + xinf) * math.sqrt(nx) * (1 + delta_hat / float(ev_lo))
        lam = [mp.mpf(0)] * m
        for a, r in enumerate(W):
            lam[r] = lamW[a]
        tau = mp.mpf(10) ** (-30)
        _, g, _ = P.fgH(x)
        cert = max([abs(g[j] + sum(P.A[r][j] * lam[r] for r in W)) for j in range(nx)]) < tau
        ratio = math.inf
        for r in range(m):
            row = sum(P.A[r][j] * x[j] for j in range(nx))
            lo_r, hi_r = P.lb[r], P.ub[r]
            cert &= (row >= lo_r - tau * (1 + abs(lo_r))) and (row <= hi_r + tau * (1 + abs(hi_r)))
            if r in W:
                if lo_r != hi_r:      # an equality row's multiplier may have either sign: no decision
                    cert &= (lam[r] >= 0) if (up >> r) & 1 else (lam[r] <= 0)
                    ratio = min(ratio, float(abs(lam[r])) / bnd)
            else:
                rn = float(mp.norm(mp.lu_solve(L, mp.matrix(P.A[r]))))
                slack = min(row - lo_r, hi_r - row)
                ratio = min(ratio, float(slack) / (rn * (bnd + float(mp.sqrt(ev_hi)) * e_stop)
                                                   + C * U * (1 + float(max(abs(lo_r), abs(hi_r))))))
        # reduced Hessian: M is positive definite here, hence also on the null space of A_W
    return {"x": np.array([float(v) for v in x]), "lam": np.array([float(v) for v in lam]), "xm": x, "lamW": lamW,
            "W": W, "cert": bool(cert), "kappa": kappa, "kappa_K": kappa_K, "kappa_M": kappa_M,
            "rank_ratio": rank_ratio, "rank_ratio_plain": bad.get("rank_ratio_plain", 1.0),
            "hess_ratio": float(ev_lo / max(1, ev_hi)), "lam_min": float(ev_lo), "ratio": ratio, "scale": sn,
            "bound": bnd, "e_stop": e_stop, "Lnorm": float(mp.sqrt(ev_hi)), "Linv": float(1 / mp.sqrt(ev_lo)),
            "LT": _f(L.T.tolist())}


DDPS = 80              # digits of the derivative routes
DH = mp.mpf(10) ** -25  # their central-difference step (relative to max(1, |theta_k|))


def _theta_step(P, sid):
    with mp.workdps(DDPS):
        return DH * max(1, abs(mp.mpf(P.vals[sid])))


def _shifted(P, sid, d):
    vals = dict(P.vals)
    with mp.workdps(DDPS):
        vals[sid] = mp.mpf(vals[sid]) + d
    return MpProblem(P.prog, vals, DDPS)


def face_derivative(P, up, lo, x, sids):
    """dx*/dtheta (nx, n_theta) of the face of (up, lo), W held fixed, by a central difference of the 80-digit face
    solution (h = 1e-25): from the definition, sharing nothing with codegen/vjp.py's Phi, dag.jacobian over theta
    or the adjoint solve.  x: a point near the face's solution (the Newton start).  Columns of unread symbols are 0."""
    out = np.zeros((P.nx, len(sids)), dtype=object)
    with mp.workdps(DDPS):
        for c, sid in enumerate(sids):
            if sid is None:
                out[:, c] = mp.mpf(0)
                continue
            h = _theta_step(P, sid)
            xp = _face_newton(_shifted(P, sid, h), up, lo, x)[0]
            xq = _face_newton(_shifted(P, sid, -h), up, lo, x)[0]
            out[:, c] = [(a - b) / (2 * h) for a, b in zip(xp, xq)]
    return out


def _face_residual(P, W, b, x, lamW):
    nx, k = P.nx, len(W)
    _, g, _ = P.fgH(x)
    r = [g[j] + sum(P.A[W[a]][j] * lamW[a] for a in range(k)) for j in range(nx)]
    return r + [sum(P.A[W[a]][j] * x[j] for j in range(nx)) - b[a] for a in range(k)]


def vjp_adjoint(P, up, lo, x, lamW, xb, sids):
    """The adjoint formula of include/clik.h at 50 digits: K [u; v] = [xb; 0] with K = d(r1, r2)/d(x, lam) at x,
    theta_bar = -[u; v]' dr/dtheta with x, lam_W held fixed (dr/dx and dr/dtheta by 80-digit central differences,
    h = 1e-25).  -> (theta_bar
    (n_theta,) mpf, per-theta error scale (n_theta,) float: (|dr1/dtheta_k| |L^-1| + |dr2/dtheta_k|) |[L'u; v]|)."""
    nx = P.nx
    W, b = P.rows(up, lo)
    k = len(W)
    P80 = MpProblem(P.prog, P.vals, DDPS)
    with mp.workdps(DDPS):
        # M = dg/dx of the residual itself (prog.H may differ from it by the rounding of constants the automatic
        # differentiation folds, e.g. 2/0.3^2 of the quartic cost)
        xm, lm = [mp.mpf(v) for v in x], [mp.mpf(v) for v in lamW]
        Mcol = []
        for j in range(nx):
            h = DH * max(1, abs(xm[j]))
            xp, xq = list(xm), list(xm)
            xp[j] += h
            xq[j] -= h
            Mcol.append([(a - b) / (2 * h) for a, b in zip(P80.fgH(xp)[1], P80.fgH(xq)[1])])
    with mp.workdps(P.dps):
        _, _, H = P.fgH(xm)
        K = mp.zeros(nx + k, nx + k)
        for i in range(nx):
            for j in range(nx):
                K[i, j] = Mcol[j][i]
        for a in range(k):
            for j in range(nx):
                K[nx + a, j] = K[j, nx + a] = P.A[W[a]][j]
        w = mp.lu_solve(K, mp.matrix([mp.mpf(float(v)) for v in xb] + [0] * k))
        ev_lo = _eigs(H)[0]
        Linv = float(1 / mp.sqrt(ev_lo)) if ev_lo > 0 else math.inf
        wn = float(mp.sqrt(sum((mp.cholesky(H).T * mp.matrix([w[j] for j in range(nx)]))[j] ** 2 for j in range(nx))
                           + sum(w[nx + a] ** 2 for a in range(k)))) if ev_lo > 0 else math.inf
    tb, scale = [], []
    with mp.workdps(DDPS):
        for sid in sids:
            if sid is None:
                tb.append(mp.mpf(0))
                scale.append(0.0)
                continue
            h = _theta_step(P, sid)
            rp = _face_residual(_shifted(P, sid, h), W, _shifted(P, sid, h).rows(up, lo)[1], xm, lm)
            Pm = _shifted(P, sid, -h)
            rm = _face_residual(Pm, W, Pm.rows(up, lo)[1], xm, lm)
            d = [(a - c) / (2 * h) for a, c in zip(rp, rm)]
            tb.append(-sum(w[i] * d[i] for i in range(nx + k)))
            n1 = math.sqrt(sum(float(v) ** 2 for v in d[:nx]))
            n2 = math.sqrt(sum(float(v) ** 2 for v in d[nx:]))
            scale.append((n1 * Linv + n2) * wn)
    return tb, np.array(scale)


def vjp_bound(kappa, scale):
    return C * U * kappa * scale + ATOL


def ls_multipliers(P, up, lo, x):
    """lam_W = argmin |D^1/2 (g(x) + A_W' lam)| at 50 digits at the point x, in the metric of clik_duals.cuh (QP
    D = H^-1, NLP D = I) -> (lam (m,) float64, lam_W (mpf), |(D^1/2 A_W')^+|_2 (inf where rank deficient),
    g(x) (mpf))."""
    W, _ = P.rows(up, lo)
    k = len(W)
    with mp.workdps(P.dps):
        xm = [mp.mpf(float(v)) for v in x]
        _, g, _ = P.fgH(xm)
        lam = np.zeros(P.m)
        if not k:
            return lam, [], 0.0, g
        d = [1 / mp.sqrt(h) for h in P.h] if P.qp else [mp.mpf(1)] * P.nx
        Aw = mp.matrix([[P.A[r][j] * d[j] for j in range(P.nx)] for r in W])
        G = Aw * Aw.T
        lo_ev = _eigs(G)[0]
        if lo_ev <= 0:
            return np.full(P.m, np.nan), None, math.inf, g
        sol = mp.lu_solve(G, -(Aw * mp.matrix([g[j] * d[j] for j in range(P.nx)])))
        for a, r in enumerate(W):
            lam[r] = float(sol[a])
        return lam, [sol[a] for a in range(k)], float(1 / mp.sqrt(lo_ev)), g


def nlp_residuals(P, x, up, lo, lam, tol=TOL_NLP):
    """Backward error of a returned NLP point x (float64) with its multipliers lam on its own working set, at 50
    digits, as the ratio to its bound (module comment above the face section): the stationarity residual
    |g(x) + A' lam|_j over (k + 1) C u (|g_j| + sum_r |a_rj lam_r|) + (|M|_inf + delta_hat) 100 tol (1 + |x|_inf),
    and the held-row residual / bound violation over (k + 1) C u (sum_j |a_rj x_j| + |b_r|) + |a_r|_1 100 tol
    (1 + |x|_inf) (a line-search step of rule 2 stops short of the face by at most |p|)."""
    nx, m = P.nx, P.m
    W, b = P.rows(up, lo)
    k1 = len(W) + 1
    with mp.workdps(P.dps):
        xm = [mp.mpf(float(v)) for v in x]
        lm = [mp.mpf(float(v)) for v in lam]
        _, g, H = P.fgH(xm)
        xinf = max(abs(v) for v in xm)
        hmax = max([mp.mpf(1)] + [abs(H[j, j]) for j in range(nx)])
        dhat = 0 if _eigs(H)[0] > 2e-12 * hmax else 1e-8 * hmax
        Minf = max(sum(abs(H[i, j]) for j in range(nx)) for i in range(nx))
        exact = exact_step(P, dhat)
        stop_g = 0 if exact else (Minf + dhat) * 100 * tol * (1 + xinf)
        stop_r = 0 if exact else 100 * tol * (1 + xinf)
        # the subproblem is solved in the metric of L (M = L L'): its backward error reaches x through L, so the
        # rounding of its terms s_L = |L'x| + |L^-1 c| + |L^-1 A' lam| (c = g - M x) counts with |L|_2 there
        ev_lo, ev_hi = _eigs(H)
        Linv_rows = [mp.mpf(0)] * m
        round_g = mp.mpf(0)
        try:
            L = mp.cholesky(H) if ev_lo > 0 else None
        except ValueError:       # positive definite below mpmath's tolerance: a shifted step, the stop terms cover it
            L = None
        if L is not None:
            xv = mp.matrix(xm)
            at_lam = mp.matrix([sum(P.A[r][j] * lm[r] for r in range(m)) for j in range(nx)])
            sL = mp.norm(L.T * xv) + mp.norm(mp.lu_solve(L, mp.matrix(g) - H * xv)) + mp.norm(mp.lu_solve(L, at_lam))
            round_g = k1 * C * U * mp.sqrt(ev_hi) * sL
            Linv_rows = [mp.norm(mp.lu_solve(L, mp.matrix(P.A[r]))) * k1 * C * U * sL for r in range(m)]
        worst = mp.mpf(0)
        for j in range(nx):
            at = [P.A[r][j] * lm[r] for r in range(m)]
            res = abs(g[j] + sum(at))
            worst = max(worst, res / (k1 * C * U * (abs(g[j]) + sum(abs(t) for t in at)) + round_g + stop_g
                                      + mp.mpf(10) ** -300))
        for r in range(m):
            terms = [P.A[r][j] * xm[j] for j in range(nx)]
            row = sum(terms)
            a1 = sum(abs(a) for a in P.A[r])
            if r in W:
                br = b[W.index(r)]
                dev = abs(row - br)
            else:
                br = mp.mpf(0)
                dev = max(P.lb[r] - row, row - P.ub[r], 0)
            worst = max(worst, dev / (k1 * C * U * (sum(abs(t) for t in terms) + abs(br)) + Linv_rows[r] + a1 * stop_r
                                      + mp.mpf(10) ** -300))
    return float(worst)
