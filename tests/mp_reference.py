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
