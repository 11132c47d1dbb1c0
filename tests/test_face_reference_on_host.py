"""The NLP step, the multipliers and the QP / NLP VJP at and near kinematic singularities, against the 50-digit face
solutions of tests/mp_reference.py.  The host (g++) build of the VJP image (the default image plus
clik_<kind>_vjp_kernel) runs through the harness of test_vjp_on_host.py on the singular families of
test_singular_on_host.py, on the benchmark samplers, on a sweep of the task-speed cost's damping eps through the NLP
step's shift threshold down to an exactly singular Hessian, and on Moe-2016's rows with the task-speed cost.

Criteria (derived in mp_reference.py, above the face section), where kappa u < 1e-2:
  NLP x in the L metric within C u kappa s + |L'| E_stop; the kernel's working set certified wherever the 50-digit
  decision margin exceeds its bound; NLP multipliers within C u kappa s + |A_W^+| |g(x) - g(x_ref)|; theta_bar within
  C u kappa (per-theta scale) + the error the kernel's x* and lam carry into Phi (evaluated at 50 digits).
Whatever kappa: every status-0 NLP point passes the backward-error check on its own working set; theta_bar and the
multipliers are NaN only inside the NaN bands and NaN wherever the bands require it; an all-zero cotangent gives
exactly 0 on every instance, solved or not.  The last test prints the largest ratios of error to bound."""
import ctypes

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import cs, fk, scenarios
import mp_reference as mr
from nlp_oracle import constraint_rows
from test_kernel_code_on_host import _p
from test_singular_on_host import family_batch
from test_vjp_on_host import _full_inputs, host_step, host_vjp, kkt_reference, theta_rows, vjp_library

OBSERVED = {}
NAN_ALLOWED, NAN_REQUIRED = 1e-12 * mr.RANK_BAND, 1e-12 / mr.RANK_BAND
EPS = (1e-3, 1e-6, 1e-9, 1e-12, 1e-14, 0.0)


def _note(key, v):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(v))


def taskspeed_cost(spec, p, eps):
    """|J_p(q) dq|^2 + eps |dq|^2 for the position p(q) (eps = 0: no damping, an exactly singular Hessian)."""
    q, dq = spec.robot_var, spec.robot_vel_var
    v = cs.mtimes(cs.jacobian(p, q), dq)
    return cs.dot(v, v) + eps * cs.dot(dq, dq) if eps else cs.dot(v, v)


def make_case(name):
    """-> (kind, scenario whose sampler and families give the inputs, controller)."""
    if name in ("ur5_qp", "ur5_moe2016_qp"):
        sc = scenarios.get(name)
        return "qp", sc, sc.make_controller()
    if name in scenarios.NLP_REGISTRY:
        sc = scenarios.get(name)
        return "nlp", sc, sc.make_controller()
    if name.startswith("eps_"):
        sc = scenarios.get("ur5_qp")
        p = fk.ur5()["T_fk"](sc.spec.robot_var)[:3, 3]
        return "nlp", sc, cc.ReactiveNLPController(sc.spec, taskspeed_cost(sc.spec, p, float(name[4:])))
    if name.startswith("offaxis_eps_"):
        # a task point off the tool axis: J_p has no structurally zero column, so at eps = 0 the Hessian is singular
        # without a zero row, and its trailing Cholesky pivots are rounding noise of either sign
        sc = scenarios.get("ur5_qp")
        T = fk.ur5()["T_fk"](sc.spec.robot_var)
        p = cs.mtimes(T[:3, :3], cs.DM([0.1, 0.05, 0.08])) + T[:3, 3]
        return "nlp", sc, cc.ReactiveNLPController(sc.spec, taskspeed_cost(sc.spec, p, float(name[12:])))
    if name == "quartic_offset":
        # ur5_nlp_quartic's cost plus 1e6: the cost is large, so the rounding floor of stopping rule 2 (|dF| <= 1e-15 |F|)
        # ends the iteration there, not rule 1
        sc = scenarios.get("ur5_nlp_quartic")
        return "nlp", sc, cc.ReactiveNLPController(sc.spec, sc.cost_expr + 1e6)
    assert name == "moe2016_taskspeed"
    sc = scenarios.get("ur5_moe2016_qp")
    p = cs.vertcat(*[c.expression for c in sc.spec.constraints if c.label.startswith("colav")])
    return "nlp", sc, cc.ReactiveNLPController(sc.spec, taskspeed_cost(sc.spec, p, 1e-3))


def program(kind, ctrl):
    return ctrl._prog if kind == "nlp" else ctrl._program()


def host_duals(lib, ctrl, kind, inp, sol, status, active):
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    lam = np.full((ctrl._qm, N), -7.0)
    getattr(lib, "clik_%s_duals_kernel" % kind)(
        ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y), _p(sol),
        _p(np.ascontiguousarray(status, dtype=np.int32)), _p(np.ascontiguousarray(active, dtype=np.uint32)), _p(lam))
    return lam


def subsample(inp, idx):
    return {k: (v[..., idx] if k != "t" else v[idx]) for k, v in inp.items() if v is not None and k != "delta"}


def nan_band(kernel_nan, f, kind, what):
    """The NaN rule of theta_bar: NaN only where the face's rank ratio or (NLP) the Hessian's ratio, or the face's rank
    ratio in the plain metric of the NLP multipliers (clik_vjp.cuh computes lam first), is below NAN_ALLOWED, and NaN
    wherever the rank ratio or the Hessian's ratio is below NAN_REQUIRED."""
    low = min(f["rank_ratio"], f["hess_ratio"] if kind == "nlp" else 1.0)
    if kernel_nan:
        allowed = min(low, f.get("rank_ratio_plain", 1.0) if kind == "nlp" else 1.0)
        assert allowed < NAN_ALLOWED, (what, "NaN theta_bar on a regular face", f["rank_ratio"], f["hess_ratio"])
        _note("vjp NaN instances (inside the band)", OBSERVED.get("vjp NaN instances (inside the band)", 0) + 1)
    else:
        assert low > NAN_REQUIRED, (what, "finite theta_bar where the band requires NaN", f["rank_ratio"],
                                    f["hess_ratio"])


def check_batch(name, kind, ctrl, lib, inp, xb_seed=1, both_bits=False):
    """Every criterion of the module docstring on the batch `inp`, host build (every instance against the referee).
    both_bits: every held equality row (lb = ub) is handed to the multipliers and the VJP with both mask bits set, a
    working set the API accepts (it describes the same face, so theta_bar must not change)."""
    sol, status, active = host_step(lib, ctrl, kind, inp)
    if both_bits:
        _, lb, ub = constraint_rows(program(kind, ctrl), inp)
        eq = ((lb == ub) * (1 << np.arange(lb.shape[1]))).sum(axis=1).astype(np.uint32)
        held = (active[0] | active[1]) & eq
        assert held.any()
        active = np.ascontiguousarray(np.stack([active[0] | held, active[1] | held]))
    _, full = theta_rows(ctrl, inp)
    zero = host_vjp(lib, ctrl, kind, full, sol, status, active, np.zeros_like(sol))
    assert np.all(zero == 0.0), (name, "an all-zero cotangent must give exactly 0")
    xb = np.random.default_rng(xb_seed).standard_normal(sol.shape)
    tb = host_vjp(lib, ctrl, kind, full, sol, status, active, xb)
    lam = host_duals(lib, ctrl, kind, inp, sol, status, active)
    return check_outputs(name, kind, ctrl, inp, sol, status, active, lam, xb, tb)


def check_outputs(name, kind, ctrl, inp, sol, status, active, lam, xb, tb, tol=mr.TOL_NLP):
    """The referee's checks of one batch's step (sol, status, active), multipliers lam and theta_bar tb for the
    cotangent xb.  -> instance counts."""
    prog = program(kind, ctrl)
    rows, _ = theta_rows(ctrl, inp)
    sids = mr.theta_symbols(prog, rows)
    N = sol.shape[1]
    counts = {"solved": 0, "claim": 0, "undecided": 0}
    for i in range(N):
        what = (name, i)
        if status[i] != 0:
            assert np.isnan(tb[:, i]).all(), what
            continue
        counts["solved"] += 1
        up, lo = int(active[0, i]), int(active[1, i])
        P = mr.mp_problem(prog, inp, i)
        f = mr.face_solve(P, up, lo, sol[:, i], tol)
        nan_band(np.isnan(tb[:, i]).any(), f, kind, what)
        assert np.isnan(tb[:, i]).all() or np.isfinite(tb[:, i]).all(), what
        if kind == "nlp":
            # multipliers: the rank rule of the multiplier kernel (metric D = I)
            plain = f.get("rank_ratio_plain", 1.0)
            if np.isnan(lam[:, i]).any():
                assert np.isnan(lam[:, i]).all() and plain < NAN_ALLOWED, (what, "NaN multipliers", plain)
            else:
                assert plain > NAN_REQUIRED, (what, "finite multipliers on a dependent face", plain)
            # backward error on its own working set, whatever kappa
            lk = lam[:, i] if np.isfinite(lam[:, i]).all() else mr.ls_multipliers(P, up, lo, sol[:, i])[0]
            if np.isfinite(lk).all():
                r = mr.nlp_residuals(P, sol[:, i], up, lo, lk, tol)
                _note("nlp backward error " + name, r)
                assert r <= 1.0, (what, "backward error / bound", r)
        if f["xm"] is None or f["kappa"] * mr.U >= mr.CLAIM:
            continue
        counts["claim"] += 1
        if f["ratio"] > 1.0:
            assert f["cert"], (what, "the kernel's working set fails the 50-digit certificate", f["ratio"])
        else:
            counts["undecided"] += 1
        if kind == "nlp":
            rx = np.linalg.norm(f["LT"] @ (sol[:, i] - f["x"])) / (f["bound"] + f["Lnorm"] * f["e_stop"])
            _note("nlp x " + name, rx)
            assert rx <= 1.0, (what, "x error / bound", rx, f["kappa"])
            if np.isfinite(lam[:, i]).all():
                _, _, ainv, gk = mr.ls_multipliers(P, up, lo, sol[:, i])
                _, _, _, gr = mr.ls_multipliers(P, up, lo, f["x"])
                dg = float(np.sqrt(sum((float(a) - float(b)) ** 2 for a, b in zip(gk, gr))))
                rl = np.linalg.norm(lam[:, i] - f["lam"]) / (f["bound"] + ainv * dg)
                _note("nlp lam " + name, rl)
                assert rl <= 1.0, (what, "multiplier error / bound", rl, f["kappa"])
        if np.isnan(tb[:, i]).any():
            continue
        ref, scale = mr.vjp_adjoint(P, up, lo, f["xm"], f["lamW"], xb[:, i], sids)
        ref = np.array([float(v) for v in ref])
        # what the kernel's own x* and lam carry into Phi, at 50 digits
        _, lam_k, _, _ = mr.ls_multipliers(P, up, lo, sol[:, i])
        carried = 0.0
        if lam_k is not None:
            at_k, _ = mr.vjp_adjoint(P, up, lo, sol[:, i], lam_k, xb[:, i], sids)
            carried = np.abs(np.array([float(v) for v in at_k]) - ref)
        rv = np.abs(tb[:, i] - ref) / (mr.vjp_bound(f["kappa"], scale) + carried)
        _note("%s vjp %s" % (kind, name), rv.max())
        assert rv.max() <= 1.0, (what, "theta_bar error / bound", rv.max(), f["kappa"])
    _note("undecided " + name, counts["undecided"])
    return counts


_LIB = {}


def case(name, tmp_path):
    if name not in _LIB:
        kind, sc, ctrl = make_case(name)
        d = tmp_path / name
        d.mkdir(exist_ok=True)
        _LIB[name] = (kind, sc, ctrl, vjp_library(ctrl, d))
    return _LIB[name]


def family_sub(sc, stride):
    """One draw per delta of every family (reachable and unreachable targets), every `stride`-th instance."""
    inp, labels = family_batch(sc, 1)
    idx = np.arange(0, inp["q"].shape[1], stride)
    return subsample(inp, idx), inp["delta"][idx]


# ---- the referee's own checks ------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["ur5_nlp_taskspeed", "ur5_nlp_quartic", "eps_1e-14", "moe2016_taskspeed"])
def test_program_derivatives_agree_with_mp_diff(name, tmp_path):
    """prog.g and prog.H against mp.diff of prog.F, on a sampler point and a family point.  Where the automatic
    differentiation folds a constant of F into a new fp64 constant (the quartic cost's 1/0.3 and 2/0.3^2) the derivative
    graph is exact only to that constant's rounding, so the tolerance is 8u there; elsewhere 1e-40."""
    kind, sc, ctrl, lib = case(name, tmp_path)
    prog = program(kind, ctrl)
    consts = [{n.val for n in mr.dag.topo(nodes) if n.op == "const"} for nodes in ([prog.F], list(prog.g) + prog.H)]
    tol = 8 * mr.U if consts[1] - consts[0] - {0.0} - {2 * c for c in consts[0]} else 1e-40
    fam, _ = family_sub(sc, 29)
    for inp in ({k: v for k, v in sc.sample(2, seed=3).items() if v is not None}, fam):
        P = mr.mp_problem(prog, inp, 0)
        x = np.random.default_rng(2).uniform(-0.5, 0.5, prog.nx)
        err = mr.check_derivatives(P, x)
        _note("referee: prog.g / prog.H vs mp.diff " + name, err)
        assert err < tol, (name, err)


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic"])
def test_derivative_routes_agree(name, tmp_path):
    """face_derivative (central difference of the 80-digit face solution) and the adjoint formula at 50 digits agree
    to 1e-30 on the benchmark sampler; for the QP both agree with test_vjp_on_host.kkt_reference within its 1e-9."""
    kind, sc, ctrl, lib = case(name, tmp_path)
    prog = program(kind, ctrl)
    inp = {k: v for k, v in sc.sample(6, seed=17).items() if v is not None}
    sol, status, active = host_step(lib, ctrl, kind, inp)
    assert np.all(status == 0)
    rows, full = theta_rows(ctrl, inp)
    sids = mr.theta_symbols(prog, rows)
    xb = np.random.default_rng(4).standard_normal(sol.shape)
    refs = np.zeros((len(rows), sol.shape[1]))
    for i in range(sol.shape[1]):
        P = mr.mp_problem(prog, inp, i)
        up, lo = int(active[0, i]), int(active[1, i])
        f = mr.face_solve(P, up, lo, sol[:, i])
        assert f["cert"], (name, i)
        ta, _ = mr.vjp_adjoint(P, up, lo, f["xm"], f["lamW"], xb[:, i], sids)
        D = mr.face_derivative(P, up, lo, f["xm"], sids)
        with mr.mp.workdps(mr.DDPS):
            tc = [sum(mr.mp.mpf(float(xb[j, i])) * D[j, c] for j in range(prog.nx)) for c in range(len(sids))]
            gap = max(abs(a - b) / (1 + abs(b)) for a, b in zip(ta, tc))
        _note("referee: adjoint vs face derivative", gap)
        assert gap < 1e-30, (name, i, float(gap))
        refs[:, i] = [float(v) for v in tc]
    if kind == "qp":
        kkt = kkt_reference(sc.spec, full, rows, sol, active, xb)
        err = np.abs(kkt - refs).max(axis=0) / (1 + np.abs(refs).max(axis=0))
        _note("referee: face derivative vs kkt_reference", err.max())
        assert err.max() <= 1e-9, err.max()


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_taskspeed"])
def test_vjp_with_equality_rows_held_at_both_bits(name, tmp_path):
    """The soft position rows are equality rows; held at both bits their bound derivative counts once."""
    kind, sc, ctrl, lib = case(name, tmp_path)
    inp, _ = family_sub(sc, 4)
    counts = check_batch(name + " both bits", kind, ctrl, lib, inp, both_bits=True)
    assert counts["claim"] >= counts["solved"] // 3, counts
    # and against the same instances' theta_bar on the kernel's own (single-bit) masks: the same face
    sol, status, active = host_step(lib, ctrl, kind, inp)
    _, lb, ub = constraint_rows(program(kind, ctrl), inp)
    eq = ((lb == ub) * (1 << np.arange(lb.shape[1]))).sum(axis=1).astype(np.uint32)
    held = (active[0] | active[1]) & eq
    both = np.ascontiguousarray(np.stack([active[0] | held, active[1] | held]))
    _, full = theta_rows(ctrl, inp)
    xb = np.random.default_rng(2).standard_normal(sol.shape)
    one = host_vjp(lib, ctrl, kind, full, sol, status, active, xb)
    two = host_vjp(lib, ctrl, kind, full, sol, status, both, xb)
    assert np.array_equal(np.isnan(one), np.isnan(two))
    ok = np.isfinite(one).all(axis=0)
    gap = np.abs(one - two)[:, ok].max(axis=0) / (1 + np.abs(one[:, ok]).max(axis=0))
    _note("both bits vs single bit, relative " + name, gap.max())
    assert gap.max() <= 8 * mr.U, gap.max()


# ---- QP VJP --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_qp_vjp_near_singularities(name, tmp_path):
    kind, sc, ctrl, lib = case(name, tmp_path)
    inp, _ = family_sub(sc, 1 if name == "ur5_moe2016_qp" else 2)
    counts = check_batch(name, kind, ctrl, lib, inp)
    assert counts["claim"] >= counts["solved"] // 3, counts
    samp = {k: v for k, v in sc.sample(32, seed=9).items() if v is not None}
    counts = check_batch(name + " sampler", kind, ctrl, lib, samp)
    assert counts["claim"] == 32, counts


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_qp_vjp_on_dependent_faces(name, tmp_path):
    """The working sets of test_multipliers_rank_rule_on_dependent_faces handed to the VJP kernel: a joint-limit row
    with the speed row of the same joint (exactly dependent), and the three Moe-2016 box rows on the singular
    families (their rank ratio sweeps through 1e-12).  The NaN band must hold on every instance, both ways."""
    kind, sc, ctrl, lib = case(name, tmp_path)
    prog = program(kind, ctrl)
    inp, _ = family_sub(sc, 1)
    sol, _, _ = host_step(lib, ctrl, kind, inp)
    sol = np.ascontiguousarray(np.where(np.isfinite(sol), sol, 0.0))
    N = sol.shape[1]
    if name == "ur5_qp":
        j = np.arange(N) % 6
        up = ((1 << (3 + j)) | (1 << (9 + j))).astype(np.uint32)
    else:
        up = np.full(N, 7, dtype=np.uint32)
    active = np.ascontiguousarray(np.stack([up, np.zeros(N, dtype=np.uint32)]))
    _, full = theta_rows(ctrl, inp)
    tb = host_vjp(lib, ctrl, kind, full, sol, np.zeros(N, dtype=np.int32), active, np.ones_like(sol))
    nan = np.isnan(tb).any(axis=0)
    ratios = []
    for i in range(N):
        f = mr.face_solve(mr.mp_problem(prog, inp, i), int(up[i]), 0, sol[:, i])
        nan_band(nan[i], f, kind, (name, i))
        ratios.append(f["rank_ratio"])
    ratios = np.array(ratios)
    if name == "ur5_qp":
        assert nan.all() and np.all(ratios == 0.0)
    else:
        assert nan.any() and (~nan).any() and ((ratios > NAN_REQUIRED) & (ratios < NAN_ALLOWED)).any()


_QR = r'''
extern "C" void qr(int cnt, int k, double* Q, double* R, int* ok) {
  for (int i = 0; i < cnt; ++i) ok[i] = clik::working_set_qr<9>(k, Q + i * 81, R + i * 81);
}
'''


def test_working_set_qr_is_orthonormal_on_nearly_dependent_faces(tmp_path):
    """The QR that the multipliers and the VJP share (clik_duals.cuh working_set_qr), on the three Moe-2016 box rows in
    the metric of H along the singular families, whose sigma_min / sigma_max sweeps down to the rank threshold.  Two
    Gram-Schmidt passes leave Q orthonormal to working precision whatever that ratio (|Q'Q - I| <= (k + 1) C u), and
    every accepted face reconstructs its columns, |QR - B| <= (k + 1) C u |B|; one pass would leave u sigma_max /
    sigma_min."""
    import subprocess
    from oracle_bridge import oracle_qp_problem
    from test_kernel_code_on_host import ROOT, SHIM
    src = tmp_path / "qr.cpp"
    src.write_text(SHIM + '#include "clik_duals.cuh"\nusing namespace std;\n' + _QR)
    so = tmp_path / "qr.so"
    subprocess.run(["g++", "-O0", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-I",
                    str(ROOT) + "/casclik_b200/csrc", "-o", str(so), str(src)], check=True)
    lib = ctypes.CDLL(str(so))
    sc = scenarios.get("ur5_moe2016_qp")
    inp, _ = family_batch(sc, 4)
    h, A, _, _ = oracle_qp_problem(sc.spec, subsample(inp, np.arange(inp["q"].shape[1])))
    B = A[:, :3, :] / np.sqrt(h)                                  # (N, 3, 9): the columns D^1/2 a_r
    N, k = B.shape[0], 3
    Q = np.zeros((N, 9, 9))
    Q[:, :k, :] = B
    R, ok = np.zeros((N, 9, 9)), np.zeros(N, dtype=np.int32)
    lib.qr(ctypes.c_int(N), ctypes.c_int(k), _p(Q), _p(R), _p(ok))
    bound = (k + 1) * mr.C * mr.U
    ratios = []
    for i in np.nonzero(ok)[0]:
        q, r = Q[i, :k, :], np.triu(R[i, :k, :k])                 # R[l * 9 + a]: row l, column a
        ratios.append((np.abs(q @ q.T - np.eye(k)).max() / bound,
                       np.abs(r.T @ q - B[i]).max() / (bound * np.abs(B[i]).max())))
    worst = np.max(ratios, axis=0)
    _note("working_set_qr orthogonality / bound", worst[0])
    _note("working_set_qr reconstruction / bound", worst[1])
    assert worst.max() <= 1.0, worst
    assert ok.sum() > N // 2 and (~ok.astype(bool)).any()


# ---- NLP step, multipliers and VJP ---------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["ur5_nlp_taskspeed", "ur5_nlp_quartic", "moe2016_taskspeed"])
def test_nlp_near_singularities(name, tmp_path):
    kind, sc, ctrl, lib = case(name, tmp_path)
    inp, _ = family_sub(sc, 2)
    samp = {k: v for k, v in sc.sample(16, seed=9).items() if v is not None}
    counts = check_batch(name, kind, ctrl, lib, inp)
    counts_s = check_batch(name + " sampler", kind, ctrl, lib, samp)
    assert counts_s["claim"] == 16 and counts["claim"] >= counts["solved"] // 2, (counts, counts_s)


def test_nlp_singular_hessian_without_a_zero_column(tmp_path):
    """eps = 0 with a task point off the tool axis: the Hessian is singular but no row or column is zero, so the VJP's
    rejection rests on its pivot threshold alone.  The NaN band requires NaN on every solved instance."""
    kind, sc, ctrl, lib = case("offaxis_eps_0", tmp_path)
    inp, _ = family_sub(sc, 2)
    samp = {k: v for k, v in sc.sample(32, seed=10).items() if v is not None}
    for part, data in (("", inp), (" sampler", samp)):
        counts = check_batch("offaxis_eps_0" + part, kind, ctrl, lib, data)
        assert counts["solved"] == data["q"].shape[1], counts


def last_step_ratio(lib, ctrl, inp, tol=mr.TOL_NLP):
    """|x - v|_inf / (100 tol (1 + max(|x|_inf, |v|_inf))) per solved instance, where v is the point the last SQP
    iteration started from: the same step run with max_iter = iterations - 1 (the iteration is deterministic).  Both
    stopping rules of include/clik.h bound this by 1 (rule 1 accepts |p| max(1, delta) <= tol (1 + |v|_inf), rule 2
    a line-search step alpha p, alpha <= 1, with |p| <= 100 tol (1 + |x|_inf)).  Instances of a quadratic cost solved
    by their first subproblem stop without a rule and are left out.  -> (ratios, number of instances checked)."""
    from test_nlp_kernel_on_host import run_step
    sol, status, iters, _ = run_step(lib, ctrl, inp)
    N = sol.shape[1]
    v = np.zeros_like(sol)
    for k in np.unique(iters[status == 0]):
        if k < 2:
            continue
        sel = np.nonzero((status == 0) & (iters == k))[0]
        vp, st, _, _ = run_step(lib, ctrl, subsample(inp, sel), max_iter=int(k) - 1)
        assert np.all(st == 1)
        v[:, sel] = vp
    keep = (status == 0) & ~((iters == 1) & ctrl._prog.quadratic)
    scale = 100 * tol * (1 + np.maximum(np.abs(sol).max(axis=0), np.abs(v).max(axis=0)))
    return (np.abs(sol - v).max(axis=0) / scale)[keep], int(keep.sum()) if N else 0


@pytest.mark.parametrize("name", ["ur5_nlp_quartic", "quartic_offset", "eps_1e-14", "offaxis_eps_0"])
def test_nlp_last_step_meets_the_stopping_rules(name, tmp_path):
    """The claim of include/clik.h about status 0, checked on the last step itself: the quartic cost (rule 1), the
    same cost plus 1e6 (rule 2 ends it), and the shifted iteration (eps = 1e-14, and eps = 0 off the tool axis).  On the offset cost
    the step is also checked against the referee."""
    kind, sc, ctrl, lib = case(name, tmp_path)
    inp, _ = family_sub(sc, 2)
    samp = {k: v for k, v in sc.sample(32, seed=11).items() if v is not None}
    checked = 0
    for data in (inp, samp):
        r, n = last_step_ratio(lib, ctrl, data)
        checked += n
        if n:
            _note("last step / stopping rule " + name, r.max())
            assert r.max() <= 1.0, (name, r.max(), int(np.argmax(r)))
    assert checked >= 32, checked
    if name == "quartic_offset":
        check_batch(name, kind, ctrl, lib, inp)
        check_batch(name + " sampler", kind, ctrl, lib, samp)


@pytest.mark.parametrize("eps", EPS)
def test_nlp_task_speed_damping_sweep(eps, tmp_path):
    """|J_p dq|^2 + eps |dq|^2 on ur5_qp's rows: eps crosses the step's shift threshold 1e-12 max(1, max|H_jj|)
    (eps <= 1e-14 runs the shifted iteration) and ends at an exactly singular Hessian (eps = 0), where the VJP must
    be NaN on every solved instance."""
    name = "eps_%g" % eps
    kind, sc, ctrl, lib = case(name, tmp_path)
    inp, _ = family_sub(sc, 4)
    samp = {k: v for k, v in sc.sample(8, seed=10).items() if v is not None}
    for part, data in (("", inp), (" sampler", samp)):
        counts = check_batch(name + part, kind, ctrl, lib, data)
        _note("claimed instances " + name + part, counts["claim"])
        if eps >= 1e-9:
            assert counts["claim"] >= counts["solved"] // 2, counts


def test_report_observed_maxima():
    """Runs last in this module: the largest ratios of error to bound, and the instance counts."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items())})
