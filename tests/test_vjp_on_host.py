"""Reverse-mode derivative of the QP and NLP steps (csrc/clik_vjp.cuh, clik_qp_vjp_kernel / clik_nlp_vjp_kernel):
the emitted VJP image built for the HOST with g++ (the harness of test_kernel_code_on_host.py), against known
answers, an independent NumPy KKT reference, finite differences of the step itself and each other."""
import ctypes
import subprocess

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import build, cs, scenarios
from oracle_bridge import oracle_qp_problem, orc
from test_golden_controllers import QP, load_case
from test_kernel_code_on_host import ROOT, SHIM, _inputs, _p
from test_nlp_kernel_on_host import qp_equivalent_cost, random_convex_cost

OBSERVED = {}


def _note(key, v):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(v))


def vjp_library(ctrl, tmp_path):
    """setup_problem_functions without nvcc, then the VJP image's source (ctrl._vjp_source) built with g++."""
    saved = (build.compile_cubin, build.kernel_registers)
    build.compile_cubin = lambda source, tag="skill", **kw: (b"", str(tmp_path / "skill.cubin"))
    build.kernel_registers = lambda *a, **kw: None
    try:
        ctrl.setup_problem_functions(load=False)
    finally:
        build.compile_cubin, build.kernel_registers = saved
    source, meta = ctrl._vjp_source()
    assert meta["vjp"]
    text = source.replace("__device__ const unsigned short", "static const unsigned short")
    src = tmp_path / "skill_vjp.cpp"
    src.write_text(SHIM + text)
    so = tmp_path / "skill_vjp.so"
    subprocess.run(["g++", "-O0", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-I",
                    str(ROOT) + "/casclik_b200/csrc", "-o", str(so), str(src)], check=True)
    return ctypes.CDLL(str(so))


def _full_inputs(ctrl, inp):
    t, q, x, y = _inputs(inp)
    N = q.shape[1]
    if ctrl._nxv and x is None:
        x = np.zeros((ctrl._nxv, N))
    return t, q, x, (y if ctrl._ny else None)


def host_step(lib, ctrl, kind, inp, max_iter=None):
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    sol, status = np.full((ctrl._qn, N), np.nan), np.full(N, -9, dtype=np.int32)
    active = np.zeros((2, N), dtype=np.uint32)
    if kind == "qp":
        lib.clik_qp_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
                           None, None, _p(sol), _p(status), _p(active),
                           ctypes.c_int(max_iter or 10 * (ctrl._qn + ctrl._qm)))
    else:
        iters = np.zeros(N, dtype=np.int32)
        lib.clik_nlp_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
                            None, _p(sol), _p(status), _p(iters), _p(active), ctypes.c_int(max_iter or 50))
    return sol, status, active


def host_vjp(lib, ctrl, kind, inp, sol, status, active, sol_bar):
    """-> theta_bar (n_theta, N): rows t, q, x (virtual), y (those the skill reads)."""
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    tb, qb = np.full(N, -7.0), np.full((q.shape[0], N), -7.0)
    xb = np.full((ctrl._nxv, N), -7.0) if ctrl._nxv else None
    yb = np.full((ctrl._ny, N), -7.0) if ctrl._ny else None
    getattr(lib, "clik_%s_vjp_kernel" % kind)(
        ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
        _p(np.ascontiguousarray(sol)), _p(np.ascontiguousarray(status, dtype=np.int32)),
        _p(np.ascontiguousarray(active, dtype=np.uint32)), _p(np.ascontiguousarray(sol_bar, dtype=np.float64)),
        _p(tb), _p(qb), _p(xb), _p(yb))
    return np.vstack([tb[None]] + [a for a in (qb, xb, yb) if a is not None])


def theta_rows(ctrl, inp):
    """(key, row) of every theta entry in host_vjp's order, and the inputs with every key present."""
    t, q, x, y = _full_inputs(ctrl, inp)
    full = {"t": t.copy(), "q": q.copy()}
    if x is not None:
        full["x"] = x.copy()
    if y is not None:
        full["y"] = y.copy()
    rows = [("t", None)] + [("q", j) for j in range(q.shape[0])]
    rows += [("x", j) for j in range(ctrl._nxv)] + [("y", j) for j in range(ctrl._ny)]
    return rows, full


def perturbed(inp, key, row, delta):
    out = {k: v.copy() for k, v in inp.items()}
    if row is None:
        out[key] = out[key] + delta
    else:
        out[key][row] = out[key][row] + delta
    return out


def cotangents(n, N, seed):
    return np.random.default_rng(seed).standard_normal((n, N))


# ---- known answers (SURVEY.md §8c, cart point_skill, theta = p) --------------------------------------------

def test_cart_known_answers(tmp_path):
    t, p, dp = cs.MX.sym("t"), cs.MX.sym("p"), cs.MX.sym("dp")
    eq = cc.EqualityConstraint("min_dist_cnstr", 0.75 - p, gain=1.0, constraint_type="soft", priority=1)
    lim = cc.SetConstraint("cart_limit_cnstr", p, gain=1.0, set_min=0.0, set_max=1.0)
    spd = cc.VelocitySetConstraint("speed_limit_cnstr", p, gain=10.0, set_min=-0.275, set_max=0.275)
    spec = cc.SkillSpecification("cart_qp", t, p, robot_vel_var=dp, constraints=[eq, lim, spd])
    ctrl = cc.ReactiveQPController(spec, robot_var_weights=[1.0])
    lib = vjp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(4), "q": np.array([[0.0, 0.0, 0.6, 0.6]])}
    sol, status, active = host_step(lib, ctrl, "qp", inp)
    assert np.all(status == 0)
    assert active[0, 0] & 4 and not (active[0, 2] | active[1, 2]) & 6        # Q1: speed row at ub; Q2: no inequality
    sol_bar = np.array([[1.0, 0.0, 1.0, 0.0], [0.0, 1.0, 0.0, 1.0]])
    tb = host_vjp(lib, ctrl, "qp", inp, sol, status, active, sol_bar)
    want = np.array([0.0, -1.0, -1.001 / 1.002, -0.001 / 1.002])             # dpdot/dp, deps/dp (Q1, Q2)
    assert np.abs(tb[1] - want).max() <= 1e-12, tb[1] - want
    assert np.all(tb[0] == 0.0)                                               # nothing depends on t


# ---- independent KKT reference (NumPy: K and dr/dtheta from H, A, lb, ub with central differences) ------------

def kkt_reference(spec, inp, rows, sol, active, sol_bar, **w):
    """theta_bar_k = -[u; v]' dr/dtheta_k with K [u; v] = [xb; 0] solved by NumPy per instance."""
    N = sol.shape[1]

    def mats(i_):
        h, A, lb, ub = oracle_qp_problem(spec, i_, **w)
        return [np.broadcast_to(h, (N, len(h))) if np.ndim(h) == 1 else h, A, lb, ub]
    h, A, lb, ub = mats(inp)
    m, n = A.shape[1], A.shape[2]
    uu, vv, lams, Ws = [], [], [], []
    for i in range(N):
        W = [r for r in range(m) if ((int(active[0, i]) | int(active[1, i])) >> r) & 1]
        AW = A[i][W]
        K = np.block([[np.diag(h[i]), AW.T], [AW, np.zeros((len(W), len(W)))]])
        sl = np.linalg.solve(K, np.concatenate([sol_bar[:, i], np.zeros(len(W))]))
        _, lam, st = orc.solve_qp_single(h[i], A[i], lb[i], ub[i])
        assert st == 0
        uu.append(sl[:n])
        vv.append(sl[n:])
        lams.append(lam)
        Ws.append(W)
    out = np.zeros((len(rows), N))
    for k, (key, row) in enumerate(rows):
        val = inp[key] if row is None else inp[key][row]
        hstep = 1e-3 * np.maximum(1.0, np.abs(val))
        d = []
        for sgn in (1, -1, 2, -2):
            d.append(mats(perturbed(inp, key, row, sgn * hstep)))
        dh, dA, dlb, dub = [(8 * (a - b) - (c - e)) / (12 * (hstep[:, None, None] if a.ndim == 3 else hstep[:, None]))
                            for a, b, c, e in zip(d[0], d[1], d[2], d[3])]
        for i in range(N):
            W = Ws[i]
            bsel = np.array([dub[i, r] if (int(active[0, i]) >> r) & 1 else dlb[i, r] for r in W])
            r1 = dh[i] * sol[:, i] + dA[i].T @ lams[i]
            r2 = dA[i][W] @ sol[:, i] - bsel if W else np.zeros(0)
            out[k, i] = -(uu[i] @ r1 + vv[i] @ r2)
    return out


def _check_kkt(spec, ctrl, lib, inp, seed, **w):
    sol, status, active = host_step(lib, ctrl, "qp", inp)
    rows, full = theta_rows(ctrl, inp)
    ok = status == 0
    sel = {k: (v[..., ok] if k != "t" else v[ok]) for k, v in full.items()}
    sb = cotangents(ctrl._qn, int(ok.sum()), seed)
    got = host_vjp(lib, ctrl, "qp", sel, sol[:, ok], status[ok], active[:, ok], sb)
    ref = kkt_reference(spec, sel, rows, sol[:, ok], active[:, ok], sb, **w)
    err = np.abs(got - ref).max(axis=0) / (1 + np.abs(got).max(axis=0))
    _note("qp_vs_kkt", err.max())
    assert err.max() <= 1e-9, (err.max(), int(err.argmax()))
    return int(ok.sum())


_W = {"robot_var_weights": "w_rob", "virtual_var_weights": "w_virt", "slack_var_weights": "w_slack"}


@pytest.mark.parametrize("name", QP)
def test_qp_fixtures_match_the_kkt_reference(name, tmp_path):
    spec, inp, kwargs, _ = load_case(name)
    ctrl = cc.ReactiveQPController(spec, **kwargs)
    lib = vjp_library(ctrl, tmp_path)
    w = {_W[k]: v for k, v in kwargs.items() if k in _W}
    assert _check_kkt(spec, ctrl, lib, inp, 1, **w) == inp["q"].shape[1]


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_benchmark_qp_scenarios_match_the_kkt_reference(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(96, seed=29).items() if v is not None}
    assert _check_kkt(sc.spec, ctrl, lib, inp, 2) == 96


@pytest.mark.parametrize("seed", list(range(6)) + ["dense0", "dense1"])
def test_fuzzed_qp_skills_match_the_kkt_reference(seed, tmp_path):
    from fuzz_skills import make_dense_qp_skill, make_qp_skill
    dense = isinstance(seed, str)
    spec, weights, inp = make_dense_qp_skill(int(seed[5:])) if dense else make_qp_skill(seed)
    ctrl = cc.ReactiveQPController(spec, **weights)
    lib = vjp_library(ctrl, tmp_path)
    inp = {k: (v[..., :64] if k != "t" else v[:64]) for k, v in inp.items()}
    w = {_W[k]: v for k, v in weights.items() if k in _W}
    assert _check_kkt(spec, ctrl, lib, inp, 3, **w) >= 1


# ---- finite differences of the step itself --------------------------------------------------------------

def fd_check(lib, ctrl, kind, inp, rel, tol, seed, min_count, stencil=3):
    """x_bar' (sol(theta + h e_k) - sol(theta - h e_k)) / 2h against theta_bar_k on the instances whose working set
    is the same at every point of the stencil.

    stencil=5 (the NLP): the fourth-order difference over +-h, +-2h; a pair whose quotient misses the tolerance
    passes when a central quotient at h/100 or h/1000 meets it.  A few quartic-cost instances in 2^16 bend so sharply
    in theta that the quotient at h = 1e-4 is off by O(1) and at h = 1e-3 by more, while it converges to the VJP as
    h^2 below 1e-5 (checked on the device and the host build alike).  The SQP ends with Newton steps, so its stopping
    noise (tol 1e-10) stays well below the tolerance even at h/1000."""
    sol, status, active = host_step(lib, ctrl, kind, inp)
    rows, full = theta_rows(ctrl, inp)
    N = sol.shape[1]
    sb = cotangents(ctrl._qn, N, seed)
    got = host_vjp(lib, ctrl, kind, full, sol, status, active, sb)
    scale = 1 + np.abs(got).max(axis=0)
    count = 0
    for k, (key, row) in enumerate(rows):
        val = full[key] if row is None else full[key][row]
        h = rel * np.maximum(1.0, np.abs(val))
        same = status == 0
        f = {}
        for step in ((1, -1) if stencil == 3 else (1, -1, 2, -2, 0.01, -0.01, 0.001, -0.001)):
            sp, stp, ap = host_step(lib, ctrl, kind, perturbed(full, key, row, step * h))
            same &= (stp == 0) & np.all(ap == active, axis=0)
            f[step] = np.sum(sb * sp, axis=0)
        if stencil == 3:
            err = np.abs((f[1] - f[-1]) / (2 * h) - got[k]) / scale
            ok = err <= tol
        else:
            err = np.abs((8 * (f[1] - f[-1]) - (f[2] - f[-2])) / (12 * h) - got[k]) / scale
            ok = err <= tol
            for r in (0.01, 0.001):
                ok |= np.abs((f[r] - f[-r]) / (2 * r * h) - got[k]) / scale <= tol
        if same.any():
            _note("%s_fd" % kind, err[same].max())
            bad = np.where(same & ~ok)[0]
            assert bad.size == 0, (key, row, bad[:5], err[bad[:5]])
        count += int((same & (err <= tol)).sum())
    assert count >= min_count, count
    return count


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_qp_scenarios_match_finite_differences(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(128, seed=5).items() if v is not None}
    fd_check(lib, ctrl, "qp", inp, 1e-6, 1e-6, 7, 128)


def test_qp_expression_weights_match_finite_differences(tmp_path):
    """A cost weight that depends on q and y (H(theta)) is covered by the same Phi."""
    t, q, dq, y = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2), cs.MX.sym("y", 2)
    cons = [cc.EqualityConstraint("track", cs.vertcat(q[0] + cs.sin(q[1]) - y[0], q[0] * q[1] - y[1]), gain=2.0,
                                  constraint_type="soft"),
            cc.VelocitySetConstraint("speed", q, set_min=-0.3, set_max=0.3)]
    spec = cc.SkillSpecification("wq", t, q, robot_vel_var=dq, input_var=y, constraints=cons)
    w = cs.vertcat(1.0 + q[0] * q[0], 2.0 + cs.cos(y[1]))
    ctrl = cc.ReactiveQPController(spec, robot_var_weights=w)
    lib = vjp_library(ctrl, tmp_path)
    rng = np.random.default_rng(4)
    N = 64
    inp = {"t": np.zeros(N), "q": rng.uniform(-1, 1, (2, N)), "y": rng.uniform(-1, 1, (2, N))}
    fd_check(lib, ctrl, "qp", inp, 1e-6, 1e-6, 8, 64)


@pytest.mark.parametrize("name", sorted(scenarios.NLP_REGISTRY))
def test_nlp_scenarios_match_finite_differences(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(48, seed=6).items() if v is not None}
    fd_check(lib, ctrl, "nlp", inp, 1e-4, 1e-4, 9, 48, stencil=5)


@pytest.mark.parametrize("seed", range(3))
def test_nlp_fuzzed_convex_costs_match_finite_differences(seed, tmp_path):
    from fuzz_skills import make_qp_skill
    spec, _, inp = make_qp_skill(seed)
    ctrl = cc.ReactiveNLPController(spec, random_convex_cost(spec, seed))
    lib = vjp_library(ctrl, tmp_path)
    inp = {k: (v[..., :48] if k != "t" else v[:48]) for k, v in inp.items()}
    fd_check(lib, ctrl, "nlp", inp, 1e-4, 1e-4, 10, 8, stencil=5)


@pytest.mark.parametrize("name", QP)
def test_nlp_with_twice_the_qp_objective_gives_the_qp_vjp(name, tmp_path):
    spec, inp, kwargs, _ = load_case(name)
    qc = cc.ReactiveQPController(spec, **kwargs)
    (tmp_path / "qp").mkdir()
    (tmp_path / "nlp").mkdir()
    qlib = vjp_library(qc, tmp_path / "qp")
    nc = cc.ReactiveNLPController(spec, qp_equivalent_cost(spec, qc), slack_var_weights=qc.slack_var_weights)
    nlib = vjp_library(nc, tmp_path / "nlp")
    qs, qst, qact = host_step(qlib, qc, "qp", inp)
    ns, nst, nact = host_step(nlib, nc, "nlp", inp)
    assert np.all(qst == 0) and np.all(nst == 0)
    sb = cotangents(qc._qn, qs.shape[1], 11)
    _, full = theta_rows(qc, inp)
    qg = host_vjp(qlib, qc, "qp", full, qs, qst, qact, sb)
    ng = host_vjp(nlib, nc, "nlp", full, ns, nst, nact, sb)
    keep = np.all(qact == nact, axis=0)                       # (a row with lam = 0 may be held by one of them only)
    assert keep.mean() > 0.5
    err = np.abs(ng - qg)[:, keep].max(axis=0) / (1 + np.abs(qg[:, keep]).max(axis=0))
    _note("nlp_vs_qp", err.max())
    assert err.max() <= 1e-9


# ---- NaN and zero rules ------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_unsolved_instances_nan_unless_the_cotangent_is_zero(kind, tmp_path):
    sc = scenarios.get("ur5_qp" if kind == "qp" else "ur5_nlp_quartic")
    ctrl = sc.make_controller()
    lib = vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(8, seed=3).items() if v is not None}
    inp["q"][1, 5] = np.nan                                       # invalid (4)
    sol, status, active = host_step(lib, ctrl, kind, inp)
    assert status[5] == 4
    status[2] = 2                                                 # as an infeasible instance reports it
    sb = cotangents(ctrl._qn, 8, 12)
    sb[:, [3, 5]] = 0.0                                           # solved / unsolved with a zero cotangent
    g = host_vjp(lib, ctrl, kind, inp, sol, status, active, sb)
    assert np.isnan(g[:, 2]).all()
    assert np.all(g[:, 3] == 0.0) and np.all(g[:, 5] == 0.0)
    sb[:, 5] = 1.0
    g = host_vjp(lib, ctrl, kind, inp, sol, status, active, sb)
    assert np.isnan(g[:, 5]).all()
    assert not np.isnan(np.delete(g, [2, 5], axis=1)).any()


def test_rank_deficient_working_set_gives_nan(tmp_path):
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    cons = [cc.VelocityEqualityConstraint("a", q[0] + q[1], target=0.5),
            cc.VelocitySetConstraint("b", 2.0 * (q[0] + q[1]), set_min=-5.0, set_max=5.0, priority=1)]
    spec = cc.SkillSpecification("dup", t, q, robot_vel_var=dq, constraints=cons)
    ctrl = cc.ReactiveQPController(spec)
    lib = vjp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(2), "q": np.zeros((2, 2))}
    sol, status, active = host_step(lib, ctrl, "qp", inp)
    assert np.all(status == 0)
    active[0, 1] |= 3
    g = host_vjp(lib, ctrl, "qp", inp, sol, status, active, np.ones((2, 2)))
    assert np.isnan(g[:, 1]).all() and not np.isnan(g[:, 0]).any()


# ---- emitted source ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_quartic", "ur5_nlp_taskspeed"])
def test_vjp_source_is_the_default_source_plus_one_section(name):
    """The VJP image a controller builds on demand holds its default image unchanged."""
    ctrl = scenarios.get(name).make_controller()
    saved = build.compile_cubin
    build.compile_cubin = lambda source, tag="skill", **kw: (b"", "skill.cubin")
    try:
        ctrl.setup_problem_functions(load=False)
    finally:
        build.compile_cubin = saved
    src0, meta0 = ctrl.kernel_source, ctrl.kernel_meta
    src1, meta1 = ctrl._vjp_source()
    assert not meta0["vjp"] and meta1["vjp"] and "vjp" not in src0
    head, sep, tail = src1.partition("\n\n// ---- reverse-mode derivative of the step's output (clik_vjp.cuh) ----\n")
    assert sep and tail.count("__global__") == 1 and "_vjp_kernel(" in tail
    lines = (head + "\n").split("\n")
    o19 = [ln for ln in lines if ln.lstrip().startswith("o[19] = ")]
    assert o19 == ["  o[19] = %d;   // VJP kernels (1 QP, 2 NLP)" % (2 if "nlp" in name else 1)]
    lines.remove(o19[0])
    assert "\n".join(lines) == src0
    assert meta1["vjp_eval"]["flops"] > 0


# The parent's working_set_multipliers, verbatim: the split into working_set_rows / _qr / _solve keeps its
# operations and their order, so the multiplier kernels give the same bits.
_PARENT_ROUTINE = r'''
template <int N, int M>
bool parent_multipliers(const double* A, const double* s, const double* g, unsigned up, unsigned lo, double* lam) {
  int W[N];
  double Q[N * N], R[N * N], c[N], b[N];
  int k = 0;
  bool ok = true;
  for (int r = 0; r < M; ++r) {
    lam[r] = 0.0;
    if (((up | lo) >> r) & 1u) {
      if (k < N) W[k] = r;
      ++k;
    }
  }
  if (k > N) ok = false;
  double cmax = 0.0;
  for (int a = 0; a < k && ok; ++a) {
    double* col = &Q[a * N];
    double nrm = 0.0;
    for (int j = 0; j < N; ++j) {
      col[j] = s[j] * A[W[a] * N + j];
      nrm = fma(col[j], col[j], nrm);
    }
    cmax = fmax(cmax, sqrt(nrm));
  }
  for (int a = 0; a < k && ok; ++a) {
    double* col = &Q[a * N];
    for (int pass = 0; pass < 2; ++pass) {
      for (int l = 0; l < a; ++l) {
        double dt = 0.0;
        for (int j = 0; j < N; ++j) dt = fma(Q[l * N + j], col[j], dt);
        for (int j = 0; j < N; ++j) col[j] = fma(-dt, Q[l * N + j], col[j]);
        R[l * N + a] = (pass == 0) ? dt : R[l * N + a] + dt;
      }
    }
    double nrm = 0.0;
    for (int j = 0; j < N; ++j) nrm = fma(col[j], col[j], nrm);
    nrm = sqrt(nrm);
    if (!(nrm > 1e-12 * cmax)) { ok = false; break; }
    R[a * N + a] = nrm;
    const double inv = 1.0 / nrm;
    for (int j = 0; j < N; ++j) col[j] *= inv;
  }
  if (!ok) {
    for (int r = 0; r < M; ++r) lam[r] = NAN;
    return false;
  }
  for (int j = 0; j < N; ++j) b[j] = -s[j] * g[j];
  for (int a = 0; a < k; ++a) c[a] = 0.0;
  for (int pass = 0; pass < 2; ++pass) {
    for (int a = 0; a < k; ++a) {
      double dt = 0.0;
      for (int j = 0; j < N; ++j) dt = fma(Q[a * N + j], b[j], dt);
      for (int j = 0; j < N; ++j) b[j] = fma(-dt, Q[a * N + j], b[j]);
      c[a] += dt;
    }
  }
  for (int a = k - 1; a >= 0; --a) {
    double acc = c[a];
    for (int l = a + 1; l < k; ++l) acc = fma(-R[a * N + l], c[l], acc);
    c[a] = acc / R[a * N + a];
    lam[W[a]] = c[a];
  }
  return true;
}
extern "C" void both(int cnt, const double* A, const double* s, const double* g, const unsigned* masks, double* l0,
                     double* l1) {
  for (int i = 0; i < cnt; ++i) {
    parent_multipliers<7, 12>(A + i * 84, s + i * 7, g + i * 7, masks[2 * i], masks[2 * i + 1], l0 + i * 12);
    clik::working_set_multipliers<7, 12>(A + i * 84, s + i * 7, g + i * 7, masks[2 * i], masks[2 * i + 1], l1 + i * 12);
  }
}
'''


@pytest.mark.parametrize("flags", [["-O0", "-ffp-contract=off"], ["-O2", "-ffp-contract=fast", "-mfma"]])
def test_split_multiplier_routine_gives_the_parents_bits(flags, tmp_path):
    src = tmp_path / "split.cpp"
    src.write_text(SHIM + '#include "clik_duals.cuh"\nusing namespace std;\n' + _PARENT_ROUTINE)
    so = tmp_path / "split.so"
    r = subprocess.run(["g++"] + flags + ["-std=c++17", "-shared", "-fPIC", "-I", str(ROOT) + "/casclik_b200/csrc",
                                          "-o", str(so), str(src)], capture_output=True, text=True)
    if r.returncode != 0 and "-mfma" in flags:
        pytest.skip("the host compiler has no FMA target")
    assert r.returncode == 0, r.stderr[-2000:]
    lib = ctypes.CDLL(str(so))
    rng = np.random.default_rng(13)
    cnt = 4000
    A = rng.standard_normal((cnt, 12, 7))
    A[::7, 3] = A[::7, 1] * 2.0                             # some dependent working sets
    s = rng.uniform(0.1, 30.0, (cnt, 7))
    g = rng.standard_normal((cnt, 7))
    masks = rng.integers(0, 1 << 12, (cnt, 2), dtype=np.uint32) & rng.integers(0, 1 << 12, (cnt, 2), dtype=np.uint32)
    l0, l1 = np.zeros((cnt, 12)), np.ones((cnt, 12))
    lib.both(ctypes.c_int(cnt), _p(A), _p(s), _p(g), _p(np.ascontiguousarray(masks)), _p(l0), _p(l1))
    assert np.array_equal(l0.view(np.uint64), l1.view(np.uint64))
    assert np.isnan(l0).any(axis=1).sum() > 100 and (~np.isnan(l0).any(axis=1)).sum() > 1000


def test_report_observed_maxima():
    """Runs last in this module: the largest relative deviations of the checks above."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items())})
