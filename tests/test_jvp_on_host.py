"""Forward-mode derivative and Jacobian of the QP and NLP steps (csrc/clik_jvp.cuh, clik_<kind>_jvp_kernel /
clik_<kind>_jacobian_kernel): the emitted JVP image built for the HOST with g++ (the harness of
test_vjp_on_host.py), against the host VJP (the adjoint identity), an independent NumPy KKT reference, directional
finite differences of the step itself, known answers, the 50-digit face derivative and the rules of include/clik.h."""
import ctypes
import subprocess

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import build, cs, scenarios
import mp_reference as mr
from nlp_oracle import constraint_rows
from oracle_bridge import oracle_qp_problem, orc
from test_face_reference_on_host import case, family_sub, nan_band, program
from test_golden_controllers import QP, load_case
from test_kernel_code_on_host import ROOT, SHIM, _p
from test_nlp_kernel_on_host import random_convex_cost
from test_vjp_on_host import (_W, _full_inputs, host_step, host_vjp, perturbed, theta_rows, vjp_library)
from test_vjp_api import _ctrl, _setup_without_nvcc, _wide_spec

OBSERVED = {}


def _note(key, v):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(v))


def jvp_library(ctrl, tmp_path):
    """setup_problem_functions without nvcc, then the JVP image's source (ctrl._jvp_source) built with g++."""
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._jvp_source()
    assert meta["jvp"]
    text = source.replace("__device__ const unsigned short", "static const unsigned short")
    src = tmp_path / "skill_jvp.cpp"
    src.write_text(SHIM + text)
    so = tmp_path / "skill_jvp.so"
    subprocess.run(["g++", "-O0", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-I",
                    str(ROOT) + "/casclik_b200/csrc", "-o", str(so), str(src)], check=True)
    return ctypes.CDLL(str(so))


def libraries(ctrl, tmp_path):
    """(JVP image, VJP image) of one controller, both host builds."""
    (tmp_path / "jvp").mkdir(exist_ok=True)
    (tmp_path / "vjp").mkdir(exist_ok=True)
    return jvp_library(ctrl, tmp_path / "jvp"), vjp_library(ctrl, tmp_path / "vjp")


def _split(ctrl, td):
    """theta_dot (n_theta, N) in theta_rows' order -> (t_dot, q_dot, x_dot, y_dot) arrays (None where empty)."""
    nq = ctrl.skill_spec.n_robot_var
    parts = [np.ascontiguousarray(td[0]), np.ascontiguousarray(td[1:1 + nq])]
    parts.append(np.ascontiguousarray(td[1 + nq:1 + nq + ctrl._nxv]) if ctrl._nxv else None)
    parts.append(np.ascontiguousarray(td[1 + nq + ctrl._nxv:]) if ctrl._ny else None)
    return parts


def host_jvp(lib, ctrl, kind, inp, sol, status, active, td, null=()):
    """-> sol_dot (nx, N) for the tangent td (n_theta, N); the parts named in `null` are passed as NULL."""
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    parts = [None if k in null else a for k, a in zip("tqxy", _split(ctrl, td))]
    out = np.full((ctrl._qn, N), -7.0)
    getattr(lib, "clik_%s_jvp_kernel" % kind)(
        ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
        _p(np.ascontiguousarray(sol)), _p(np.ascontiguousarray(status, dtype=np.int32)),
        _p(np.ascontiguousarray(active, dtype=np.uint32)), *[_p(a) for a in parts], _p(out))
    return out


def host_jac(lib, ctrl, kind, inp, sol, status, active):
    """-> jac (nx, n_theta, N)."""
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    nt = len(theta_rows(ctrl, inp)[0])
    out = np.full((ctrl._qn, nt, N), -7.0)
    getattr(lib, "clik_%s_jacobian_kernel" % kind)(
        ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
        _p(np.ascontiguousarray(sol)), _p(np.ascontiguousarray(status, dtype=np.int32)),
        _p(np.ascontiguousarray(active, dtype=np.uint32)), _p(out))
    return out


def tangents(ctrl, inp, seed):
    rows, _ = theta_rows(ctrl, inp)
    return np.random.default_rng(seed).standard_normal((len(rows), inp["q"].shape[1]))


# ---- the adjoint identity and the Jacobian against both ----------------------------------------------------

def check_adjoint(ctrl, kind, libs, inp, seed):
    """<xb, x_dot> = <theta_bar, theta_dot>; jac' xb = the VJP and jac theta_dot = the JVP.  -> solved count."""
    jlib, vlib = libs
    sol, status, active = host_step(jlib, ctrl, kind, inp)
    _, full = theta_rows(ctrl, inp)
    ok = status == 0
    td = tangents(ctrl, inp, seed)
    xb = np.random.default_rng(seed + 100).standard_normal(sol.shape)
    xd = host_jvp(jlib, ctrl, kind, full, sol, status, active, td)
    tb = host_vjp(vlib, ctrl, kind, full, sol, status, active, xb)
    jac = host_jac(jlib, ctrl, kind, full, sol, status, active)
    fin = ok & np.isfinite(xd).all(axis=0)
    assert np.array_equal(fin, ok & np.isfinite(tb).all(axis=0))                # the same NaN rules
    assert np.isnan(xd[:, ~fin]).all() and np.isnan(jac[:, :, ~fin]).all()
    lhs, rhs = np.sum(xb * xd, axis=0)[fin], np.sum(tb * td, axis=0)[fin]
    scale = (np.linalg.norm(xb, axis=0) * np.linalg.norm(xd, axis=0) +
             np.linalg.norm(tb, axis=0) * np.linalg.norm(td, axis=0))[fin]
    gap = np.abs(lhs - rhs) / np.where(scale > 0, scale, 1.0)        # (both sides exactly 0 where scale is)
    _note("adjoint identity", gap.max(initial=0))
    assert gap.max(initial=0) <= 1e-12, gap.max()
    jt = np.einsum("jci,ji->ci", jac, xb)[:, fin]
    jd = np.einsum("jci,ci->ji", jac, td)[:, fin]
    e1 = np.abs(jt - tb[:, fin]).max(axis=0) / (1 + np.abs(tb[:, fin]).max(axis=0))
    e2 = np.abs(jd - xd[:, fin]).max(axis=0) / (1 + np.abs(xd[:, fin]).max(axis=0))
    _note("jacobian' xb vs vjp", e1.max(initial=0))
    _note("jacobian theta_dot vs jvp", e2.max(initial=0))
    assert e1.max(initial=0) <= 1e-12 and e2.max(initial=0) <= 1e-12, (e1.max(), e2.max())
    return int(fin.sum())


@pytest.mark.parametrize("name", QP)
def test_qp_fixtures_adjoint_identity(name, tmp_path):
    spec, inp, kwargs, _ = load_case(name)
    ctrl = cc.ReactiveQPController(spec, **kwargs)
    assert check_adjoint(ctrl, "qp", libraries(ctrl, tmp_path), inp, 1) == inp["q"].shape[1]


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic"])
def test_scenarios_adjoint_identity(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    inp = {k: v for k, v in sc.sample(64, seed=31).items() if v is not None}
    assert check_adjoint(ctrl, "qp" if name.endswith("_qp") else "nlp", libraries(ctrl, tmp_path), inp, 2) >= 60


@pytest.mark.parametrize("seed", list(range(3)) + ["dense0"])
def test_fuzzed_qp_skills_adjoint_identity(seed, tmp_path):
    from fuzz_skills import make_dense_qp_skill, make_qp_skill
    dense = isinstance(seed, str)
    spec, weights, inp = make_dense_qp_skill(int(seed[5:])) if dense else make_qp_skill(seed)
    ctrl = cc.ReactiveQPController(spec, **weights)
    inp = {k: (v[..., :48] if k != "t" else v[:48]) for k, v in inp.items()}
    assert check_adjoint(ctrl, "qp", libraries(ctrl, tmp_path), inp, 3) >= 1


@pytest.mark.parametrize("seed", range(2))
def test_fuzzed_convex_nlp_costs_adjoint_identity(seed, tmp_path):
    from fuzz_skills import make_qp_skill
    spec, _, inp = make_qp_skill(seed)
    ctrl = cc.ReactiveNLPController(spec, random_convex_cost(spec, seed))
    inp = {k: (v[..., :48] if k != "t" else v[:48]) for k, v in inp.items()}
    assert check_adjoint(ctrl, "nlp", libraries(ctrl, tmp_path), inp, 4) >= 1


# ---- independent KKT reference (NumPy: K and dr/dtheta from H, A, lb, ub with central differences) ------------

def kkt_jacobian(spec, inp, rows, sol, active, **w):
    """dx*/dtheta_k from K [x_dot; lam_dot] = -[rho1_k; rho2_k] solved by NumPy per instance -> (nx, n_theta, N)."""
    N = sol.shape[1]

    def mats(i_):
        h, A, lb, ub = oracle_qp_problem(spec, i_, **w)
        return [np.broadcast_to(h, (N, len(h))) if np.ndim(h) == 1 else h, A, lb, ub]
    h, A, lb, ub = mats(inp)
    m, n = A.shape[1], A.shape[2]
    lams, Ws = [], []
    for i in range(N):
        Ws.append([r for r in range(m) if ((int(active[0, i]) | int(active[1, i])) >> r) & 1])
        _, lam, st = orc.solve_qp_single(h[i], A[i], lb[i], ub[i])
        assert st == 0
        lams.append(lam)
    out = np.zeros((n, len(rows), N))
    for k, (key, row) in enumerate(rows):
        val = inp[key] if row is None else inp[key][row]
        hstep = 1e-3 * np.maximum(1.0, np.abs(val))
        d = [mats(perturbed(inp, key, row, sgn * hstep)) for sgn in (1, -1, 2, -2)]
        dh, dA, dlb, dub = [(8 * (a - b) - (c - e)) / (12 * (hstep[:, None, None] if a.ndim == 3 else hstep[:, None]))
                            for a, b, c, e in zip(d[0], d[1], d[2], d[3])]
        for i in range(N):
            W = Ws[i]
            bsel = np.array([dub[i, r] if (int(active[0, i]) >> r) & 1 else dlb[i, r] for r in W])
            rho1 = dh[i] * sol[:, i] + dA[i].T @ lams[i]
            rho2 = dA[i][W] @ sol[:, i] - bsel if W else np.zeros(0)
            AW = A[i][W]
            K = np.block([[np.diag(h[i]), AW.T], [AW, np.zeros((len(W), len(W)))]])
            out[:, k, i] = np.linalg.solve(K, -np.concatenate([rho1, rho2]))[:n]
    return out


def _check_kkt(spec, ctrl, lib, inp, **w):
    sol, status, active = host_step(lib, ctrl, "qp", inp)
    rows, full = theta_rows(ctrl, inp)
    ok = status == 0
    sel = {k: (v[..., ok] if k != "t" else v[ok]) for k, v in full.items()}
    got = host_jac(lib, ctrl, "qp", sel, sol[:, ok], status[ok], active[:, ok])
    ref = kkt_jacobian(spec, sel, rows, sol[:, ok], active[:, ok], **w)
    err = np.abs(got - ref).max(axis=(0, 1)) / (1 + np.abs(got).max(axis=(0, 1)))
    _note("qp jacobian vs kkt", err.max())
    assert err.max() <= 1e-9, (err.max(), int(err.argmax()))
    return int(ok.sum())


@pytest.mark.parametrize("name", QP)
def test_qp_fixtures_match_the_kkt_reference(name, tmp_path):
    spec, inp, kwargs, _ = load_case(name)
    ctrl = cc.ReactiveQPController(spec, **kwargs)
    w = {_W[k]: v for k, v in kwargs.items() if k in _W}
    assert _check_kkt(spec, ctrl, jvp_library(ctrl, tmp_path), inp, **w) == inp["q"].shape[1]


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_benchmark_qp_scenarios_match_the_kkt_reference(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    inp = {k: v for k, v in sc.sample(48, seed=29).items() if v is not None}
    assert _check_kkt(sc.spec, ctrl, jvp_library(ctrl, tmp_path), inp) == 48


# ---- directional finite differences of the step itself ------------------------------------------------------

def fd_direction(lib, ctrl, kind, inp, rel, tol, seed, min_count, stencil=3):
    """(sol(theta + h theta_dot) - sol(theta - h theta_dot)) / 2h against the JVP on the instances whose working set
    is the same at every point of the stencil; the steps and stencils of test_vjp_on_host.fd_check (a random
    direction scaled so that entry k moves by at most rel max(1, |theta_k|))."""
    sol, status, active = host_step(lib, ctrl, kind, inp)
    rows, full = theta_rows(ctrl, inp)
    # direction: each entry of theta moves by at most fd_check's step, rel max(1, |theta_k|)
    theta = np.vstack([full["t"][None]] + [full[k] for k in "qxy" if k in full])
    td = tangents(ctrl, inp, seed)
    td = td / np.abs(td).max(axis=0) * np.maximum(1.0, np.abs(theta))
    got = host_jvp(lib, ctrl, kind, full, sol, status, active, td)
    scale = 1 + np.abs(got).max(axis=0)
    h = rel
    same = status == 0
    f = {}
    for step in ((1, -1) if stencil == 3 else (1, -1, 2, -2, 0.01, -0.01, 0.001, -0.001)):
        moved = {k: v.copy() for k, v in full.items()}
        for c, (key, row) in enumerate(rows):
            if row is None:
                moved[key] = moved[key] + step * h * td[c]
            else:
                moved[key][row] = moved[key][row] + step * h * td[c]
        sp, stp, ap = host_step(lib, ctrl, kind, moved)
        same &= (stp == 0) & np.all(ap == active, axis=0)
        f[step] = sp
    if stencil == 3:
        err = np.abs((f[1] - f[-1]) / (2 * h) - got).max(axis=0) / scale
        ok = err <= tol
    else:
        err = np.abs((8 * (f[1] - f[-1]) - (f[2] - f[-2])) / (12 * h) - got).max(axis=0) / scale
        ok = err <= tol
        for r in (0.01, 0.001):
            ok |= np.abs((f[r] - f[-r]) / (2 * r * h) - got).max(axis=0) / scale <= tol
    if same.any():
        _note("%s_fd" % kind, err[same].max())
    bad = np.where(same & ~ok)[0]
    assert bad.size == 0, (bad[:5], err[bad[:5]])
    assert int(same.sum()) >= min_count, int(same.sum())


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_qp_scenarios_match_directional_finite_differences(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    inp = {k: v for k, v in sc.sample(128, seed=5).items() if v is not None}
    fd_direction(jvp_library(ctrl, tmp_path), ctrl, "qp", inp, 1e-6, 1e-6, 7, 64)


@pytest.mark.parametrize("name", sorted(scenarios.NLP_REGISTRY))
def test_nlp_scenarios_match_directional_finite_differences(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    inp = {k: v for k, v in sc.sample(48, seed=6).items() if v is not None}
    fd_direction(jvp_library(ctrl, tmp_path), ctrl, "nlp", inp, 1e-4, 1e-4, 9, 24, stencil=5)


# ---- known answers (SURVEY.md §8c, cart point_skill, theta = p) --------------------------------------------

def test_cart_known_answers(tmp_path):
    t, p, dp = cs.MX.sym("t"), cs.MX.sym("p"), cs.MX.sym("dp")
    eq = cc.EqualityConstraint("min_dist_cnstr", 0.75 - p, gain=1.0, constraint_type="soft", priority=1)
    lim = cc.SetConstraint("cart_limit_cnstr", p, gain=1.0, set_min=0.0, set_max=1.0)
    spd = cc.VelocitySetConstraint("speed_limit_cnstr", p, gain=10.0, set_min=-0.275, set_max=0.275)
    spec = cc.SkillSpecification("cart_qp", t, p, robot_vel_var=dp, constraints=[eq, lim, spd])
    ctrl = cc.ReactiveQPController(spec, robot_var_weights=[1.0])
    lib = jvp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(2), "q": np.array([[0.0, 0.6]])}
    sol, status, active = host_step(lib, ctrl, "qp", inp)
    assert np.all(status == 0)
    jac = host_jac(lib, ctrl, "qp", inp, sol, status, active)
    want = np.array([[0.0, -1.0], [-1.001 / 1.002, -0.001 / 1.002]])          # (dpdot/dp, deps/dp) of Q1, Q2
    assert np.abs(jac[:, 1, :].T - want).max() <= 1e-12, jac[:, 1, :].T - want
    assert np.all(jac[:, 0, :] == 0.0)                                         # nothing depends on t
    xd = host_jvp(lib, ctrl, "qp", inp, sol, status, active, np.array([[0.0, 0.0], [1.0, 1.0]]), null="t")
    assert np.abs(xd.T - want).max() <= 1e-12


# ---- 50-digit face derivative ------------------------------------------------------------------------------

def check_face_reference(name, kind, ctrl, jlib, vlib, inp, both_bits=False):
    """The Jacobian of every instance against mp_reference.face_derivative, read through a random cotangent xb:
    xb' jac against xb' D within the bound of the VJP (mr.vjp_bound(kappa, scale) plus what the kernel's own x* and
    lam carry into the face residual, the criterion of test_face_reference_on_host.check_outputs; the Jacobian is
    the adjoint of that VJP, K being symmetric, so its rounding enters through the same factorisation) and jac
    entrywise within C u kappa (1 + |D|_max) + that carried error; NaN exactly where the VJP gives NaN, and the VJP's
    NaN bands."""
    sol, status, active = host_step(jlib, ctrl, kind, inp)
    if both_bits:
        _, lb, ub = constraint_rows(program(kind, ctrl), inp)
        eq = ((lb == ub) * (1 << np.arange(lb.shape[1]))).sum(axis=1).astype(np.uint32)
        held = (active[0] | active[1]) & eq
        assert held.any()
        active = np.ascontiguousarray(np.stack([active[0] | held, active[1] | held]))
    rows, full = theta_rows(ctrl, inp)
    prog = program(kind, ctrl)
    sids = mr.theta_symbols(prog, rows)
    jac = host_jac(jlib, ctrl, kind, full, sol, status, active)
    xb = np.random.default_rng(3).standard_normal(sol.shape)
    tb = host_vjp(vlib, ctrl, kind, full, sol, status, active, xb)
    assert np.array_equal(np.isnan(jac).any(axis=(0, 1)), np.isnan(tb).any(axis=0)), name
    checked = 0
    for i in range(sol.shape[1]):
        if status[i] != 0:
            assert np.isnan(jac[:, :, i]).all()
            continue
        up, lo = int(active[0, i]), int(active[1, i])
        P = mr.mp_problem(prog, inp, i)
        f = mr.face_solve(P, up, lo, sol[:, i])
        nan_band(np.isnan(jac[:, :, i]).any(), f, kind, (name, i))
        if np.isnan(jac[:, :, i]).any() or f["xm"] is None or f["kappa"] * mr.U >= mr.CLAIM:
            continue
        D = mr.face_derivative(P, up, lo, f["xm"], sids)
        Df = np.array([[float(v) for v in r] for r in D])
        ref, scale = mr.vjp_adjoint(P, up, lo, f["xm"], f["lamW"], xb[:, i], sids)
        _, lam_k, _, _ = mr.ls_multipliers(P, up, lo, sol[:, i])
        carried = 0.0
        if lam_k is not None:
            at_k, _ = mr.vjp_adjoint(P, up, lo, sol[:, i], lam_k, xb[:, i], sids)
            carried = np.abs(np.array([float(v) for v in at_k]) - np.array([float(v) for v in ref]))
        with mr.mp.workdps(mr.DDPS):
            proj = np.array([float(sum(mr.mp.mpf(float(xb[j, i])) * D[j, c] for j in range(prog.nx)))
                             for c in range(len(sids))])
        got = xb[:, i] @ jac[:, :, i]
        r1 = np.abs(got - proj) / (mr.vjp_bound(f["kappa"], scale) + carried)
        _note("%s jacobian' xb vs face derivative %s" % (kind, name), r1.max())
        assert r1.max() <= 1.0, (name, i, "xb' jac error / bound", r1.max(), f["kappa"])
        bound = mr.C * mr.U * f["kappa"] * (1 + np.abs(Df).max()) + mr.ATOL + np.max(carried)
        r2 = np.abs(jac[:, :, i] - Df).max() / bound
        _note("%s jacobian vs face derivative %s" % (kind, name), r2)
        assert r2 <= 1.0, (name, i, "jacobian error / bound", r2, f["kappa"])
        checked += 1
    return checked


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic"])
def test_jacobian_near_singularities_against_the_face_derivative(name, tmp_path):
    kind, sc, ctrl, vlib = case(name, tmp_path)
    (tmp_path / "jvp_lib_dir").mkdir()
    jlib = jvp_library(ctrl, tmp_path / "jvp_lib_dir")
    inp, _ = family_sub(sc, 37)
    assert check_face_reference(name, kind, ctrl, jlib, vlib, inp) >= 1
    smp = {k: v for k, v in sc.sample(4, seed=17).items() if v is not None}
    assert check_face_reference(name + " sampler", kind, ctrl, jlib, vlib, smp) == 4


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_taskspeed"])
def test_equality_rows_held_at_both_bits(name, tmp_path):
    """Equality rows handed over with both mask bits use ub, as the VJP: the same face, the same Jacobian."""
    kind, sc, ctrl, vlib = case(name, tmp_path)
    (tmp_path / "jvp_lib_dir").mkdir()
    jlib = jvp_library(ctrl, tmp_path / "jvp_lib_dir")
    inp, _ = family_sub(sc, 53)
    check_face_reference(name + " both bits", kind, ctrl, jlib, vlib, inp, both_bits=True)
    sol, status, active = host_step(jlib, ctrl, kind, inp)
    _, lb, ub = constraint_rows(program(kind, ctrl), inp)
    eq = ((lb == ub) * (1 << np.arange(lb.shape[1]))).sum(axis=1).astype(np.uint32)
    held = (active[0] | active[1]) & eq
    both = np.ascontiguousarray(np.stack([active[0] | held, active[1] | held]))
    _, full = theta_rows(ctrl, inp)
    one = host_jac(jlib, ctrl, kind, full, sol, status, active)
    two = host_jac(jlib, ctrl, kind, full, sol, status, both)
    ok = np.isfinite(one).all(axis=(0, 1))
    assert ok.sum() >= 1 and np.array_equal(ok, np.isfinite(two).all(axis=(0, 1)))
    err = np.abs(one - two)[:, :, ok].max(axis=(0, 1)) / (1 + np.abs(one[:, :, ok]).max(axis=(0, 1)))
    assert err.max() <= 1e-12, err.max()


# ---- NaN and zero rules ------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_unsolved_instances_nan_unless_the_tangent_is_zero(kind, tmp_path):
    sc = scenarios.get("ur5_qp" if kind == "qp" else "ur5_nlp_quartic")
    ctrl = sc.make_controller()
    lib = jvp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(8, seed=3).items() if v is not None}
    inp["q"][1, 5] = np.nan                                       # invalid (4)
    sol, status, active = host_step(lib, ctrl, kind, inp)
    assert status[5] == 4
    status[2] = 2                                                 # as an infeasible instance reports it
    _, full = theta_rows(ctrl, inp)
    td = tangents(ctrl, inp, 12)
    td[:, [3, 5]] = 0.0                                           # solved / unsolved with a zero tangent
    g = host_jvp(lib, ctrl, kind, full, sol, status, active, td)
    assert np.isnan(g[:, 2]).all()
    assert np.all(g[:, 3] == 0.0) and np.all(g[:, 5] == 0.0)
    z = host_jvp(lib, ctrl, kind, full, sol, status, active, td, null="tqxy")  # every tangent NULL
    assert np.all(z == 0.0)
    td[:, 5] = 1.0
    g = host_jvp(lib, ctrl, kind, full, sol, status, active, td)
    assert np.isnan(g[:, 5]).all()
    assert not np.isnan(np.delete(g, [2, 5], axis=1)).any()
    jac = host_jac(lib, ctrl, kind, full, sol, status, active)
    assert np.isnan(jac[:, :, [2, 5]]).all() and not np.isnan(np.delete(jac, [2, 5], axis=2)).any()
    # columns of theta entries the program does not read are exactly 0 (the ur5 scenarios do not read t)
    from casclik_b200.codegen.jvp import JacProgram
    jp = JacProgram(program(kind, ctrl), kind)
    unread = [c for c in range(jp.n_theta) if all(r[c] is mr.dag.ZERO for r in jp.r1 + jp.r2u + jp.r2l)]
    assert unread and np.all(np.delete(jac, [2, 5], axis=2)[:, unread] == 0.0)


def test_rank_deficient_working_set_gives_nan(tmp_path):
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    cons = [cc.VelocityEqualityConstraint("a", q[0] + q[1], target=0.5),
            cc.VelocitySetConstraint("b", 2.0 * (q[0] + q[1]), set_min=-5.0, set_max=5.0, priority=1)]
    spec = cc.SkillSpecification("dup", t, q, robot_vel_var=dq, constraints=cons)
    ctrl = cc.ReactiveQPController(spec)
    lib = jvp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(2), "q": np.zeros((2, 2))}
    sol, status, active = host_step(lib, ctrl, "qp", inp)
    assert np.all(status == 0)
    active[0, 1] |= 3
    g = host_jvp(lib, ctrl, "qp", inp, sol, status, active, np.ones((3, 2)))
    assert np.isnan(g[:, 1]).all() and not np.isnan(g[:, 0]).any()
    jac = host_jac(lib, ctrl, "qp", inp, sol, status, active)
    assert np.isnan(jac[:, :, 1]).all() and not np.isnan(jac[:, :, 0]).any()


def test_singular_hessian_gives_nan(tmp_path):
    """|J_p dq|^2 for a task point off the tool axis: the Hessian is singular without a zero row, its trailing
    Cholesky pivots rounding noise (the case of test_face_reference_on_host.test_nlp_singular_hessian...)."""
    kind, sc, ctrl, vlib = case("offaxis_eps_0", tmp_path)
    (tmp_path / "jvp_lib_dir").mkdir()
    jlib = jvp_library(ctrl, tmp_path / "jvp_lib_dir")
    inp = {k: v for k, v in sc.sample(16, seed=8).items() if v is not None}
    sol, status, active = host_step(jlib, ctrl, kind, inp)
    solved = status == 0
    assert solved.any()
    _, full = theta_rows(ctrl, inp)
    td = tangents(ctrl, inp, 9)
    xd = host_jvp(jlib, ctrl, kind, full, sol, status, active, td)
    jac = host_jac(jlib, ctrl, kind, full, sol, status, active)
    tb = host_vjp(vlib, ctrl, kind, full, sol, status, active, np.ones_like(sol))
    assert np.isnan(tb[:, solved]).all()                           # the VJP's rule on these instances
    assert np.isnan(xd[:, solved]).all() and np.isnan(jac[:, :, solved]).all()


# ---- emitted source and loading ----------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_quartic", "ur5_nlp_taskspeed"])
def test_jvp_source_is_the_default_source_plus_one_section(name, tmp_path):
    """The JVP image a controller builds on demand holds its default image unchanged; the default and VJP sources
    do not change with the JVP's emission."""
    ctrl = scenarios.get(name).make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    src0, meta0 = ctrl.kernel_source, ctrl.kernel_meta
    src1, meta1 = ctrl._jvp_source()
    assert not meta0["jvp"] and meta1["jvp"] and "jvp" not in src0 and "jacobian" not in src0
    head, sep, tail = src1.partition("\n\n// ---- forward-mode derivative of the step's output (clik_jvp.cuh) ----\n")
    assert sep and tail.count("__global__") == 2 and "_jvp_kernel(" in tail and "_jacobian_kernel(" in tail
    lines = (head + "\n").split("\n")
    o20 = [ln for ln in lines if ln.lstrip().startswith("o[20] = ")]
    assert o20 == ["  o[20] = %d;   // JVP and Jacobian kernels (1 QP, 2 NLP)" % (2 if "nlp" in name else 1)]
    lines.remove(o20[0])
    assert "\n".join(lines) == src0
    assert meta1["jvp_eval"]["flops"] > 0 and meta1["jac_eval"]["flops"] > 0
    vsrc, _ = ctrl._vjp_source()
    assert "jvp" not in vsrc and "o[20]" not in vsrc


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_more_than_32_rows_raise_and_build_no_kernel(kind, tmp_path, monkeypatch):
    ctrl = _ctrl(kind, _wide_spec(33))
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._jvp_source()
    assert not meta["jvp"] and "jvp_kernel" not in source and "o[20]" not in source
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no JVP image may be built"))
    N = 4
    for call in (lambda: ctrl.jvp_batch(np.zeros(N), np.zeros((3, N)), None, None, np.zeros((3, N)),
                                        np.zeros(N, np.int32), np.zeros((2, N), np.int32), q_dot=np.ones((3, N))),
                 lambda: ctrl.jacobian_batch(np.zeros(N), np.zeros((3, N)), None, None, np.zeros((3, N)),
                                             np.zeros(N, np.int32), np.zeros((2, N), np.int32))):
        with pytest.raises(ValueError, match="at most 32 constraint rows"):
            call()
    assert ctrl._jvp is None


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_numpy_inputs_raise_without_building_the_image(name, tmp_path, monkeypatch):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no JVP image may be built"))
    inp = sc.sample(4, seed=1)
    N = 4
    args = (inp["t"], inp["q"], None, inp["y"], np.zeros((ctrl._qn, N)), np.zeros(N, np.int32),
            np.zeros((2, N), np.int32))
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.jvp_batch(*args, q_dot=np.ones((6, N)))
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.jacobian_batch(*args)
    assert ctrl._jvp is None


def test_abi_rejects_a_null_skill():
    from casclik_b200 import runtime
    lib = runtime.load_library()
    for name in ("clik_qp_jvp", "clik_nlp_jvp"):
        assert getattr(lib, name)(None, 4, None, 0, *([None] * 12)) == 1
        assert b"skill is NULL" in lib.clik_last_error()
    for name in ("clik_qp_jacobian", "clik_nlp_jacobian"):
        assert getattr(lib, name)(None, 4, None, 0, *([None] * 8)) == 1
        assert b"skill is NULL" in lib.clik_last_error()


def test_report_observed_maxima():
    """Runs last in this module: the largest relative deviations and error/bound ratios of the checks above."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items())})
