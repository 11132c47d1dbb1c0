"""Reverse-mode derivative of the QP and NLP closed-loop rollouts (csrc/clik_rollout_vjp.cuh,
clik_<kind>_rollout_tape_kernel / clik_<kind>_rollout_vjp_kernel): the emitted rollout-VJP image built for the HOST
with g++ (the harness of test_rollout_jvp_on_host.py), against the primal rollout kernel, a host loop of the step and
step-VJP kernels of the same image, the tangent and Jacobian rollouts of the rollout-JVP image (the adjoint
identity), finite differences, known answers and the rules of include/clik.h."""
import ctypes
import subprocess

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import build, cs, scenarios
from test_golden_controllers import load_case
from test_kernel_code_on_host import ROOT, SHIM, _p
from test_rollout_jvp_on_host import (Run, _cart, _tracking, composed, host_rollout, host_rollout_jac,
                                      host_rollout_jvp, host_step_warm, kind_of, rel, rollout_library)
from test_vjp_api import _ctrl, _setup_without_nvcc, _wide_spec
from test_vjp_on_host import _full_inputs, host_vjp, theta_rows

OBSERVED = {}
SCENARIOS = ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic"]
FIXTURES = ["qp/ur5_qp", "qp/ur5_moe2016", "qp/cart_path", "qp/kitchen_sink"]


def _note(key, v):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(v))


def rollout_vjp_library(ctrl, tmp_path):
    """setup_problem_functions without nvcc, then the rollout-VJP image's source built with g++."""
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._rollout_vjp_source()
    assert meta["rollout_vjp"]
    text = source.replace("__device__ const unsigned short", "static const unsigned short")
    src = tmp_path / "skill_rollout_vjp.cpp"
    src.write_text(SHIM + text)
    so = tmp_path / "skill_rollout_vjp.so"
    subprocess.run(["g++", "-O0", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-I",
                    str(ROOT) + "/casclik_b200/csrc", "-o", str(so), str(src)], check=True)
    return ctypes.CDLL(str(so))


def libraries(ctrl, tmp_path):
    """(rollout-VJP image, rollout-JVP image) of one controller, both host builds."""
    (tmp_path / "vjp").mkdir(exist_ok=True)
    (tmp_path / "jvp").mkdir(exist_ok=True)
    return rollout_vjp_library(ctrl, tmp_path / "vjp"), rollout_library(ctrl, tmp_path / "jvp")


def host_tape(lib, ctrl, inp, run):
    """clik_<kind>_rollout_tape_kernel -> (q, x, sol, n_failed, tape) with the tape's step-major blocks."""
    q, x, sol, failed, args = run.head(ctrl, inp)
    N, K = q.shape[1], run.steps
    tape = {"q": np.full((K, q.shape[0], N), -7.0), "x": np.full((K, ctrl._nxv, N), -7.0) if ctrl._nxv else None,
            "sol": np.full((K, ctrl._qn, N), -7.0), "status": np.full((K, N), -9, dtype=np.int32),
            "active": np.full((K, 2, N), 7, dtype=np.uint32)}
    getattr(lib, "clik_%s_rollout_tape_kernel" % kind_of(ctrl))(
        *args, *[_p(tape[k]) for k in ("q", "x", "sol", "status", "active")])
    return q, x, sol, failed, tape


def host_sweep(lib, ctrl, inp, run, tape, cq=None, cx=None, cs_=None):
    """clik_<kind>_rollout_vjp_kernel over `tape` along the cotangents (q_bar_K, x_bar_K, sol_bar) -> p_bar
    (n_theta, N) in theta_rows' order."""
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    tb, qb = np.full(N, -7.0), np.full((q.shape[0], N), -7.0)
    xb = np.full((ctrl._nxv, N), -7.0) if ctrl._nxv else None
    yb = np.full((ctrl._ny, N), -7.0) if ctrl._ny else None
    c = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)  # noqa: E731
    cq, cx, cs_ = c(cq), c(cx), c(cs_)
    keep = [None if a is None else a.copy() for a in (cq, cx, cs_)]
    getattr(lib, "clik_%s_rollout_vjp_kernel" % kind_of(ctrl))(
        ctypes.c_longlong(N), ctypes.c_longlong(N), ctypes.c_int(run.steps), ctypes.c_double(run.dt), _p(t),
        ctypes.c_int(1), _p(y), ctypes.c_double(run.vq), ctypes.c_double(run.vx),
        *[_p(tape[k]) for k in ("q", "x", "sol", "status", "active")], _p(cq), _p(cx), _p(cs_), _p(tb), _p(qb),
        _p(xb), _p(yb))
    assert all(a is None or np.array_equal(a, k) for a, k in zip((cq, cx, cs_), keep))     # inputs only
    return np.vstack([tb[None]] + [a for a in (qb, xb, yb) if a is not None])


def composed_tape(lib, ctrl, inp, run):
    """The tape as a host loop of the warm-started step kernel (composed() of the rollout-JVP tests, recording)."""
    rows, full = theta_rows(ctrl, inp)
    nq, nxv, N = ctrl.skill_spec.n_robot_var, ctrl._nxv, full["q"].shape[1]
    ns = nq + nxv
    state = {k: v.copy() for k, v in full.items()}
    t0 = full["t"].copy()
    warm = np.zeros((2, N), dtype=np.uint32) if kind_of(ctrl) == "qp" else np.zeros((ctrl._qn, N))
    vmax = np.array([run.vq] * nq + [run.vx] * nxv)[:, None]
    out = {"q": [], "x": [], "sol": [], "status": [], "active": []}
    for k in range(run.steps):
        state["t"] = t0 + run.dt * float(k)
        out["q"].append(state["q"].copy())
        if nxv:
            out["x"].append(state["x"].copy())
        sol, status, active = host_step_warm(lib, ctrl, state, warm)
        for key, a in (("sol", sol), ("status", status), ("active", active)):
            out[key].append(a.copy())
        v = np.where(status == 0, sol, 0.0)
        warm = active if kind_of(ctrl) == "qp" else v
        state["q"] = state["q"] + np.clip(v[:nq], -vmax[:nq], vmax[:nq]) * run.dt
        if nxv:
            state["x"] = state["x"] + np.clip(v[nq:ns], -vmax[nq:], vmax[nq:]) * run.dt
    return {k: (np.array(v) if v else None) for k, v in out.items()}


def composed_sweep(lib, ctrl, inp, run, tape, cq=None, cx=None, cs_=None):
    """The sweep as a host loop of the step VJP kernel over the tape slices, with the clip mask and the accumulation
    in NumPy (the order of the sweep kernel)."""
    rows, full = theta_rows(ctrl, inp)
    nq, nxv, N = ctrl.skill_spec.n_robot_var, ctrl._nxv, full["q"].shape[1]
    ns = nq + nxv
    vmax = np.array([run.vq] * nq + [run.vx] * nxv)[:, None]
    aq = np.zeros((nq, N)) if cq is None else cq.copy()
    ax = (np.zeros((nxv, N)) if cx is None else cx.copy()) if nxv else np.zeros((0, N))
    tb, yb = np.zeros(N), np.zeros((ctrl._ny, N))
    for k in range(run.steps - 1, -1, -1):
        sb = np.zeros((ctrl._qn, N))
        sb[:ns] = run.dt * np.vstack([aq, ax])
        if k == run.steps - 1 and cs_ is not None:
            sb = sb + cs_
        sol = tape["sol"][k]
        sb[:ns] = np.where(np.abs(sol[:ns]) < vmax, sb[:ns], 0.0)
        state = {"t": full["t"] + run.dt * float(k), "q": tape["q"][k]}
        if nxv:
            state["x"] = tape["x"][k]
        if ctrl._ny:
            state["y"] = full["y"]
        th = host_vjp(lib, ctrl, kind_of(ctrl), state, sol, tape["status"][k], tape["active"][k], sb)
        tb = tb + th[0]
        aq = aq + th[1:1 + nq]
        ax = ax + th[1 + nq:1 + ns]
        yb = yb + th[1 + ns:]
    return np.vstack([tb[None], aq, ax, yb])


def cotangents(ctrl, N, seed):
    r = np.random.default_rng(seed)
    nq = ctrl.skill_spec.n_robot_var
    return r.standard_normal((nq, N)), (r.standard_normal((ctrl._nxv, N)) if ctrl._nxv else None), \
        r.standard_normal((ctrl._qn, N))


def nan_cols(a):
    return np.isnan(a).any(axis=0)


def _speed_limit(ctrl, inp, lib, frac):
    N = inp["q"].shape[1]
    sol, _, _ = host_step_warm(lib, ctrl, theta_rows(ctrl, inp)[1], np.zeros((2, N), np.uint32)
                               if kind_of(ctrl) == "qp" else np.zeros((ctrl._qn, N)))
    return frac * float(np.nanmax(np.abs(sol[:ctrl.skill_spec.n_robot_var])))


# ---- tape, sweep, composed loop and the adjoint identity ---------------------------------------------------

def check_rollout_vjp(ctrl, libs, inp, run, seed, name):
    """Primal and tape bit for bit; the sweep against the composed step-VJP loop; the adjoint identity against
    rollout_jvp and unit cotangents against rollout_jacobian.  -> the number of finite instances."""
    vlib, jlib = libs
    _, full = theta_rows(ctrl, inp)
    N = full["q"].shape[1]
    prim = host_rollout(vlib, ctrl, full, run)
    q, x, sol, failed, tape = host_tape(vlib, ctrl, full, run)
    for g, w in zip((q, x, sol, failed), prim):
        if g is not None:
            assert np.array_equal(g, w)
    ref = composed_tape(vlib, ctrl, full, run)
    for key in ("q", "x", "sol", "status", "active"):
        if tape[key] is not None:
            assert np.array_equal(tape[key], ref[key]), key
    cq, cx, csol = cotangents(ctrl, N, seed)
    pb = host_sweep(vlib, ctrl, full, run, tape, cq, cx, csol)
    want = composed_sweep(vlib, ctrl, full, run, tape, cq, cx, csol)
    bad = nan_cols(pb)
    assert np.array_equal(bad, nan_cols(want)) and np.isnan(pb[:, bad]).all()
    e = rel(pb[:, ~bad], want[:, ~bad]).max(initial=0)
    _note("sweep vs composed %s" % name, e)
    assert np.array_equal(pb[:, ~bad], want[:, ~bad]), e
    # adjoint identity against the tangent rollout
    td = np.random.default_rng(seed + 100).standard_normal(pb.shape)
    _, _, _, _, qd, xd, sd = host_rollout_jvp(jlib, ctrl, full, run, td)
    lhs = (cq * qd).sum(axis=0) + (csol * sd).sum(axis=0) + ((cx * xd).sum(axis=0) if cx is not None else 0.0)
    rhs = (pb * td).sum(axis=0)
    ndot = lambda *a: np.sqrt(sum((b ** 2).sum(axis=0) for b in a if b is not None))  # noqa: E731
    scale = ndot(cq, cx, csol) * ndot(qd, xd, sd) + ndot(pb) * ndot(td)
    ok = ~bad & np.isfinite(lhs) & np.isfinite(rhs)
    e = (np.abs(lhs - rhs)[ok] / scale[ok]).max(initial=0)
    _note("adjoint identity %s" % name, e)
    assert e <= 1e-12, e
    # unit cotangents: the rows of the Jacobian rollout
    jac = host_rollout_jac(jlib, ctrl, full, run)[4]
    nq, ns = ctrl.skill_spec.n_robot_var, ctrl.skill_spec.n_robot_var + ctrl._nxv
    for s in range(ns):
        uq, ux = np.zeros((nq, N)), (np.zeros((ctrl._nxv, N)) if ctrl._nxv else None)
        (uq if s < nq else ux)[s if s < nq else s - nq] = 1.0
        row = host_sweep(vlib, ctrl, full, run, tape, uq, ux, None)
        fin = ~nan_cols(row) & ~np.isnan(jac[s]).any(axis=0)
        e = rel(row[:, fin], jac[s][:, fin]).max(initial=0)
        _note("unit cotangent vs jacobian row %s" % name, e)
        assert e <= 1e-13, (s, e)
    return int(ok.sum())


@pytest.mark.parametrize("name", FIXTURES)
def test_qp_fixtures_tape_sweep_and_adjoint(name, tmp_path):
    spec, inp, kwargs, _ = load_case(name)
    ctrl = cc.ReactiveQPController(spec, **kwargs)
    libs = libraries(ctrl, tmp_path)
    vq = _speed_limit(ctrl, inp, libs[0], 0.5)
    run = Run(25, 0.01, vq, 0.5 * vq)
    assert check_rollout_vjp(ctrl, libs, inp, run, 1, name) >= 0.9 * inp["q"].shape[1]
    trace = composed(libs[0], ctrl, theta_rows(ctrl, inp)[1], run)["trace"]
    assert any((~keep).any() for _, _, keep in trace)        # the clip holds on some step


@pytest.mark.parametrize("name", SCENARIOS)
def test_scenarios_tape_sweep_and_adjoint(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    libs = libraries(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(24, seed=41).items() if v is not None}
    vq = _speed_limit(ctrl, inp, libs[0], 0.7)
    run = Run(25, 0.008, vq, vq)
    assert check_rollout_vjp(ctrl, libs, inp, run, 2, name) >= 20
    trace = composed(libs[0], ctrl, theta_rows(ctrl, inp)[1], run)["trace"]
    assert any((~keep).any() for _, _, keep in trace)


# ---- finite differences ------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENARIOS)
def test_scenarios_match_finite_differences_of_a_scalar_functional(name, tmp_path):
    """L = <c_q, q_K> + <c_s, sol>: (L(p + h d) - L(p - h d)) / 2h against <p_bar, d>, on the instances whose +-h
    rollouts keep the working-set and clip sequence of the rollout at p."""
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = rollout_vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(32, seed=43).items() if v is not None}
    rows, full = theta_rows(ctrl, inp)
    N = full["q"].shape[1]
    run = Run(25, 0.008, _speed_limit(ctrl, inp, lib, 0.7), np.inf)
    cq, _, csol = cotangents(ctrl, N, 45)
    pb = host_sweep(lib, ctrl, full, run, host_tape(lib, ctrl, full, run)[4], cq, None, csol)
    theta = np.vstack([full["t"][None]] + [full[k] for k in "qxy" if k in full])
    d = np.random.default_rng(44).standard_normal(theta.shape)
    d = d / np.abs(d).max(axis=0) * np.maximum(1.0, np.abs(theta))
    base = composed(lib, ctrl, full, run)["trace"]
    h = 1e-6
    same = np.ones(N, dtype=bool)
    L = {}
    for sgn in (1, -1):
        moved = {k: v.copy() for k, v in full.items()}
        for c, (key, row) in enumerate(rows):
            if row is None:
                moved[key] = moved[key] + sgn * h * d[c]
            else:
                moved[key][row] = moved[key][row] + sgn * h * d[c]
        for (s0, a0, k0), (s1, a1, k1) in zip(base, composed(lib, ctrl, moved, run)["trace"]):
            same &= (s0 == 0) & (s1 == 0) & np.all(a0 == a1, axis=0) & np.all(k0 == k1, axis=0)
        q, _, sol, _ = host_rollout(lib, ctrl, moved, run)
        L[sgn] = (cq * q).sum(axis=0) + (csol * sol).sum(axis=0)
    fd = (L[1] - L[-1]) / (2 * h)
    got = (pb * d).sum(axis=0)
    err = np.abs(fd - got) / (1 + np.abs(got))
    _note("finite differences %s" % name, err[same].max(initial=0))
    assert same.mean() >= 0.9, same.mean()
    assert err[same].max() <= 1e-6, err[same].max()


# ---- known answers -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_hard_tracking_known_answers(kind, tmp_path):
    """p_dot = -k (p - a sin wt) + a w cos wt with q_bar_K = 1: q_bar_0 = prod of (1 - k dt), factor 1 where the clip
    holds, and t_bar_0 from the scalar recursion."""
    kg, a, w, dt, K = 2.0, 0.4, 3.0, 0.02, 25
    ctrl = _tracking(kind, kg, a, w)
    lib = rollout_vjp_library(ctrl, tmp_path)
    p0 = np.array([[-1.0, -0.3, 0.0, 0.2, 0.9, 2.0]])
    t0 = np.array([0.0, 0.1, 0.5, 1.0, 1.5, 0.3])
    inp = {"t": t0, "q": p0}
    for vmax in (np.inf, 0.8):
        run = Run(K, dt, vmax)
        _, _, _, failed, tape = host_tape(lib, ctrl, inp, run)
        assert np.all(failed == 0)
        pb = host_sweep(lib, ctrl, inp, run, tape, np.ones((1, 6)))
        p, dp0, dt0 = p0[0].copy(), np.ones(6), np.zeros(6)
        clipped = np.zeros(6, dtype=bool)
        for k in range(K):
            tk = t0 + dt * k
            v = -kg * (p - a * np.sin(w * tk)) + a * w * np.cos(w * tk)
            hold = np.abs(v) >= vmax
            clipped |= hold
            fac = np.where(hold, 1.0, 1.0 - kg * dt)
            force = np.where(hold, 0.0, dt * (kg * a * w * np.cos(w * tk) - a * w * w * np.sin(w * tk)))
            dp0 = fac * dp0
            dt0 = fac * dt0 + force
            p = p + np.clip(v, -vmax, vmax) * dt
        if vmax == np.inf:
            assert np.abs(dp0 - (1 - kg * dt) ** K).max() <= 1e-15
        else:
            assert clipped.any()
        for got, want in ((pb[1], dp0), (pb[0], dt0)):
            e = np.abs(got - want).max() / (1 + np.abs(want).max())
            _note("hard tracking %s vmax %s" % (kind, vmax), e)
            assert e <= 1e-12, (vmax, got - want)


def test_cart_known_answers(tmp_path):
    """SURVEY.md §8c cart: the factor of q_bar per step is 1 - dt 1.001/1.002 on the soft row, 1 on the speed row;
    nothing depends on t."""
    ctrl = _cart()
    lib = rollout_vjp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(6), "q": np.array([[0.0, 0.2, 0.5, 0.6, 0.9, 1.0]])}
    run = Run(25, 0.05)
    _, _, _, failed, tape = host_tape(lib, ctrl, inp, run)
    assert np.all(failed == 0)
    pb = host_sweep(lib, ctrl, inp, run, tape, np.ones((1, 6)))
    at_speed = np.abs(np.abs(tape["sol"][:, 0]) - 0.275) <= 1e-12
    assert 0 < at_speed.sum() < at_speed.size
    want = np.prod(np.where(at_speed, 1.0, 1.0 - run.dt * 1.001 / 1.002), axis=0)
    assert np.abs(pb[1] - want).max() <= 1e-12, pb[1] - want
    assert np.all(pb[0] == 0.0)


# ---- rules -------------------------------------------------------------------------------------------------

def test_zero_cotangents_and_failed_steps(tmp_path):
    ctrl = _cart()
    lib = rollout_vjp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(4), "q": np.array([[0.5, 1.6, 0.5, 1.6]])}    # 1.6: outside the feasible band
    run = Run(10, 0.05)
    _, _, _, failed, tape = host_tape(lib, ctrl, inp, run)
    assert failed[0] == 0 and failed[1] > 0 and np.any(tape["status"][:, 1] != 0)
    pb = host_sweep(lib, ctrl, inp, run, tape, np.array([[1.0, 1.0, 0.0, 0.0]]))
    assert np.isfinite(pb[:, 0]).all() and np.isnan(pb[:, 1]).all()
    assert np.all(pb[:, 2:] == 0.0)                                   # zero cotangents give exactly 0
    assert np.all(host_sweep(lib, ctrl, inp, run, tape) == 0.0)        # NULL cotangents too
    sb = np.zeros((ctrl._qn, 4))
    sb[0, 1] = 1.0
    pb = host_sweep(lib, ctrl, inp, run, tape, None, None, sb)
    assert np.isnan(pb[:, 1]).all() and np.all(pb[:, [0, 2, 3]] == 0.0)


def test_steps_zero(tmp_path):
    sc = scenarios.get("ur5_qp")
    ctrl = sc.make_controller()
    lib = rollout_vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(8, seed=2).items() if v is not None}
    _, full = theta_rows(ctrl, inp)
    run = Run(0, 0.01)
    q, _, sol, failed, tape = host_tape(lib, ctrl, full, run)
    assert np.array_equal(q, full["q"]) and np.all(sol == 0.0) and np.all(failed == 0)
    cq, _, csol = cotangents(ctrl, 8, 3)
    pb = host_sweep(lib, ctrl, full, run, {k: None for k in tape}, cq, None, csol)
    assert np.array_equal(pb[1:7], cq) and np.all(pb[0] == 0.0) and np.all(pb[7:] == 0.0)


def test_rank_deficient_working_set_gives_nan(tmp_path):
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    cons = [cc.VelocityEqualityConstraint("a", q[0] + q[1], target=0.5),
            cc.VelocityEqualityConstraint("b", 2.0 * (q[0] + q[1]), target=1.0)]
    spec = cc.SkillSpecification("dup", t, q, robot_vel_var=dq, constraints=cons)
    ctrl = cc.ReactiveQPController(spec)
    lib = rollout_vjp_library(ctrl, tmp_path)
    inp = {"t": np.zeros(2), "q": np.zeros((2, 2))}
    run = Run(3, 0.1)
    _, _, _, failed, tape = host_tape(lib, ctrl, inp, run)
    assert np.all(failed == 0) and np.all((tape["active"][:, 0] | tape["active"][:, 1]) == 3)
    pb = host_sweep(lib, ctrl, inp, run, tape, np.array([[0.0, 1.0], [0.0, 1.0]]))
    assert np.all(pb[:, 0] == 0.0) and np.isnan(pb[:, 1]).all()


def test_singular_hessian_gives_nan(tmp_path):
    from test_face_reference_on_host import make_case
    kind, sc, ctrl = make_case("offaxis_eps_0")
    lib = rollout_vjp_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(8, seed=8).items() if v is not None}
    _, full = theta_rows(ctrl, inp)
    run = Run(3, 0.01)
    _, _, _, failed, tape = host_tape(lib, ctrl, full, run)
    solved = failed == 0
    assert solved.any()
    cq, _, csol = cotangents(ctrl, 8, 9)
    pb = host_sweep(lib, ctrl, full, run, tape, cq, None, csol)
    assert np.isnan(pb[:, solved]).all()


# ---- emitted source and loading ----------------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENARIOS)
def test_rollout_vjp_source_is_the_vjp_source_plus_one_section(name, tmp_path):
    ctrl = scenarios.get(name).make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    kind = "nlp" if "nlp" in name else "qp"
    vsrc, vmeta = ctrl._vjp_source()
    src, meta = ctrl._rollout_vjp_source()
    assert not vmeta["rollout_vjp"] and meta["rollout_vjp"]
    head, sep, tail = src.partition("\n\n// ---- reverse-mode derivative of the closed-loop rollout "
                                    "(clik_rollout_vjp.cuh) ----\n")
    assert sep and tail.count("__global__") == 2
    assert ("clik_%s_rollout_tape_kernel(" % kind) in tail and ("clik_%s_rollout_vjp_kernel(" % kind) in tail
    lines = (head + "\n").split("\n")
    o22 = [ln for ln in lines if ln.lstrip().startswith("o[22] = ")]
    assert o22 == ["  o[22] = %d;   // taped rollout and reverse sweep kernels (1 QP, 2 NLP)"
                   % (2 if kind == "nlp" else 1)]
    lines.remove(o22[0])
    # (the VJP section's text differs from one emission to the next in the order of commutative operands: compare
    # what precedes it, and its kernels)
    marker = "\n\n// ---- reverse-mode derivative of the step's output (clik_vjp.cuh) ----\n"
    mine, theirs = "\n".join(lines).partition(marker), vsrc.partition(marker)
    assert mine[0] == theirs[0] and mine[1] == theirs[1]
    kernels = lambda text: [ln for ln in text.split("\n") if "__global__" in ln]  # noqa: E731
    assert kernels(mine[2]) == kernels(theirs[2])
    for s in (ctrl.kernel_source, vsrc, ctrl._jvp_source()[0], ctrl._rollout_jvp_source()[0]):
        assert "rollout_vjp" not in s and "rollout_tape" not in s and "o[22]" not in s


def test_initial_value_qp_has_no_rollout_vjp_section():
    from casclik_b200.codegen import emit_skill
    prog = _cart()._program()
    prog.emit_rollout = False
    src, meta = emit_skill(qp=prog, label="x", vjp=True, rollout_vjp=True)
    assert meta["vjp"] and not meta["rollout_vjp"] and "rollout_vjp" not in src and "o[22]" not in src


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_more_than_32_rows_raise_and_build_no_kernel(kind, tmp_path, monkeypatch):
    ctrl = _ctrl(kind, _wide_spec(33))
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._rollout_vjp_source()
    assert not meta["rollout_vjp"] and "rollout_vjp_kernel" not in source and "o[22]" not in source
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no image may be built"))
    N = 4
    for call in (lambda: ctrl.rollout_vjp(np.zeros(N), np.zeros((3, N)), 5, 0.01, q_bar=np.ones((3, N))),
                 lambda: ctrl.rollout_batch_differentiable(np.zeros(N), np.zeros((3, N)), 5, 0.01)):
        with pytest.raises(ValueError, match="at most 32 constraint rows"):
            call()
    assert ctrl._rollout_vjp is None


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_numpy_inputs_raise_without_building_the_image(name, tmp_path, monkeypatch):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no image may be built"))
    inp = sc.sample(4, seed=1)
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.rollout_vjp(inp["t"], inp["q"], 5, 0.01, input_var=inp["y"], q_bar=np.ones((6, 4)))
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.rollout_batch_differentiable(inp["t"], inp["q"], 5, 0.01, input_var=inp["y"])
    assert ctrl._rollout_vjp is None


def test_abi_rejects_a_null_skill():
    from casclik_b200 import runtime
    lib = runtime.load_library()
    for name in ("clik_qp_rollout_tape", "clik_nlp_rollout_tape"):
        assert getattr(lib, name)(None, 4, 3, 0.01, None, 0, None, None, None, 1.0, 1.0, None, None, 0,
                                  *([None] * 6)) == 1
        assert b"skill is NULL" in lib.clik_last_error()
    for name in ("clik_qp_rollout_vjp", "clik_nlp_rollout_vjp"):
        assert getattr(lib, name)(None, 4, 3, 0.01, None, 0, None, 1.0, 1.0, *([None] * 13)) == 1
        assert b"skill is NULL" in lib.clik_last_error()


def test_report_observed_maxima():
    """Runs last in this module: the largest deviations of the checks above."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items())})
