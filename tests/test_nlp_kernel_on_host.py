"""The NLP controller's kernel source — the translation unit the expression compiler emits for a skill plus
csrc/clik_nlp.cuh / clik_qp.cuh — compiled for the HOST with g++ and the shims of test_kernel_code_on_host.py
(one "thread", grid-stride loop over all instances), against the reference-generated QP fixture, SciPy's
SLSQP and a first-order KKT certificate.  A harness for the device code's logic, not a product path; the GPU
tests run the same source as sm_100a code (test_gpu_nlp.py)."""
import ctypes

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import cs, scenarios
from nlp_oracle import Instance, constraint_rows, nlp_kkt_residuals, slsqp
from oracle_bridge import orc
from test_golden_controllers import QP, VECTORS, golden_qp, load_case
from test_kernel_code_on_host import _host_library, _inputs, _p

MU = cc.ReactiveNLPController.weight_shifter


def run_step(lib, ctrl, inp, x0=None, max_iter=50):
    t, q, x, y = _inputs(inp)
    N = q.shape[1]
    if ctrl._nxv and x is None:
        x = np.zeros((ctrl._nxv, N))
    n = ctrl._qn
    sol = np.full((n, N), np.nan)
    status, iters = np.full(N, -9, dtype=np.int32), np.full(N, -9, dtype=np.int32)
    active = np.zeros((2, N), dtype=np.uint32)
    x0 = None if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
    lib.clik_nlp_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x),
                        _p(y if ctrl._ny else None), _p(x0), _p(sol), _p(status), _p(iters), _p(active),
                        ctypes.c_int(max_iter))
    return sol, status, iters, active


def qp_equivalent_cost(spec, qc):
    """mu*sum(w_rob dq^2) + mu*sum(w_virt dx^2): with the slack term of get_cost_expr, twice the QP
    controller's objective, so both controllers have the same minimiser."""
    dq = spec.robot_vel_var
    cost = MU * cs.dot(qc.robot_var_weights * dq, dq)
    if spec.virtual_var is not None and spec.n_virtual_var:
        dx = spec.virtual_vel_var
        cost = cost + MU * cs.dot(qc.virtual_var_weights * dx, dx)
    return cost


@pytest.mark.parametrize("name", QP)
def test_quadratic_cost_reproduces_the_reference_qp_minimisers(name, tmp_path):
    spec, inp, kwargs, outputs = load_case(name)
    qc = cc.ReactiveQPController(spec, **kwargs)
    ctrl = cc.ReactiveNLPController(spec, qp_equivalent_cost(spec, qc), slack_var_weights=qc.slack_var_weights)
    lib = _host_library(ctrl, tmp_path)
    assert ctrl.kernel_meta["nlp_quadratic"]
    gx, gh, gA, glb, gub = golden_qp(outputs)
    sol, status, iters, active = run_step(lib, ctrl, inp)
    assert np.all(status == 0) and np.all(iters == 1)
    for i in range(gx.shape[0]):
        assert np.abs(sol[:, i] - gx[i]).max() <= 1e-7 * (1 + np.abs(gx[i]).max()), i
        _, lam, st = orc.solve_qp_single(gh, gA[i], glb[i], gub[i])
        assert st == 0
        firm = np.abs(lam) > 1e-9                      # rows with a vanishing multiplier may go either way
        for r in np.nonzero(firm[:32])[0]:
            assert bool((int(active[0, i]) >> r) & 1) == (lam[r] > 0), (i, r)
            assert bool((int(active[1, i]) >> r) & 1) == (lam[r] < 0), (i, r)


def _check_against_slsqp(ctrl, lib, inp, n_check=64):
    prog = ctrl._prog
    sol, status, iters, active = run_step(lib, ctrl, inp)
    A, lb, ub = constraint_rows(prog, inp)
    N = inp["q"].shape[1]
    solved = 0
    for i in range(min(N, n_check)):
        _, _, qst = orc.solve_qp_single(np.ones(prog.nx), A[i], lb[i], ub[i])
        if qst != 0:                                    # the constraint rows have no feasible point
            assert status[i] == 2, i
            continue
        assert status[i] == 0, (i, status[i], iters[i])
        solved += 1
        inst = Instance(prog, inp, i)
        x = sol[:, i]
        F, g = inst.fg(x)
        kk = nlp_kkt_residuals(g, A[i], lb[i], ub[i], x)
        gs = 1.0 + np.abs(g).max()
        assert kk["primal"] < 1e-8 * (1 + np.abs(A[i] @ x).max()), (i, kk)
        assert kk["stationarity"] < 1e-8 * gs and kk["sign"] < 1e-8 * gs, (i, kk)
        x0, _, _ = orc.solve_qp_single(np.ones(prog.nx), A[i], lb[i], ub[i])   # a feasible start
        xs, Fs, ok = slsqp(inst, A[i], lb[i], ub[i], x0)
        assert ok, i
        assert abs(F - Fs) <= 1e-6 * (1 + abs(Fs)), (i, F, Fs)
        assert np.abs(x - xs).max() <= 1e-6 * (1 + np.abs(xs).max()), (i, np.abs(x - xs).max())
    return solved, iters[:n_check]


@pytest.mark.parametrize("name", sorted(scenarios.NLP_REGISTRY))
def test_scenarios_against_slsqp_and_kkt(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = _host_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(64, seed=0).items() if v is not None}
    solved, iters = _check_against_slsqp(ctrl, lib, inp)
    assert solved == 64
    if name == "ur5_nlp_taskspeed":
        assert ctrl.kernel_meta["nlp_quadratic"] and np.all(iters == 1)
    else:
        assert not ctrl.kernel_meta["nlp_quadratic"] and iters.max() > 2


def random_convex_cost(spec, seed):
    """mu*sum(a dq^2) + sum(b dq^4) + (c'dq)^2 + d'dq (+ mu*dx^2): convex, not quadratic."""
    rng = np.random.default_rng(40_000 + seed)
    dq = spec.robot_vel_var
    n = spec.n_robot_var
    a, b, c, d = (cs.DM(rng.uniform(lo, hi, n)) for lo, hi in ((0.5, 2.0), (0.5, 5.0), (-1.0, 1.0), (-0.01, 0.01)))
    u2 = dq * dq
    cost = MU * cs.dot(a, u2) + cs.dot(b, u2 * u2) + cs.dot(c, dq) ** 2 + cs.dot(d, dq)
    if spec.virtual_var is not None and spec.n_virtual_var:
        cost = cost + MU * cs.dot(spec.virtual_vel_var, spec.virtual_vel_var)
    return cost


@pytest.mark.parametrize("seed", range(4))
def test_fuzzed_skills_with_a_random_convex_cost(seed, tmp_path):
    from fuzz_skills import make_qp_skill
    spec, _, inp = make_qp_skill(seed)
    ctrl = cc.ReactiveNLPController(spec, random_convex_cost(spec, seed))
    lib = _host_library(ctrl, tmp_path)
    assert not ctrl.kernel_meta["nlp_quadratic"]
    if ctrl._nxv and "x" not in inp:
        inp = dict(inp, x=np.zeros((ctrl._nxv, inp["q"].shape[1])))
    inp = {k: (v[..., :64] if k != "t" else v[:64]) for k, v in inp.items()}
    solved, _ = _check_against_slsqp(ctrl, lib, inp)
    assert solved >= 16


def test_nonconvex_cost_returns_a_first_order_point(tmp_path):
    """|dq|^2 - (c'dq)^2 (|c| > 1: indefinite) inside the speed box: the Hessian is shifted until it is
    positive definite; the result is solved (0) or a stalled line search (5), and where solved it passes
    the first-order certificate.  No parity claim: other local minima exist."""
    sc = scenarios.get("ur5_qp")
    spec = sc.spec
    dq = spec.robot_vel_var
    c = cs.DM([0.3, -0.5, 0.8, 0.1, 0.4, -0.2])
    ctrl = cc.ReactiveNLPController(spec, cs.dot(dq, dq) - cs.dot(c, dq) ** 2)
    lib = _host_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(32, seed=3).items() if v is not None}
    sol, status, iters, _ = run_step(lib, ctrl, inp, max_iter=500)   # shifted steps converge linearly
    assert set(np.unique(status)) <= {0, 5} and (status == 0).any()
    A, lb, ub = constraint_rows(ctrl._prog, inp)
    for i in np.nonzero(status == 0)[0]:
        F, g = Instance(ctrl._prog, inp, i).fg(sol[:, i])
        kk = nlp_kkt_residuals(g, A[i], lb[i], ub[i], sol[:, i])
        gs = 1.0 + np.abs(g).max()
        assert kk["primal"] < 1e-8 and kk["stationarity"] < 1e-7 * gs and kk["sign"] < 1e-7 * gs, (i, kk)


def test_status_paths(tmp_path):
    # hard rows that contradict each other: infeasible (2)
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    cons = [cc.VelocitySetConstraint("a", q[0], set_min=0.5, set_max=1.0),
            cc.VelocitySetConstraint("b", q[0], set_min=-1.0, set_max=-0.5, priority=1)]
    spec = cc.SkillSpecification("infeasible", t, q, robot_vel_var=dq, constraints=cons)
    ctrl = cc.ReactiveNLPController(spec, cs.dot(dq, dq))
    (tmp_path / "a").mkdir()
    lib = _host_library(ctrl, tmp_path / "a")
    _, status, _, _ = run_step(lib, ctrl, {"t": np.zeros(3), "q": np.zeros((2, 3))})
    assert np.all(status == 2)
    # a NaN input: invalid (4); the other instances are unaffected
    sc = scenarios.get("ur5_nlp_quartic")
    ctrl = sc.make_controller()
    (tmp_path / "b").mkdir()
    lib = _host_library(ctrl, tmp_path / "b")
    inp = {k: v for k, v in sc.sample(8, seed=1).items() if v is not None}
    inp["q"][2, 3] = np.nan
    sol, status, iters, active = run_step(lib, ctrl, inp)
    assert status[3] == 4 and iters[3] == 0 and active[0, 3] == 0 and np.all(np.delete(status, 3) == 0)
    # the SQP cap: one iteration is not enough for the quartic cost (1)
    inp["q"][2, 3] = 1.0
    _, status, iters, _ = run_step(lib, ctrl, inp, max_iter=1)
    assert np.all(status == 1) and np.all(iters == 1)


@pytest.mark.parametrize("name", [n for n in QP if VECTORS[n].get("rollout")])
def test_rollout_matches_a_loop_of_warm_started_steps(name, tmp_path):
    spec, inp, kwargs, outputs = load_case(name)
    qc = cc.ReactiveQPController(spec, **kwargs)
    dq = spec.robot_vel_var
    cost = qp_equivalent_cost(spec, qc) + cs.sum1((dq * dq) * (dq * dq))   # not quadratic: several iterations
    ctrl = cc.ReactiveNLPController(spec, cost, slack_var_weights=qc.slack_var_weights)
    lib = _host_library(ctrl, tmp_path)
    cfg = VECTORS[name]["rollout"]["config"]
    n, steps, dt = cfg["n"], cfg["steps"], cfg["dt"]
    inf = float("inf")
    vq = inf if cfg["max_speed"] is None else cfg["max_speed"]
    vx = inf if cfg["max_virtual_speed"] is None else cfg["max_virtual_speed"]
    t, q, x, y = _inputs(inp)
    nq = q.shape[0]
    qs = np.ascontiguousarray(q[:, :n])
    xs = None if x is None else np.ascontiguousarray(x[:, :n])
    ys = None if y is None else np.ascontiguousarray(y[:, :n])
    ts = np.ascontiguousarray(t[:n])
    # the loop: step k at t0 + k*dt from the previous solution (0 after a failed step), clip, Euler
    ql, xl = qs.copy(), None if xs is None else xs.copy()
    warm = np.zeros((ctrl._qn, n))
    failed = np.zeros(n, dtype=np.int32)
    for k in range(steps):
        step_in = {"t": ts + dt * k, "q": ql}
        if xl is not None:
            step_in["x"] = xl
        if ys is not None:
            step_in["y"] = ys
        sol, status, _, _ = run_step(lib, ctrl, step_in, x0=warm)
        bad = status != 0
        failed += bad
        sol[:, bad] = 0.0
        warm = sol.copy()
        ql = ql + np.clip(sol[:nq], -vq, vq) * dt
        if xl is not None:
            xl = xl + np.clip(sol[nq:nq + xl.shape[0]], -vx, vx) * dt
    nf = np.full(n, -9, dtype=np.int32)
    last = np.full((ctrl._qn, n), np.nan)
    lib.clik_nlp_rollout_kernel(ctypes.c_longlong(n), ctypes.c_longlong(n), ctypes.c_int(steps), ctypes.c_double(dt),
                                _p(ts), ctypes.c_int(1), _p(qs), _p(xs), _p(ys), ctypes.c_double(vq), ctypes.c_double(vx),
                                _p(last), _p(nf), ctypes.c_int(50))
    assert np.array_equal(nf, failed)
    assert np.abs(qs - ql).max() <= 1e-9 * (1 + np.abs(ql).max())
    if xs is not None:
        assert np.abs(xs - xl).max() <= 1e-9 * (1 + np.abs(xl).max())
