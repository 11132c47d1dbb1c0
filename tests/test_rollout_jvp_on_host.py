"""Forward-mode derivative of the QP and NLP closed-loop rollouts (csrc/clik_jvp.cuh, clik_<kind>_rollout_jvp_kernel /
clik_<kind>_rollout_jacobian_kernel): the emitted rollout-JVP image built for the HOST with g++ (the harness of
test_jvp_on_host.py), against the composed loop of the step, step-JVP and step-Jacobian kernels of the same image,
the primal rollout kernel, finite differences of the rollout, known answers and the rules of include/clik.h."""
import ctypes
import subprocess

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import build, cs, scenarios
from test_golden_controllers import load_case
from test_jvp_on_host import _split, host_jac, host_jvp
from test_kernel_code_on_host import ROOT, SHIM, _p
from test_vjp_api import _ctrl, _setup_without_nvcc, _wide_spec
from test_vjp_on_host import _full_inputs, theta_rows

OBSERVED = {}
SCENARIOS = ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic"]
FIXTURES = ["qp/ur5_qp", "qp/ur5_moe2016", "qp/cart_path", "qp/kitchen_sink"]


def _note(key, v):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(v))


def rollout_library(ctrl, tmp_path):
    """setup_problem_functions without nvcc, then the rollout-JVP image's source built with g++."""
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._rollout_jvp_source()
    assert meta["rollout_jvp"]
    text = source.replace("__device__ const unsigned short", "static const unsigned short")
    src = tmp_path / "skill_rollout_jvp.cpp"
    src.write_text(SHIM + text)
    so = tmp_path / "skill_rollout_jvp.so"
    subprocess.run(["g++", "-O0", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-I",
                    str(ROOT) + "/casclik_b200/csrc", "-o", str(so), str(src)], check=True)
    return ctypes.CDLL(str(so))


def kind_of(ctrl):
    return "nlp" if isinstance(ctrl, cc.ReactiveNLPController) else "qp"


def max_iter(ctrl):
    return 10 * (ctrl._qn + ctrl._qm) if kind_of(ctrl) == "qp" else 50


class Run(object):
    """One rollout's configuration: steps, dt and the speed limits (inf: no clip)."""

    def __init__(self, steps, dt, vq=np.inf, vx=np.inf):
        self.steps, self.dt, self.vq, self.vx = steps, dt, vq, vx

    def head(self, ctrl, inp):
        """(state copies, primal argument list, outputs) of the rollout kernels' common arguments."""
        t, q, x, y = _full_inputs(ctrl, inp)
        q, x = q.copy(), (None if x is None else x.copy())
        N = q.shape[1]
        sol, failed = np.full((ctrl._qn, N), -7.0), np.full(N, -9, dtype=np.int32)
        args = [ctypes.c_longlong(N), ctypes.c_longlong(N), ctypes.c_int(self.steps), ctypes.c_double(self.dt), _p(t),
                ctypes.c_int(1), _p(q), _p(x), _p(y), ctypes.c_double(self.vq), ctypes.c_double(self.vx), _p(sol),
                _p(failed), ctypes.c_int(max_iter(ctrl))]
        return q, x, sol, failed, args


def host_rollout(lib, ctrl, inp, run):
    """clik_<kind>_rollout_kernel -> (q, x, sol, n_failed)."""
    q, x, sol, failed, args = run.head(ctrl, inp)
    getattr(lib, "clik_%s_rollout_kernel" % kind_of(ctrl))(*args)
    return q, x, sol, failed


def host_rollout_jvp(lib, ctrl, inp, run, td, null=()):
    """clik_<kind>_rollout_jvp_kernel along td (n_theta, N) -> (q, x, sol, n_failed, q_dot, x_dot, sol_dot)."""
    q, x, sol, failed, args = run.head(ctrl, inp)
    N = q.shape[1]
    parts = [None if k in null else a for k, a in zip("tqxy", _split(ctrl, td))]
    keep = [np.array(a, copy=True) if a is not None else None for a in parts]
    qd = np.full((q.shape[0], N), -7.0)
    xd = np.full((ctrl._nxv, N), -7.0) if ctrl._nxv else None
    sd = np.full((ctrl._qn, N), -7.0)
    getattr(lib, "clik_%s_rollout_jvp_kernel" % kind_of(ctrl))(*args, *[_p(a) for a in parts], _p(qd), _p(xd), _p(sd))
    assert all(a is None or np.array_equal(a, k) for a, k in zip(parts, keep))     # tangents are inputs only
    return q, x, sol, failed, qd, xd, sd


def host_rollout_jac(lib, ctrl, inp, run):
    """clik_<kind>_rollout_jacobian_kernel -> (q, x, sol, n_failed, jac (n_s, n_theta, N))."""
    q, x, sol, failed, args = run.head(ctrl, inp)
    nt = len(theta_rows(ctrl, inp)[0])
    jac = np.full((q.shape[0] + ctrl._nxv, nt, q.shape[1]), -7.0)
    getattr(lib, "clik_%s_rollout_jacobian_kernel" % kind_of(ctrl))(*args, _p(jac))
    return q, x, sol, failed, jac


def host_step_warm(lib, ctrl, inp, warm):
    """The step kernel warm-started as the rollout: QP from the working set `warm` (2, N), NLP from the point
    `warm` (nx, N)."""
    t, q, x, y = _full_inputs(ctrl, inp)
    N = q.shape[1]
    sol, status = np.full((ctrl._qn, N), np.nan), np.full(N, -9, dtype=np.int32)
    active = np.zeros((2, N), dtype=np.uint32)
    warm = np.ascontiguousarray(warm)
    if kind_of(ctrl) == "qp":
        lib.clik_qp_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
                           None, _p(warm), _p(sol), _p(status), _p(active), ctypes.c_int(max_iter(ctrl)))
    else:
        iters = np.zeros(N, dtype=np.int32)
        lib.clik_nlp_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
                            _p(warm), _p(sol), _p(status), _p(iters), _p(active), ctypes.c_int(max_iter(ctrl)))
    return sol, status, active


def composed(lib, ctrl, inp, run, td=None, jacobian=False):
    """The rollout as a host loop of the step kernel (warm-started as the rollout), the step JVP (td) or step
    Jacobian (jacobian=True) kernel, the clip mask and the Euler update.  -> dict with q, x, sol, failed, the
    tangent (qd, xd, sd) or P (n_s, n_theta, N), and per step the working sets and clip masks ("trace")."""
    kind = kind_of(ctrl)
    rows, full = theta_rows(ctrl, inp)
    nq, nxv, N = ctrl.skill_spec.n_robot_var, ctrl._nxv, full["q"].shape[1]
    ns, nt = nq + nxv, len(rows)
    state = {k: v.copy() for k, v in full.items()}
    t0 = full["t"].copy()
    warm = np.zeros((2, N), dtype=np.uint32) if kind == "qp" else np.zeros((ctrl._qn, N))
    vmax = np.array([run.vq] * nq + [run.vx] * nxv)[:, None]
    failed = np.zeros(N, dtype=np.int32)
    last = np.zeros((ctrl._qn, N))
    if td is not None:
        td = td.copy()
        sd = np.zeros((ctrl._qn, N))
    P = np.zeros((ns, nt, N))
    for a in range(ns):
        P[a, 1 + a] = 1.0
    trace = []
    for k in range(run.steps):
        state["t"] = t0 + run.dt * float(k)
        sol, status, active = host_step_warm(lib, ctrl, state, warm)
        keep = np.abs(sol[:ns]) < vmax                                 # the clip does not hold
        trace.append((status.copy(), active.copy(), keep.copy()))
        if td is not None:
            sd = host_jvp(lib, ctrl, kind, state, sol, status, active, td)
            sd[:ns] = np.where(keep, sd[:ns], 0.0)
            td[1:1 + ns] = td[1:1 + ns] + sd[:ns] * run.dt
        if jacobian:
            J = host_jac(lib, ctrl, kind, state, sol, status, active)[:ns]
            T = np.zeros((nt, nt, N))                                  # d theta_k / dp
            T[0, 0] = 1.0
            T[1:1 + ns] = P
            for c in range(1 + ns, nt):
                T[c, c] = 1.0
            P = P + run.dt * np.where(keep[:, None], np.einsum("scn,cdn->sdn", J, T), 0.0)
        ok = status == 0
        failed += ~ok
        v = np.where(ok, sol, 0.0)
        if kind == "qp":
            warm = active
        else:
            warm = v
        last = v.copy()
        last[:ns] = np.clip(v[:ns], -vmax, vmax)
        state["q"] = state["q"] + last[:nq] * run.dt
        if nxv:
            state["x"] = state["x"] + last[nq:ns] * run.dt
    out = {"q": state["q"], "x": state.get("x") if nxv else None, "sol": last, "failed": failed, "trace": trace, "P": P}
    if td is not None:
        out.update(qd=td[1:1 + nq], xd=td[1 + nq:1 + ns] if nxv else None,
                   sd=sd if run.steps else np.zeros((ctrl._qn, N)))
    return out


def tangents(ctrl, inp, seed):
    rows, _ = theta_rows(ctrl, inp)
    return np.random.default_rng(seed).standard_normal((len(rows), inp["q"].shape[1]))


def nan_set(*arrs):
    return np.any([np.isnan(a).any(axis=0) for a in arrs if a is not None], axis=0)


def rel(a, b):
    """max |a - b| / (1 + max |b|) per instance (last axis)."""
    a, b = a.reshape(-1, a.shape[-1]), b.reshape(-1, b.shape[-1])
    return np.abs(a - b).max(axis=0) / (1 + np.abs(b).max(axis=0))


def _same_primal(got, want):
    for g, w in zip(got, want):
        if g is not None or w is not None:
            assert np.array_equal(g, w), np.abs(g - w).max()


# ---- the fused rollouts against the composed loop and the primal kernel ---------------------------------------

def check_against_composed(ctrl, lib, inp, run, seed, name):
    """The tangent rollout against the composed loop (bit for bit: the structured step kernel takes the rollout's
    working-set warm start), the same NaN instances, the primal outputs of both new kernels bit-identical to the
    rollout kernel, and the Jacobian rollout against unit-tangent rollouts (1e-14) and the composed jacobian chain
    (1e-13).  -> the number of finite instances."""
    _, full = theta_rows(ctrl, inp)
    td = tangents(ctrl, inp, seed)
    prim = host_rollout(lib, ctrl, full, run)
    got = host_rollout_jvp(lib, ctrl, full, run, td)
    _same_primal(got[:4], prim)
    ref = composed(lib, ctrl, full, run, td=td, jacobian=True)
    assert kind_of(ctrl) == "nlp" or ctrl.kernel_meta.get("qp_structured")
    q, x, sol, failed, qd, xd, sd = got
    for g, w in ((q, ref["q"]), (x, ref["x"]), (sol, ref["sol"])):
        if g is not None:
            e = rel(g, w).max()
            _note("primal vs composed %s" % name, e)
            assert np.array_equal(g, w), e
    assert np.array_equal(failed, ref["failed"])
    bad = nan_set(qd, xd, sd)
    assert np.array_equal(bad, nan_set(ref["qd"], ref["xd"], ref["sd"]))
    assert np.isnan(qd[:, bad]).all() and np.isnan(sd[:, bad]).all()
    ok = ~bad
    for g, w in ((qd, ref["qd"]), (xd, ref["xd"]), (sd, ref["sd"])):
        if g is not None:
            e = rel(g[:, ok], w[:, ok]).max(initial=0)
            _note("tangent vs composed %s" % name, e)
            assert np.array_equal(g[:, ok], w[:, ok]), e
    # Jacobian rollout
    jq, jx, jsol, jfailed, jac = host_rollout_jac(lib, ctrl, full, run)
    _same_primal((jq, jx, jsol, jfailed), prim)
    jbad = np.isnan(jac).any(axis=(0, 1))
    assert np.isnan(jac[:, :, jbad]).all()
    e = rel(jac[:, :, ~jbad], ref["P"][:, :, ~jbad]).max(initial=0)
    _note("jacobian vs composed chain %s" % name, e)
    assert e <= 1e-13, e
    nt = jac.shape[1]
    for c in range(nt):
        unit = np.zeros_like(td)
        unit[c] = 1.0
        _, _, _, _, uq, ux, _ = host_rollout_jvp(lib, ctrl, full, run, unit)
        col = uq if ux is None else np.vstack([uq, ux])
        assert np.array_equal(nan_set(col), jbad)
        e = rel(jac[:, c, ~jbad], col[:, ~jbad]).max(initial=0)
        _note("jacobian column vs unit tangent %s" % name, e)
        assert e <= 1e-13, (c, e)
    # jac . td = the tangent rollout
    lin = np.einsum("scn,cn->sn", jac, td)
    tan = qd if xd is None else np.vstack([qd, xd])
    e = rel(lin[:, ok], tan[:, ok]).max(initial=0)
    _note("jacobian . tangent vs tangent rollout %s" % name, e)
    assert e <= 1e-12, e
    return int(ok.sum())


def _speed_limit(ctrl, inp, lib, frac=0.5):
    """A max_speed that clips part of the steps: frac of the largest first-step robot speed."""
    sol, _, _ = host_step_warm(lib, ctrl, _full_inputs_dict(ctrl, inp), np.zeros((2, inp["q"].shape[1]), np.uint32)
                               if kind_of(ctrl) == "qp" else np.zeros((ctrl._qn, inp["q"].shape[1])))
    nq = ctrl.skill_spec.n_robot_var
    return frac * float(np.nanmax(np.abs(sol[:nq])))


def _full_inputs_dict(ctrl, inp):
    return theta_rows(ctrl, inp)[1]


@pytest.mark.parametrize("name", FIXTURES)
def test_qp_fixtures_against_the_composed_loop(name, tmp_path):
    spec, inp, kwargs, _ = load_case(name)
    ctrl = cc.ReactiveQPController(spec, **kwargs)
    lib = rollout_library(ctrl, tmp_path)
    vq = _speed_limit(ctrl, inp, lib)
    run = Run(25, 0.01, vq, 0.5 * vq)
    n = check_against_composed(ctrl, lib, inp, run, 1, name)
    assert n >= 0.9 * inp["q"].shape[1]
    # some instance saturates the clip on some step
    trace = composed(lib, ctrl, _full_inputs_dict(ctrl, inp), run)["trace"]
    assert any((~keep).any() for _, _, keep in trace)


@pytest.mark.parametrize("name", SCENARIOS)
def test_scenarios_against_the_composed_loop(name, tmp_path):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = rollout_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(24, seed=41).items() if v is not None}
    vq = _speed_limit(ctrl, inp, lib, 0.7)
    run = Run(25, 0.008, vq, vq)
    assert check_against_composed(ctrl, lib, inp, run, 2, name) >= 20
    trace = composed(lib, ctrl, _full_inputs_dict(ctrl, inp), run)["trace"]
    assert any((~keep).any() for _, _, keep in trace)


# ---- finite differences of the rollout ---------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENARIOS)
def test_scenarios_match_finite_differences_of_the_rollout(name, tmp_path):
    """(rollout(p + h td) - rollout(p - h td)) / 2h against the tangent rollout, on the instances whose +-h rollouts
    keep the working-set and clip sequence of the rollout at p (the composed loop's trace)."""
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    lib = rollout_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(32, seed=43).items() if v is not None}
    rows, full = theta_rows(ctrl, inp)
    vq = _speed_limit(ctrl, inp, lib, 0.7)
    run = Run(25, 0.008, vq, vq)
    theta = np.vstack([full["t"][None]] + [full[k] for k in "qxy" if k in full])
    td = tangents(ctrl, inp, 44)
    td = td / np.abs(td).max(axis=0) * np.maximum(1.0, np.abs(theta))
    _, _, _, _, qd, _, _ = host_rollout_jvp(lib, ctrl, full, run, td)
    base = composed(lib, ctrl, full, run)["trace"]
    h = 1e-6
    same = np.ones(inp["q"].shape[1], dtype=bool)
    ends = {}
    for sgn in (1, -1):
        moved = {k: v.copy() for k, v in full.items()}
        for c, (key, row) in enumerate(rows):
            if row is None:
                moved[key] = moved[key] + sgn * h * td[c]
            else:
                moved[key][row] = moved[key][row] + sgn * h * td[c]
        tr = composed(lib, ctrl, moved, run)["trace"]
        for (s0, a0, k0), (s1, a1, k1) in zip(base, tr):
            same &= (s0 == 0) & (s1 == 0) & np.all(a0 == a1, axis=0) & np.all(k0 == k1, axis=0)
        ends[sgn] = host_rollout(lib, ctrl, moved, run)[0]
    fd = (ends[1] - ends[-1]) / (2 * h)
    err = rel(fd, qd)
    _note("finite differences %s" % name, err[same].max(initial=0))
    assert same.mean() >= 0.9, same.mean()
    assert err[same].max() <= 1e-6, err[same].max()


# ---- known answers -----------------------------------------------------------------------------------------

def _tracking(kind, k_gain, a, w):
    t, p, dp = cs.MX.sym("t"), cs.MX.sym("p"), cs.MX.sym("dp")
    eq = cc.EqualityConstraint("track", p - a * cs.sin(w * t), gain=k_gain)
    spec = cc.SkillSpecification("track_%s" % kind, t, p, robot_vel_var=dp, constraints=[eq])
    if kind == "qp":
        return cc.ReactiveQPController(spec, robot_var_weights=[1.0])
    return cc.ReactiveNLPController(spec, 0.5 * dp * dp)


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_hard_tracking_known_answers(kind, tmp_path):
    """p_dot = -k (p - a sin wt) + a w cos wt: dp_K/dp_0 = (1 - k dt)^K, dp_K/dt0 from the scalar recursion, and
    both with the factor 1 (and no forcing) on the steps where max_speed clips."""
    kg, a, w, dt, K = 2.0, 0.4, 3.0, 0.02, 25
    ctrl = _tracking(kind, kg, a, w)
    lib = rollout_library(ctrl, tmp_path)
    p0 = np.array([[-1.0, -0.3, 0.0, 0.2, 0.9, 2.0]])
    t0 = np.array([0.0, 0.1, 0.5, 1.0, 1.5, 0.3])
    inp = {"t": t0, "q": p0}
    for vmax in (np.inf, 0.8):
        run = Run(K, dt, vmax)
        _, _, _, failed, jac = host_rollout_jac(lib, ctrl, inp, run)
        assert np.all(failed == 0)
        # the recursion in NumPy, from the primal trajectory
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
        for got, want in ((jac[0, 1], dp0), (jac[0, 0], dt0)):
            e = np.abs(got - want).max() / (1 + np.abs(want).max())
            _note("hard tracking %s vmax %s" % (kind, vmax), e)
            assert e <= 1e-12, (vmax, got - want)
        _, _, _, _, qd, _, _ = host_rollout_jvp(lib, ctrl, inp, run, np.array([np.ones(6), np.zeros(6)]))
        assert np.abs(qd[0] - dt0).max() <= 1e-12 * (1 + np.abs(dt0).max())


def _cart():
    t, p, dp = cs.MX.sym("t"), cs.MX.sym("p"), cs.MX.sym("dp")
    eq = cc.EqualityConstraint("min_dist_cnstr", 0.75 - p, gain=1.0, constraint_type="soft", priority=1)
    lim = cc.SetConstraint("cart_limit_cnstr", p, gain=1.0, set_min=0.0, set_max=1.0)
    spd = cc.VelocitySetConstraint("speed_limit_cnstr", p, gain=10.0, set_min=-0.275, set_max=0.275)
    spec = cc.SkillSpecification("cart_qp", t, p, robot_vel_var=dp, constraints=[eq, lim, spd])
    return cc.ReactiveQPController(spec, robot_var_weights=[1.0])


def test_cart_known_answers(tmp_path):
    """SURVEY.md §8c cart: along a trajectory whose working set is the soft row alone or the speed row, the factor
    of dp_K/dp_0 per step is 1 - dt 1.001/1.002 or 1; replayed from the primal trajectory."""
    ctrl = _cart()
    lib = rollout_library(ctrl, tmp_path)
    inp = {"t": np.zeros(6), "q": np.array([[0.0, 0.2, 0.5, 0.6, 0.9, 1.0]])}
    run = Run(25, 0.05)
    ref = composed(lib, ctrl, inp, run)
    _, _, _, failed, jac = host_rollout_jac(lib, ctrl, inp, run)
    assert np.all(failed == 0)
    want = np.ones(6)
    speed_steps = 0
    p = inp["q"][0].copy()
    for k in range(run.steps):
        sol, status, _ = host_step_warm(lib, ctrl, {"t": np.zeros(6), "q": p[None].copy()},
                                        ref["trace"][k - 1][1] if k else np.zeros((2, 6), np.uint32))
        at_speed = np.abs(np.abs(sol[0]) - 0.275) <= 1e-12
        speed_steps += at_speed.sum()
        want = want * np.where(at_speed, 1.0, 1.0 - run.dt * 1.001 / 1.002)
        p = p + sol[0] * run.dt
    assert speed_steps > 0 and speed_steps < 6 * run.steps
    assert np.array_equal(p, ref["q"][0])
    assert np.abs(jac[0, 1] - want).max() <= 1e-12, jac[0, 1] - want
    assert np.all(jac[0, 0] == 0.0)                                            # nothing depends on t


# ---- rules -------------------------------------------------------------------------------------------------

def test_failed_steps_give_nan_unless_the_tangent_is_zero(tmp_path):
    ctrl = _cart()
    lib = rollout_library(ctrl, tmp_path)
    inp = {"t": np.zeros(4), "q": np.array([[0.5, 1.6, 0.5, 1.6]])}    # 1.6: outside the feasible band
    run = Run(10, 0.05)
    td = np.array([[0.0, 0.0, 0.0, 0.0], [1.0, 1.0, 0.0, 0.0]])
    q, _, _, failed, qd, _, sd = host_rollout_jvp(lib, ctrl, inp, run, td)
    assert failed[0] == 0 and failed[1] > 0
    assert np.isfinite(qd[:, 0]).all() and np.isnan(qd[:, 1]).all() and np.isnan(sd[:, 1]).all()
    assert np.all(qd[:, 2:] == 0.0) and np.all(sd[:, 2:] == 0.0)             # zero tangents stay exactly 0
    z = host_rollout_jvp(lib, ctrl, inp, run, td, null="tqxy")
    assert np.all(z[4] == 0.0) and np.all(z[6] == 0.0)
    jac = host_rollout_jac(lib, ctrl, inp, run)[4]
    assert np.isnan(jac[:, :, [1, 3]]).all() and np.isfinite(jac[:, :, [0, 2]]).all()


def test_steps_zero(tmp_path):
    sc = scenarios.get("ur5_qp")
    ctrl = sc.make_controller()
    lib = rollout_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(8, seed=2).items() if v is not None}
    _, full = theta_rows(ctrl, inp)
    td = tangents(ctrl, inp, 3)
    q, _, sol, failed, qd, _, sd = host_rollout_jvp(lib, ctrl, full, Run(0, 0.01), td)
    assert np.array_equal(q, full["q"]) and np.all(sol == 0.0) and np.all(failed == 0)
    assert np.array_equal(qd, td[1:7]) and np.all(sd == 0.0)
    jac = host_rollout_jac(lib, ctrl, full, Run(0, 0.01))[4]
    eye = np.zeros_like(jac)
    for a in range(6):
        eye[a, 1 + a] = 1.0
    assert np.array_equal(jac, eye)


def test_rank_deficient_working_set_gives_nan(tmp_path):
    """Two consistent equality rows on one velocity combination: the working set holds both, A_W is rank-deficient."""
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    cons = [cc.VelocityEqualityConstraint("a", q[0] + q[1], target=0.5),
            cc.VelocityEqualityConstraint("b", 2.0 * (q[0] + q[1]), target=1.0)]
    spec = cc.SkillSpecification("dup", t, q, robot_vel_var=dq, constraints=cons)
    ctrl = cc.ReactiveQPController(spec)
    lib = rollout_library(ctrl, tmp_path)
    inp = {"t": np.zeros(2), "q": np.zeros((2, 2))}
    sol, status, active = host_step_warm(lib, ctrl, inp, np.zeros((2, 2), np.uint32))
    assert np.all(status == 0) and np.all((active[0] | active[1]) == 3)
    td = np.array([[0.0, 1.0], [0.0, 1.0], [0.0, 1.0]])
    _, _, _, failed, qd, _, sd = host_rollout_jvp(lib, ctrl, inp, Run(3, 0.1), td)
    assert np.all(failed == 0)
    assert np.all(qd[:, 0] == 0.0) and np.isnan(qd[:, 1]).all() and np.isnan(sd[:, 1]).all()
    jac = host_rollout_jac(lib, ctrl, inp, Run(3, 0.1))[4]
    assert np.isnan(jac).all()


def test_singular_hessian_gives_nan(tmp_path):
    from test_face_reference_on_host import make_case
    kind, sc, ctrl = make_case("offaxis_eps_0")
    lib = rollout_library(ctrl, tmp_path)
    inp = {k: v for k, v in sc.sample(8, seed=8).items() if v is not None}
    _, full = theta_rows(ctrl, inp)
    q, _, _, failed, qd, _, sd = host_rollout_jvp(lib, ctrl, full, Run(3, 0.01), tangents(ctrl, inp, 9))
    solved = failed == 0
    assert solved.any()
    assert np.isnan(qd[:, solved]).all() and np.isnan(sd[:, solved]).all()
    jac = host_rollout_jac(lib, ctrl, full, Run(3, 0.01))[4]
    assert np.isnan(jac[:, :, solved]).all()


# ---- emitted source and loading ----------------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENARIOS)
def test_rollout_jvp_source_is_the_jvp_source_plus_one_section(name, tmp_path):
    ctrl = scenarios.get(name).make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    kind = "nlp" if "nlp" in name else "qp"
    src0, meta0 = ctrl.kernel_source, ctrl.kernel_meta
    jsrc, jmeta = ctrl._jvp_source()
    src1, meta1 = ctrl._rollout_jvp_source()
    assert not meta0["rollout_jvp"] and not jmeta["rollout_jvp"] and meta1["rollout_jvp"]
    head, sep, tail = src1.partition("\n\n// ---- forward-mode derivative of the closed-loop rollout ----\n")
    assert sep and tail.count("__global__") == 2
    assert ("clik_%s_rollout_jvp_kernel(" % kind) in tail and ("clik_%s_rollout_jacobian_kernel(" % kind) in tail
    jtail = src1.partition("\n\n// ---- forward-mode derivative of the step's output (clik_jvp.cuh) ----\n")[2]
    assert jtail.count("__global__") == 4
    lines = (head + "\n").split("\n")
    o21 = [ln for ln in lines if ln.lstrip().startswith("o[21] = ")]
    assert o21 == ["  o[21] = %d;   // tangent and Jacobian rollout kernels (1 QP, 2 NLP)" % (2 if kind == "nlp" else 1)]
    lines.remove(o21[0])
    # (the JVP section's text differs from one emission to the next in the order of commutative operands: compare
    # what precedes it, and its kernels)
    jvp_marker = "\n\n// ---- forward-mode derivative of the step's output (clik_jvp.cuh) ----\n"
    mine, theirs = "\n".join(lines).partition(jvp_marker), jsrc.partition(jvp_marker)
    assert mine[0] == theirs[0] and mine[1] == theirs[1]
    kernels = lambda text: [ln for ln in text.split("\n") if "__global__" in ln]  # noqa: E731
    assert kernels(mine[2]) == kernels(theirs[2])
    for src in (src0, jsrc, ctrl._vjp_source()[0]):
        assert "rollout_jvp" not in src and "o[21]" not in src


def test_initial_value_qp_has_no_rollout_section():
    from casclik_b200.codegen import emit_skill
    ctrl = _cart()
    prog = ctrl._program()
    prog.emit_rollout = False
    src, meta = emit_skill(qp=prog, label="x", jvp=True, rollout_jvp=True)
    assert meta["jvp"] and not meta["rollout_jvp"] and "rollout_jvp" not in src and "o[21]" not in src


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_more_than_32_rows_raise_and_build_no_kernel(kind, tmp_path, monkeypatch):
    ctrl = _ctrl(kind, _wide_spec(33))
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._rollout_jvp_source()
    assert not meta["rollout_jvp"] and "rollout_jvp_kernel" not in source and "o[21]" not in source
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no image may be built"))
    N = 4
    for call in (lambda: ctrl.rollout_jvp(np.zeros(N), np.zeros((3, N)), 5, 0.01, q_dot=np.ones((3, N))),
                 lambda: ctrl.rollout_jacobian(np.zeros(N), np.zeros((3, N)), 5, 0.01)):
        with pytest.raises(ValueError, match="at most 32 constraint rows"):
            call()
    assert ctrl._rollout_jvp is None


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_numpy_inputs_raise_without_building_the_image(name, tmp_path, monkeypatch):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no image may be built"))
    inp = sc.sample(4, seed=1)
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.rollout_jvp(inp["t"], inp["q"], 5, 0.01, input_var=inp["y"], q_dot=np.ones((6, 4)))
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.rollout_jacobian(inp["t"], inp["q"], 5, 0.01, input_var=inp["y"])
    assert ctrl._rollout_jvp is None


def test_abi_rejects_a_null_skill():
    from casclik_b200 import runtime
    lib = runtime.load_library()
    for name in ("clik_qp_rollout_jvp", "clik_nlp_rollout_jvp"):
        assert getattr(lib, name)(None, 4, 3, 0.01, None, 0, None, None, None, 1.0, 1.0, None, None, 0,
                                  *([None] * 8)) == 1
        assert b"skill is NULL" in lib.clik_last_error()
    for name in ("clik_qp_rollout_jacobian", "clik_nlp_rollout_jacobian"):
        assert getattr(lib, name)(None, 4, 3, 0.01, None, 0, None, None, None, 1.0, 1.0, None, None, 0,
                                  None, None) == 1
        assert b"skill is NULL" in lib.clik_last_error()


def test_report_observed_maxima():
    """Runs last in this module: the largest deviations of the checks above."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items())})
