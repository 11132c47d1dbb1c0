"""Forward-mode derivative of the QP and NLP closed-loop rollouts on the GPU (rollout_jvp, rollout_jacobian): against
the host build of the same kernel source, against the composed device loop of solve_batch + jvp_batch /
jacobian_batch at 2^16 instances, the primal outputs against rollout_batch and the hard-tracking known answers at
2^18, and the step, JVP and rollout outputs unchanged by the new image."""
import numpy as np
import pytest

from test_gpu_vjp import ALL, QP_SCENARIOS, _dev_inputs, _setup, _torch, _up
from test_jvp_on_host import _split
from test_rollout_jvp_on_host import (Run, _tracking, composed, host_rollout_jac, host_rollout_jvp, rollout_library,
                                      tangents)
from test_vjp_on_host import theta_rows

pytestmark = pytest.mark.gpu


def _speed(ctrl, t, q, x, y, frac):
    """frac of the largest first-step robot speed: a clip that holds on part of the steps."""
    sol = ctrl.solve_batch(t, q, x, y)[0]
    return frac * float(sol[:ctrl.skill_spec.n_robot_var].abs().amax())


def _clone(*a):
    return [None if v is None else v.clone() for v in a]


def _rel(a, b):
    a, b = a.reshape(-1, a.shape[-1]), b.reshape(-1, b.shape[-1])
    return (a - b).abs().amax(dim=0) / (1 + b.abs().amax(dim=0))


def _ulp_sensitivity(lib, ctrl, full, run, td, seed):
    """Per instance, how far the host tangent (q_dot, sol_dot) and Jacobian rollouts move, relative, when every state
    input moves by about 5 ulps (1e-15 relative, two random draws).  It measures how much the rollout amplifies
    rounding-level changes: a closed loop that is unstable over the steps (Moe-2016's box rows with gain 500 multiply
    by 1 - 500 dt = -3 per step where they hold) amplifies them by many orders of magnitude."""
    _, _, _, _, qd, _, sd = host_rollout_jvp(lib, ctrl, full, run, td)
    jac = host_rollout_jac(lib, ctrl, full, run)[4]
    rng = np.random.default_rng(seed)
    out = np.zeros((3, full["q"].shape[1]))
    for _ in range(2):
        moved = {k: (v * (1 + 1e-15 * rng.standard_normal(v.shape)) if k != "t" else v.copy()) for k, v in full.items()}
        _, _, _, _, mqd, _, msd = host_rollout_jvp(lib, ctrl, moved, run, td)
        mjac = host_rollout_jac(lib, ctrl, moved, run)[4]
        for r, (a, b) in enumerate(((mqd, qd), (msd, sd), (mjac, jac))):
            a, b = a.reshape(-1, a.shape[-1]), b.reshape(-1, b.shape[-1])
            out[r] = np.fmax(out[r], np.abs(a - b).max(axis=0) / (1 + np.abs(b).max(axis=0)))
    return out


@pytest.mark.parametrize("name", ALL)
def test_device_rollouts_agree_with_the_host_build(name, tmp_path):
    """On the instances whose host and device rollouts take the same working set and clip decision at every step
    (the device loop of composed_device, which the fused kernels equal bit for bit, against the host composed loop):
    within 1e-12 relative plus 10 times what the host rollout itself moves under ulp-level changes of its inputs
    (_ulp_sensitivity), since the two builds round differently.  Elsewhere the two builds' roundings took different
    faces and the tangents differ by design."""
    sc, ctrl, inp = _setup(name, 256, seed=51)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    t, q, x, y = _dev_inputs(ctrl, inp)
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 10, 0.008
    td = tangents(ctrl, inp, 52)
    td[:, 3] = 0.0
    parts = [_up(a) if a is not None else None for a in _split(ctrl, td)]
    qa, xa = _clone(q, x)
    dev = ctrl.rollout_jvp(t, qa, steps, dt, xa, y, max_speed=vq, max_virtual_speed=vq, t_dot=parts[0],
                           q_dot=parts[1], x_dot=parts[2], y_dot=parts[3])
    qb, xb = _clone(q, x)
    djac = ctrl.rollout_jacobian(t, qb, steps, dt, xb, y, max_speed=vq, max_virtual_speed=vq)["jac"].cpu().numpy()
    dtrace = []
    composed_device(ctrl, kind, t, q, x, y, steps, dt, vq, trace=dtrace)
    hc = sc.make_controller()
    lib = rollout_library(hc, tmp_path)
    _, full = theta_rows(hc, inp)
    run = Run(steps, dt, vq, vq)
    _, _, _, hfailed, hqd, _, hsd = host_rollout_jvp(lib, hc, full, run, td)
    hjac = host_rollout_jac(lib, hc, full, run)[4]
    htrace = composed(lib, hc, full, run)["trace"]
    same = np.ones(q.shape[1], dtype=bool)
    for (s0, a0, k0), (s1, a1, k1) in zip(htrace, dtrace):
        same &= (s0 == s1) & np.all(a0 == a1.astype(np.uint32), axis=0) & np.all(k0 == k1, axis=0)
    assert np.array_equal(dev["n_failed"].cpu().numpy(), hfailed)
    dqd, dsd = dev["q_dot"].cpu().numpy(), dev["sol_dot"].cpu().numpy()
    bad = np.isnan(hqd).any(axis=0)
    assert np.array_equal(np.isnan(dqd).any(axis=0)[same], bad[same])
    assert np.array_equal(np.isnan(djac).any(axis=(0, 1))[same], bad[same])
    assert np.all(dqd[:, 3] == 0.0) and np.all(dsd[:, 3] == 0.0)
    ok = same & ~bad
    sens = _ulp_sensitivity(lib, hc, full, run, td, 59)
    errs = [np.abs(a - b).reshape(-1, a.shape[-1]).max(axis=0) / (1 + np.abs(b).reshape(-1, b.shape[-1]).max(axis=0))
            for a, b in ((dqd, hqd), (dsd, hsd), (djac, hjac))]
    ratio = [(e / (1e-12 + 10 * s))[ok] for e, s in zip(errs, sens)]
    print("%s: device vs host on %d of %d instances with the same decisions: max relative deviation q_dot %.2e, "
          "sol_dot %.2e, jac %.2e; largest deviation / (1e-12 + 10 x ulp sensitivity) %.2e; instances whose ulp "
          "sensitivity exceeds 1e-12: %d" % (name, int(same.sum()), same.size, errs[0][ok].max(), errs[1][ok].max(),
                                           errs[2][ok].max(), max(r.max() for r in ratio),
                                           int((sens.max(axis=0) > 1e-12).sum())))
    assert same.mean() >= 0.9
    assert all(r.max() <= 1.0 for r in ratio)


def composed_device(ctrl, kind, t, q, x, y, steps, dt, vq, td=None, jacobian=False, trace=None):
    """The rollout as a device loop of solve_batch (warm-started as the rollout) + jvp_batch / jacobian_batch + the
    clip mask + Euler.  -> (q, x, sol, failed, q_dot, x_dot, sol_dot, P); `trace` (a list) gets (status, active,
    clip mask) of every step as NumPy arrays."""
    torch = _torch()
    nq, nxv, N = ctrl.skill_spec.n_robot_var, ctrl._nxv, q.shape[1]
    ns = nq + nxv
    nt = 1 + ns + ctrl._ny
    q, x = _clone(q, x)
    t0 = t.clone()
    warm_a = torch.zeros((2, N), dtype=torch.int32, device=q.device)
    warm_x = torch.zeros((ctrl._qn, N), dtype=torch.float64, device=q.device)
    failed = torch.zeros(N, dtype=torch.int32, device=q.device)
    last = torch.zeros((ctrl._qn, N), dtype=torch.float64, device=q.device)
    sd = torch.zeros_like(last)
    if td is not None:
        td = [None if a is None else a.clone() for a in td]
    P = torch.zeros((ns, nt, N), dtype=torch.float64, device=q.device)
    for a in range(ns):
        P[a, 1 + a] = 1.0
    for k in range(steps):
        tk = t0 + dt * float(k)
        if kind == "qp":
            sol, status, active = ctrl.solve_batch(tk, q, x, y, warm_active=warm_a)
        else:
            sol, status, active, _ = ctrl.solve_batch(tk, q, x, y, warmstart=warm_x)
        keep = sol[:ns].abs() < vq
        if trace is not None:
            trace.append(tuple(a.cpu().numpy() for a in (status, active, keep)))
        if td is not None:
            sd = ctrl.jvp_batch(tk, q, x, y, sol, status, active, *td)
            sd[:ns] = torch.where(keep, sd[:ns], 0.0)
            td[1] = td[1] + sd[:nq] * dt
            if nxv:
                td[2] = td[2] + sd[nq:ns] * dt
        if jacobian:
            J = ctrl.jacobian_batch(tk, q, x, y, sol, status, active)[:ns]
            T = torch.zeros((nt, nt, N), dtype=torch.float64, device=q.device)
            T[0, 0] = 1.0
            T[1:1 + ns] = P
            for c in range(1 + ns, nt):
                T[c, c] = 1.0
            step = torch.bmm(J.permute(2, 0, 1), T.permute(2, 0, 1)).permute(1, 2, 0)
            P = P + dt * torch.where(keep[:, None], step, 0.0)
        ok = status == 0
        failed += (~ok).int()
        v = torch.where(ok, sol, 0.0)
        warm_a, warm_x = active, v
        last = v.clone()
        last[:ns] = v[:ns].clamp(-vq, vq)
        q += last[:nq] * dt
        if nxv:
            x += last[nq:ns] * dt
    return q, x, last, failed, (td[1] if td else None), (td[2] if td else None), sd, P


@pytest.mark.parametrize("name", ALL)
def test_device_rollouts_agree_with_the_composed_device_loop_at_2_16(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 16, seed=53)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    t, q, x, y = _dev_inputs(ctrl, inp)
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 25, 0.008
    parts = [_up(a) if a is not None else None for a in _split(ctrl, tangents(ctrl, inp, 54))]
    qa, xa = _clone(q, x)
    got = ctrl.rollout_jvp(t, qa, steps, dt, xa, y, max_speed=vq, max_virtual_speed=vq, t_dot=parts[0],
                           q_dot=parts[1], x_dot=parts[2], y_dot=parts[3])
    qb, xb = _clone(q, x)
    jr = ctrl.rollout_jacobian(t, qb, steps, dt, xb, y, max_speed=vq, max_virtual_speed=vq)
    rq, _, rsol, rfailed, rqd, _, rsd, P = composed_device(ctrl, kind, t, q, x, y, steps, dt, vq, parts, True)
    assert torch.equal(qa, rq) and torch.equal(got["sol"], rsol) and torch.equal(got["n_failed"], rfailed)
    bad = torch.isnan(got["q_dot"]).any(dim=0)
    assert torch.equal(bad, torch.isnan(rqd).any(dim=0) | torch.isnan(rsd).any(dim=0))
    e1 = _rel(got["q_dot"][:, ~bad], rqd[:, ~bad]).max().item()
    e2 = _rel(got["sol_dot"][:, ~bad], rsd[:, ~bad]).max().item()
    jbad = torch.isnan(jr["jac"]).any(dim=0).any(dim=0)
    e3 = _rel(jr["jac"][:, :, ~jbad], P[:, :, ~jbad]).max().item()
    print("%s at 2^16, K=25: max relative deviation fused vs composed: q_dot %.2e, sol_dot %.2e, jac %.2e; "
          "bit-identical tangent: %s; NaN instances %d" % (name, e1, e2, e3, e1 == 0.0 and e2 == 0.0,
                                                          int(bad.sum())))
    assert e1 <= 1e-12 and e2 <= 1e-12 and e3 <= 1e-12
    assert int(bad.sum()) <= (1 << 16) // 10


@pytest.mark.parametrize("name", ALL)
def test_primal_outputs_are_those_of_rollout_batch_at_2_18(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 18, seed=55)
    t, q, x, y = _dev_inputs(ctrl, inp)
    vq = _speed(ctrl, t, q, x, y, 0.7)
    outs = []
    for call in ("rollout_batch", "rollout_jvp", "rollout_jacobian"):
        qa, xa = _clone(q, x)
        r = getattr(ctrl, call)(t, qa, 50, 0.008, xa, y, max_speed=vq, max_virtual_speed=vq)
        outs.append((qa, xa, r["sol"], r["n_failed"]))
    for o in outs[1:]:
        assert all(a is None and b is None or torch.equal(a, b) for a, b in zip(outs[0], o))


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_hard_tracking_known_answers_at_2_18(kind):
    torch = _torch()
    kg, a, w, dt, K = 2.0, 0.4, 3.0, 0.02, 25
    ctrl = _tracking(kind, kg, a, w)
    ctrl.setup_solver()
    N = 1 << 18
    rng = np.random.default_rng(56)
    p0, t0 = rng.uniform(-1.5, 1.5, (1, N)), rng.uniform(0.0, 2.0, N)
    for vmax in (np.inf, 0.8):
        q = _up(p0)
        r = ctrl.rollout_jacobian(_up(t0), q, K, dt, max_speed=None if vmax == np.inf else vmax)
        jac = r["jac"].cpu().numpy()
        assert int(r["n_failed"].sum()) == 0
        p, dp0, dt0 = p0[0].copy(), np.ones(N), np.zeros(N)
        margin = np.full(N, np.inf)
        for k in range(K):
            tk = t0 + dt * k
            v = -kg * (p - a * np.sin(w * tk)) + a * w * np.cos(w * tk)
            margin = np.minimum(margin, np.abs(np.abs(v) - vmax))
            hold = np.abs(v) >= vmax
            fac = np.where(hold, 1.0, 1.0 - kg * dt)
            dp0 = fac * dp0
            dt0 = fac * dt0 + np.where(hold, 0.0, dt * (kg * a * w * np.cos(w * tk) - a * w * w * np.sin(w * tk)))
            p = p + np.clip(v, -vmax, vmax) * dt
        # instances whose clip decision the NumPy recursion might take differently (|v| within 1e-9 of vmax) are
        # left out
        sure = margin > 1e-9
        assert sure.mean() > 0.99
        e1 = np.abs(jac[0, 1] - dp0)[sure].max()
        e2 = np.abs(jac[0, 0] - dt0)[sure].max() / (1 + np.abs(dt0).max())
        print("%s vmax %s: dp_K/dp_0 %.2e, dp_K/dt_0 %.2e" % (kind, vmax, e1, e2))
        assert e1 <= 1e-12 and e2 <= 1e-12
        assert np.abs(q.cpu().numpy()[0] - p)[sure].max() <= 1e-12


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_step_jvp_and_rollout_outputs_unchanged_by_the_new_image(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 4096, seed=57)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    t, q, x, y = _dev_inputs(ctrl, inp)
    parts = [_up(a) if a is not None else None for a in _split(ctrl, tangents(ctrl, inp, 58))]

    def outputs():
        sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
        qa, xa = _clone(q, x)
        r = ctrl.rollout_batch(t, qa, 20, 0.008, xa, y, max_speed=0.5)
        return [sol, status, active, ctrl.jvp_batch(t, q, x, y, sol, status, active, *parts),
                ctrl.jacobian_batch(t, q, x, y, sol, status, active), qa, r["sol"], r["n_failed"]]
    before = outputs()
    qa, xa = _clone(q, x)
    ctrl.rollout_jvp(t, qa, 5, 0.008, xa, y, q_dot=parts[1])
    after = outputs()
    for a, b in zip(before, after):
        assert torch.equal(a.nan_to_num(), b.nan_to_num()) and torch.equal(a.isnan(), b.isnan())
    assert ctrl._rollout_jvp is not None and kind in ("qp", "nlp")
