"""Reverse-mode derivative of the QP and NLP closed-loop rollouts on the GPU (rollout_vjp,
rollout_batch_differentiable): the sweep against the composed device loop of vjp_batch over the tape at 2^16
instances, the adjoint identity against rollout_jvp at 2^18 and rollout_jacobian at 2^16, the primal outputs against
rollout_batch and the hard-tracking known answers at 2^18, the host build of the same source, torch autograd, the ABI
checks, and the step, derivative and rollout outputs unchanged by the new image."""
import ctypes

import numpy as np
import pytest

from test_gpu_rollout_jvp import _clone, _rel, _speed
from test_gpu_vjp import ALL, QP_SCENARIOS, _dev_inputs, _setup, _torch, _up
from test_jvp_on_host import _split
from test_rollout_jvp_on_host import Run, _tracking, composed, tangents
from test_rollout_vjp_on_host import host_sweep, host_tape, rollout_vjp_library
from test_vjp_on_host import theta_rows

pytestmark = pytest.mark.gpu


def _kind(name):
    return "qp" if name in QP_SCENARIOS else "nlp"


def _cot(ctrl, N, seed):
    """Random cotangents (q_bar_K, x_bar_K, sol_bar) on the device."""
    r = np.random.default_rng(seed)
    return (_up(r.standard_normal((ctrl.skill_spec.n_robot_var, N))),
            _up(r.standard_normal((ctrl._nxv, N))) if ctrl._nxv else None, _up(r.standard_normal((ctrl._qn, N))))


def _pbar(r):
    torch = _torch()
    return torch.cat([r["t_bar"][None]] + [r[k] for k in ("q_bar", "x_bar", "y_bar") if r[k] is not None])


def _tape(ctrl, kind, t, q, x, y, steps, dt, vq):
    """The private tape of the rollout (state copies), through the controllers' shared body."""
    from casclik_b200.controllers import base_controller as bc
    qa, xa = _clone(q, x)
    b = bc._rollout_batch(ctrl, "rollout_vjp", t, qa, xa, y)
    mi = ctrl._max_iter(None) if kind == "nlp" else int(ctrl.options.get("max_iter", 0) or 0)
    sol, failed, tape = bc._rollout_tape(ctrl, kind, b, steps, dt, vq, vq, mi)
    return qa, xa, sol, failed, tape


def _sweep_sensitivity(ctrl, kind, t, y, steps, dt, vq, tape, cq, cx, csol, seed):
    """Per instance, how far the device sweep moves, relative (max |change| / (1 + max |p_bar|)), when the tape's
    states and solutions move by about 5 ulps (1e-15 relative, two random draws) at fixed working sets and clip
    decisions: the ulp-sensitivity method of DESIGN.md §4.8 applied to the sweep.  A closed loop that is unstable over
    the steps (Moe-2016's box rows with gain 500 multiply by 1 - 500 dt = -3 per step where they hold) amplifies
    rounding-level changes by many orders of magnitude, and two compilations of the same face solve round
    differently.  -> (p_bar, sensitivity, p_bar of the moved tapes)."""
    torch = _torch()
    from casclik_b200.controllers import base_controller as bc
    q0 = tape["q"][0] if steps else None
    x0 = tape["x"][0] if (steps and ctrl._nxv) else None

    def sweep(tp):
        bb = bc._rollout_batch(ctrl, "rollout_vjp", t, q0.contiguous(), None if x0 is None else x0.contiguous(), y)
        return torch.cat([a if a.dim() == 2 else a[None] for a in bc._rollout_sweep(
            ctrl, kind, bb, steps, dt, vq, vq, tp, cq, cx, csol) if a is not None])
    base = sweep(tape)
    g = torch.Generator(device=base.device).manual_seed(seed)
    sens = torch.zeros(base.shape[1], dtype=torch.float64, device=base.device)
    others = []
    for _ in range(2):
        moved = dict(tape)
        for k in ("q", "x", "sol"):
            if tape[k] is not None:
                moved[k] = tape[k] * (1 + 1e-15 * torch.randn(tape[k].shape, dtype=torch.float64,
                                                              device=base.device, generator=g))
        others.append(sweep(moved))
        sens = torch.fmax(sens, _rel(others[-1], base))
    return base, sens, others


@pytest.mark.parametrize("name", ALL)
def test_sweep_matches_the_composed_device_loop_at_2_16(name):
    """K vjp_batch launches over the tape slices with the clip mask and the accumulation in torch."""
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 16, seed=61)
    kind = _kind(name)
    t, q, x, y = _dev_inputs(ctrl, inp)
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 25, 0.008
    cq, cx, csol = _cot(ctrl, q.shape[1], 62)
    qa, xa = _clone(q, x)
    got = ctrl.rollout_vjp(t, qa, steps, dt, xa, y, max_speed=vq, max_virtual_speed=vq, q_bar=cq, x_bar=cx,
                           sol_bar=csol)
    qt, xt, sol, failed, tape = _tape(ctrl, kind, t, q, x, y, steps, dt, vq)
    assert torch.equal(qa, qt) and torch.equal(got["sol"], sol) and torch.equal(got["n_failed"], failed)
    nq, nxv = ctrl.skill_spec.n_robot_var, ctrl._nxv
    ns = nq + nxv
    aq = cq.clone()
    ax = cx.clone() if nxv else torch.zeros((0, q.shape[1]), dtype=torch.float64, device=q.device)
    tb = torch.zeros_like(t)
    yb = torch.zeros((ctrl._ny, q.shape[1]), dtype=torch.float64, device=q.device)
    for k in range(steps - 1, -1, -1):
        sb = torch.zeros((ctrl._qn, q.shape[1]), dtype=torch.float64, device=q.device)
        sb[:ns] = dt * torch.cat([aq, ax])
        if k == steps - 1:
            sb = sb + csol
        sk = tape["sol"][k]
        sb[:ns] = torch.where(sk[:ns].abs() < vq, sb[:ns], 0.0)
        o = ctrl.vjp_batch(t + dt * float(k), tape["q"][k], tape["x"][k] if nxv else None, y, sk, tape["status"][k],
                           tape["active"][k], sb.contiguous())
        tb, aq = tb + o[0], aq + o[1]
        if nxv:
            ax = ax + o[2]
        if ctrl._ny:
            yb = yb + o[3]
    want = torch.cat([tb[None], aq, ax, yb])
    pb = _pbar(got)
    bad = torch.isnan(pb).any(dim=0)
    assert torch.equal(bad, torch.isnan(want).any(dim=0))
    err = _rel(pb[:, ~bad], want[:, ~bad])
    _, sens, _ = _sweep_sensitivity(ctrl, kind, t, y, steps, dt, vq, tape, cq, cx, csol, 60)
    ratio = (err / (1e-13 + 10 * sens[~bad])).max().item()
    print("%s at 2^16, K=25: sweep vs composed vjp_batch loop: max relative deviation %.2e, bit-identical %s, NaN "
          "instances %d; instances above 1e-13 %d; largest deviation / (1e-13 + 10 x ulp sensitivity) %.2e"
          % (name, err.max().item(), torch.equal(pb[:, ~bad], want[:, ~bad]), int(bad.sum()),
             int((err > 1e-13).sum()), ratio))
    assert ratio <= 1.0
    assert int(bad.sum()) <= (1 << 16) // 10


@pytest.mark.parametrize("name", ALL)
def test_adjoint_identity_against_rollout_jvp_at_2_18(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 18, seed=63)
    t, q, x, y = _dev_inputs(ctrl, inp)
    N = q.shape[1]
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 50, 0.008
    cq, cx, csol = _cot(ctrl, N, 64)
    parts = [_up(a) if a is not None else None for a in _split(ctrl, tangents(ctrl, inp, 65))]
    qa, xa = _clone(q, x)
    rv = ctrl.rollout_vjp(t, qa, steps, dt, xa, y, max_speed=vq, max_virtual_speed=vq, q_bar=cq, x_bar=cx,
                          sol_bar=csol)
    qb, xb = _clone(q, x)
    rj = ctrl.rollout_jvp(t, qb, steps, dt, xb, y, max_speed=vq, max_virtual_speed=vq, t_dot=parts[0],
                          q_dot=parts[1], x_dot=parts[2], y_dot=parts[3])
    assert torch.equal(qa, qb) and torch.equal(rv["sol"], rj["sol"])
    pd = torch.cat([parts[0][None]] + [a for a in parts[1:] if a is not None])
    pb = _pbar(rv)
    lhs = (cq * rj["q_dot"]).sum(0) + (csol * rj["sol_dot"]).sum(0)
    cn = cq.square().sum(0) + csol.square().sum(0)
    dn = rj["q_dot"].square().sum(0) + rj["sol_dot"].square().sum(0)
    if cx is not None:
        lhs = lhs + (cx * rj["x_dot"]).sum(0)
        cn, dn = cn + cx.square().sum(0), dn + rj["x_dot"].square().sum(0)
    rhs = (pb * pd).sum(0)
    scale = cn.sqrt() * dn.sqrt() + pb.norm(dim=0) * pd.norm(dim=0)
    ok = torch.isfinite(lhs) & torch.isfinite(rhs)
    err = ((lhs - rhs).abs() / scale)[ok]
    # the sweep's own ulp sensitivity, in the same measure
    tape = _tape(ctrl, _kind(name), t, q, x, y, steps, dt, vq)[4]
    _, _, others = _sweep_sensitivity(ctrl, _kind(name), t, y, steps, dt, vq, tape, cq, cx, csol, 62)
    sens = torch.stack([((o * pd).sum(0) - rhs).abs() / scale for o in others]).amax(0)[ok]
    ratio = (err / (1e-12 + 10 * sens)).max().item()
    print("%s at 2^18, K=50: adjoint identity max %.2e (median %.2e) on %d instances; NaN on either side %d; "
          "instances above 1e-12 %d; largest deviation / (1e-12 + 10 x ulp sensitivity) %.2e"
          % (name, err.max().item(), err.median().item(), int(ok.sum()), int((~ok).sum()), int((err > 1e-12).sum()),
             ratio))
    assert ratio <= 1.0
    assert int((~ok).sum()) <= N // 10


@pytest.mark.parametrize("name", ALL)
def test_unit_cotangents_give_the_rows_of_rollout_jacobian_at_2_16(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 16, seed=66)
    t, q, x, y = _dev_inputs(ctrl, inp)
    N = q.shape[1]
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 25, 0.008
    qa, xa = _clone(q, x)
    jac = ctrl.rollout_jacobian(t, qa, steps, dt, xa, y, max_speed=vq, max_virtual_speed=vq)["jac"]
    nq, ns = ctrl.skill_spec.n_robot_var, ctrl.skill_spec.n_robot_var + ctrl._nxv
    tape = _tape(ctrl, _kind(name), t, q, x, y, steps, dt, vq)[4]
    worst, above, ratio = 0.0, 0, 0.0
    for s in range(ns):
        uq = torch.zeros((nq, N), dtype=torch.float64, device=q.device)
        ux = torch.zeros((ctrl._nxv, N), dtype=torch.float64, device=q.device) if ctrl._nxv else None
        (uq if s < nq else ux)[s if s < nq else s - nq] = 1.0
        qb, xb = _clone(q, x)
        row = _pbar(ctrl.rollout_vjp(t, qb, steps, dt, xb, y, max_speed=vq, max_virtual_speed=vq, q_bar=uq,
                                     x_bar=ux))
        fin = ~torch.isnan(row).any(dim=0) & ~torch.isnan(jac[s]).any(dim=0)
        assert fin.float().mean().item() >= 0.9
        err = _rel(row[:, fin], jac[s][:, fin])
        _, sens, _ = _sweep_sensitivity(ctrl, _kind(name), t, y, steps, dt, vq, tape, uq, ux, None, 80 + s)
        worst = max(worst, err.max().item())
        above += int((err > 1e-13).sum())
        ratio = max(ratio, (err / (1e-13 + 10 * sens[fin])).max().item())
    print("%s at 2^16, K=25: unit cotangents vs rollout_jacobian rows: max relative deviation %.2e; entries above "
          "1e-13 %d; largest deviation / (1e-13 + 10 x ulp sensitivity) %.2e" % (name, worst, above, ratio))
    assert ratio <= 1.0


@pytest.mark.parametrize("name", ALL)
def test_primal_outputs_are_those_of_rollout_batch_at_2_18(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 18, seed=67)
    t, q, x, y = _dev_inputs(ctrl, inp)
    vq = _speed(ctrl, t, q, x, y, 0.7)
    qa, xa = _clone(q, x)
    r = ctrl.rollout_batch(t, qa, 50, 0.008, xa, y, max_speed=vq, max_virtual_speed=vq)
    qb, xb = _clone(q, x)
    v = ctrl.rollout_vjp(t, qb, 50, 0.008, xb, y, max_speed=vq, max_virtual_speed=vq, q_bar=torch.ones_like(q))
    qK, xK, sol, failed = ctrl.rollout_batch_differentiable(t, q, 50, 0.008, x, y, max_speed=vq,
                                                            max_virtual_speed=vq)
    for got in ((qb, xb, v["sol"], v["n_failed"]), (qK, xK, sol, failed)):
        assert all(a is None and b is None or torch.equal(a, b) for a, b in zip((qa, xa, r["sol"], r["n_failed"]),
                                                                               got))


@pytest.mark.parametrize("name", ALL)
def test_device_sweep_agrees_with_the_host_build(name, tmp_path):
    """On the instances whose host and device rollouts take the same working set and clip decision at every step:
    within 1e-12 relative plus 10 times what the host sweep itself moves when every state input moves by about 5
    ulps (the ulp-sensitivity bound of DESIGN.md §4.8), since the two builds round differently."""
    from test_gpu_rollout_jvp import composed_device
    sc, ctrl, inp = _setup(name, 256, seed=68)
    kind = _kind(name)
    t, q, x, y = _dev_inputs(ctrl, inp)
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 10, 0.008
    cq, cx, csol = _cot(ctrl, 256, 69)
    qa, xa = _clone(q, x)
    dev = _pbar(ctrl.rollout_vjp(t, qa, steps, dt, xa, y, max_speed=vq, max_virtual_speed=vq, q_bar=cq, x_bar=cx,
                                 sol_bar=csol)).cpu().numpy()
    dtrace = []
    composed_device(ctrl, kind, t, q, x, y, steps, dt, vq, trace=dtrace)
    hc = sc.make_controller()
    lib = rollout_vjp_library(hc, tmp_path)
    _, full = theta_rows(hc, inp)
    run = Run(steps, dt, vq, vq)
    c = [None if a is None else a.cpu().numpy() for a in (cq, cx, csol)]
    host = host_sweep(lib, hc, full, run, host_tape(lib, hc, full, run)[4], *c)
    htrace = composed(lib, hc, full, run)["trace"]
    same = np.ones(256, dtype=bool)
    for (s0, a0, k0), (s1, a1, k1) in zip(htrace, dtrace):
        same &= (s0 == s1) & np.all(a0 == a1.astype(np.uint32), axis=0) & np.all(k0 == k1, axis=0)
    rng = np.random.default_rng(70)
    sens = np.zeros(256)
    for _ in range(2):
        moved = {k: (v * (1 + 1e-15 * rng.standard_normal(v.shape)) if k != "t" else v.copy()) for k, v in full.items()}
        m = host_sweep(lib, hc, moved, run, host_tape(lib, hc, moved, run)[4], *c)
        sens = np.fmax(sens, np.abs(m - host).max(axis=0) / (1 + np.abs(host).max(axis=0)))
    bad = np.isnan(host).any(axis=0)
    assert np.array_equal(np.isnan(dev).any(axis=0)[same], bad[same])
    ok = same & ~bad
    err = np.abs(dev - host).max(axis=0) / (1 + np.abs(host).max(axis=0))
    ratio = (err / (1e-12 + 10 * sens))[ok]
    print("%s: device vs host sweep on %d of 256 instances with the same decisions: max relative deviation %.2e; "
          "largest deviation / (1e-12 + 10 x ulp sensitivity) %.2e" % (name, int(same.sum()), err[ok].max(),
                                                                     ratio.max()))
    assert same.mean() >= 0.9
    assert ratio.max() <= 1.0


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_hard_tracking_known_answers_at_2_18(kind):
    kg, a, w, dt, K = 2.0, 0.4, 3.0, 0.02, 25
    ctrl = _tracking(kind, kg, a, w)
    ctrl.setup_solver()
    N = 1 << 18
    rng = np.random.default_rng(71)
    p0, t0 = rng.uniform(-1.5, 1.5, (1, N)), rng.uniform(0.0, 2.0, N)
    for vmax in (np.inf, 0.8):
        r = ctrl.rollout_vjp(_up(t0), _up(p0), K, dt, max_speed=None if vmax == np.inf else vmax,
                             q_bar=_up(np.ones((1, N))))
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
        sure = margin > 1e-9
        assert sure.mean() > 0.99
        e1 = np.abs(r["q_bar"].cpu().numpy()[0] - dp0)[sure].max()
        e2 = np.abs(r["t_bar"].cpu().numpy() - dt0)[sure].max() / (1 + np.abs(dt0).max())
        print("%s vmax %s: q_bar_0 %.2e, t_bar_0 %.2e" % (kind, vmax, e1, e2))
        assert e1 <= 1e-12 and e2 <= 1e-12


@pytest.mark.parametrize("name", ALL)
def test_autograd_through_the_rollout(name):
    """loss.backward() equals rollout_vjp bit for bit, forward_ad equals rollout_jvp bit for bit, the inputs are not
    modified, and a shared one-element t0 gets the summed t_bar."""
    torch = _torch()
    import torch.autograd.forward_ad as fwAD
    sc, ctrl, inp = _setup(name, 4096, seed=72)
    t, q, x, y = _dev_inputs(ctrl, inp)
    N = q.shape[1]
    vq = _speed(ctrl, t, q, x, y, 0.7)
    steps, dt = 20, 0.008
    cq, cx, csol = _cot(ctrl, N, 73)
    kw = dict(max_speed=vq, max_virtual_speed=vq)
    leaves = [a.clone().requires_grad_(True) if a is not None else None for a in (t, q, x, y)]
    saved = [a.detach().clone() if a is not None else None for a in leaves]
    qK, xK, sol, failed = ctrl.rollout_batch_differentiable(leaves[0], leaves[1], steps, dt, leaves[2], leaves[3], **kw)
    loss = (cq * qK).sum() + (csol * sol).sum() + ((cx * xK).sum() if cx is not None else 0.0)
    loss.backward()
    for a, s in zip(leaves, saved):
        assert a is None or torch.equal(a.detach(), s)
    qa, xa = _clone(q, x)
    ref = ctrl.rollout_vjp(t, qa, steps, dt, xa, y, q_bar=cq, x_bar=cx, sol_bar=csol, **kw)
    assert torch.equal(qK, qa) and torch.equal(sol, ref["sol"]) and torch.equal(failed, ref["n_failed"])
    for a, k in zip(leaves, ("t_bar", "q_bar", "x_bar", "y_bar")):
        if a is not None:
            assert torch.equal(a.grad, ref[k]), k
    # a shared t0
    t1 = torch.tensor(0.3, dtype=torch.float64, device=q.device, requires_grad=True)
    qK1, _, sol1, _ = ctrl.rollout_batch_differentiable(t1, q, steps, dt, x, y, **kw)
    ((cq * qK1).sum() + (csol * sol1).sum()).backward()
    qa, xa = _clone(q, x)
    r1 = ctrl.rollout_vjp(torch.tensor(0.3, dtype=torch.float64, device=q.device), qa, steps, dt, xa, y, q_bar=cq,
                          sol_bar=csol, **kw)
    assert torch.equal(t1.grad, r1["t_bar"].sum())
    # forward mode
    parts = [_up(a) if a is not None else None for a in _split(ctrl, tangents(ctrl, inp, 74))]
    with fwAD.dual_level():
        duals = [fwAD.make_dual(a, d) if a is not None else None for a, d in zip((t, q, x, y), parts)]
        outs = ctrl.rollout_batch_differentiable(duals[0], duals[1], steps, dt, duals[2], duals[3], **kw)
        tq = fwAD.unpack_dual(outs[0]).tangent
        tsol = fwAD.unpack_dual(outs[2]).tangent
        tx = fwAD.unpack_dual(outs[1]).tangent if outs[1] is not None else None
    qa, xa = _clone(q, x)
    rj = ctrl.rollout_jvp(t, qa, steps, dt, xa, y, t_dot=parts[0], q_dot=parts[1], x_dot=parts[2], y_dot=parts[3],
                          **kw)
    eq = lambda a, b: torch.equal(a.nan_to_num(), b.nan_to_num()) and torch.equal(a.isnan(), b.isnan())  # noqa
    assert eq(tq, rj["q_dot"]) and eq(tsol, rj["sol_dot"]) and (tx is None or eq(tx, rj["x_dot"]))
    for a, s in zip((t, q, x, y), saved):
        assert a is None or torch.equal(a, s)


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_outputs_unchanged_by_the_new_image(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 4096, seed=75)
    t, q, x, y = _dev_inputs(ctrl, inp)
    parts = [_up(a) if a is not None else None for a in _split(ctrl, tangents(ctrl, inp, 76))]
    sb = _up(np.random.default_rng(77).standard_normal((ctrl._qn, q.shape[1])))

    def outputs():
        sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
        qa, xa = _clone(q, x)
        r = ctrl.rollout_batch(t, qa, 20, 0.008, xa, y, max_speed=0.5)
        qb, xb = _clone(q, x)
        rj = ctrl.rollout_jvp(t, qb, 20, 0.008, xb, y, max_speed=0.5, q_dot=parts[1])
        return [sol, status, active, *[a for a in ctrl.vjp_batch(t, q, x, y, sol, status, active, sb) if a is not None],
                ctrl.jvp_batch(t, q, x, y, sol, status, active, *parts), qa, r["sol"], r["n_failed"], qb, rj["q_dot"],
                rj["sol_dot"]]
    before = outputs()
    qa, xa = _clone(q, x)
    ctrl.rollout_vjp(t, qa, 5, 0.008, xa, y, q_bar=torch.ones_like(q))
    after = outputs()
    for a, b in zip(before, after):
        assert torch.equal(a.nan_to_num(), b.nan_to_num()) and torch.equal(a.isnan(), b.isnan())
    assert ctrl._rollout_vjp is not None


def test_abi_checks_with_a_loaded_image():
    """steps < 0, a NULL tape with steps > 0, a NULL output and an image without the kernels: CLIK_ERR_INVALID
    before any launch; steps = 0 passes the cotangent through."""
    torch = _torch()
    from casclik_b200 import runtime
    from casclik_b200.controllers.base_controller import vjp_image
    sc, ctrl, inp = _setup("ur5_qp", 64, seed=78)
    t, q, x, y = _dev_inputs(ctrl, inp)
    lib = runtime.load_library()
    skill = vjp_image(ctrl, "qp", 0, "rollout_vjp")
    p = lambda a: None if a is None else ctypes.c_void_p(a.data_ptr())  # noqa: E731
    N, f = 64, lambda *s: torch.zeros(s, dtype=torch.float64, device=q.device)  # noqa: E731
    tape = [f(3, 6, N), None, f(3, ctrl._qn, N), torch.zeros((3, N), dtype=torch.int32, device=q.device),
            torch.zeros((3, 2, N), dtype=torch.int32, device=q.device)]
    sol, failed = f(ctrl._qn, N), torch.zeros(N, dtype=torch.int32, device=q.device)
    head = lambda steps, h: (h, N, steps, 0.01, p(t), 1, p(q.clone()), None, p(y), 1.0, 1.0, p(sol), p(failed), 0)  # noqa
    assert lib.clik_qp_rollout_tape(*head(-1, skill.handle), *[p(a) for a in tape], None) == 1
    assert b"steps < 0" in lib.clik_last_error()
    assert lib.clik_qp_rollout_tape(*head(3, skill.handle), None, None, *[p(a) for a in tape[2:]], None) == 1
    assert b"required when steps > 0" in lib.clik_last_error()
    out = [f(N), f(6, N), None, f(ctrl._ny, N)]
    sweep = lambda steps, h, tp, o: lib.clik_qp_rollout_vjp(h, N, steps, 0.01, p(t), 1, p(y), 1.0, 1.0,  # noqa
                                                             *[p(a) for a in tp], p(f(6, N)), None, None,
                                                             *[p(a) for a in o], None)
    assert sweep(-1, skill.handle, tape, out) == 1 and b"steps < 0" in lib.clik_last_error()
    assert sweep(3, skill.handle, [None] * 5, out) == 1
    assert sweep(3, skill.handle, tape, [out[0], None, None, out[3]]) == 1
    assert b"q_bar are required" in lib.clik_last_error()
    default = ctrl._skill(0)
    assert sweep(3, default.handle, tape, out) == 1 and b"rollout_vjp=True" in lib.clik_last_error()
    assert lib.clik_qp_rollout_tape(*head(3, default.handle), *[p(a) for a in tape], None) == 1
    cq = _up(np.random.default_rng(79).standard_normal((6, N)))
    assert lib.clik_qp_rollout_vjp(skill.handle, N, 0, 0.01, p(t), 1, p(y), 1.0, 1.0, *([None] * 5), p(cq), None,
                                   None, *[p(a) for a in out], None) == 0
    torch.cuda.synchronize()
    assert torch.equal(out[1], cq) and torch.all(out[0] == 0) and torch.all(out[3] == 0)


def test_missing_virtual_var_raises_before_building(monkeypatch):
    from casclik_b200 import build
    from test_golden_controllers import load_case
    import casclik_b200 as cc
    torch = _torch()
    spec, inp, kwargs, _ = load_case("qp/cart_path")
    ctrl = cc.ReactiveQPController(spec, **kwargs)
    ctrl.setup_solver()
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no image may be built"))
    q = torch.zeros((spec.n_robot_var, 4), dtype=torch.float64, device="cuda")
    for call in (lambda: ctrl.rollout_vjp(0.0, q, 5, 0.01), lambda: ctrl.rollout_batch_differentiable(0.0, q, 5, 0.01)):
        with pytest.raises(ValueError, match="virtual_var"):
            call()
    assert ctrl._rollout_vjp is None
