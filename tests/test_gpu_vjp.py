"""Reverse-mode derivative of the QP and NLP steps on the GPU (vjp_batch, solve_batch_differentiable): against the
host build of the same kernel source, against finite differences of the device step at 2^16 instances, through
torch autograd, and with the step and multiplier outputs unchanged by the VJP image."""
import numpy as np
import pytest

from casclik_b200 import runtime, scenarios
from test_vjp_on_host import host_step, host_vjp, theta_rows, vjp_library

pytestmark = pytest.mark.gpu

QP_SCENARIOS = ("ur5_qp", "ur5_moe2016_qp")
ALL = QP_SCENARIOS + ("ur5_nlp_taskspeed", "ur5_nlp_quartic")


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _up(a):
    torch = _torch()
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _setup(name, N, seed):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    inp = {k: v for k, v in sc.sample(N, seed=seed).items() if v is not None}
    return sc, ctrl, inp


def _dev_inputs(ctrl, inp):
    x = inp.get("x")
    if ctrl._nxv and x is None:
        x = np.zeros((ctrl._nxv, inp["q"].shape[1]))
    return _up(inp["t"]), _up(inp["q"]), _up(x), _up(inp.get("y") if ctrl._ny else None)


def _theta_bar(out):
    return np.vstack([out[0].cpu().numpy()[None]] + [a.cpu().numpy() for a in out[1:] if a is not None])


@pytest.mark.parametrize("name", ALL)
def test_device_vjp_agrees_with_the_host_build(name, tmp_path):
    sc, ctrl, inp = _setup(name, 512, seed=21)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    sb = np.random.default_rng(3).standard_normal((ctrl._qn, 512))
    sb[:, 7] = 0.0
    dev = _theta_bar(ctrl.vjp_batch(t, q, x, y, sol, status, active, _up(sb)))
    hc = sc.make_controller()
    lib = vjp_library(hc, tmp_path)
    _, full = theta_rows(hc, inp)
    hs, hst, hact = sol.cpu().numpy(), status.cpu().numpy(), active.cpu().numpy().astype(np.uint32)
    host = host_vjp(lib, hc, kind, full, hs, hst, hact, sb)
    assert np.all(hst == 0) and np.all(dev[:, 7] == 0.0)
    err = np.abs(dev - host).max(axis=0) / (1 + np.abs(host).max(axis=0))
    print("%s: max relative deviation device vs host %.2e" % (name, err.max()))
    assert err.max() <= 1e-12


@pytest.mark.parametrize("name", ALL)
def test_device_finite_differences_at_2_16(name):
    torch = _torch()
    N = 1 << 16
    sc, ctrl, inp = _setup(name, N, seed=22)
    qp = name in QP_SCENARIOS
    rel, tol = (1e-6, 1e-6) if qp else (1e-4, 1e-4)     # the steps and stencils of test_vjp_on_host.fd_check
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    sb = torch.randn((ctrl._qn, N), dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    got = _theta_bar(ctrl.vjp_batch(t, q, x, y, sol, status, active, sb))
    base = {"t": t, "q": q, "x": x, "y": y}
    rows = [("t", None)] + [("q", j) for j in range(q.shape[0])]
    rows += [("x", j) for j in range(ctrl._nxv)] + [("y", j) for j in range(ctrl._ny)]
    scale = torch.from_numpy(1 + np.abs(got).max(axis=0)).cuda()
    counted, worst = 0, 0.0
    for k, (key, row) in enumerate(rows):
        val = base[key] if row is None else base[key][row]
        h = rel * torch.clamp(val.abs(), min=1.0)
        same = status == 0
        f = {}
        for step in ((1, -1) if qp else (1, -1, 2, -2, 0.01, -0.01, 0.001, -0.001)):
            inp2 = {kk: (vv.clone() if vv is not None else None) for kk, vv in base.items()}
            if row is None:
                inp2[key] = inp2[key] + step * h
            else:
                inp2[key][row] += step * h
            sp, stp, ap = ctrl.solve_batch(inp2["t"], inp2["q"], inp2["x"], inp2["y"])[:3]
            same &= (stp == 0) & torch.all(ap == active, dim=0)
            f[step] = (sb * sp).sum(dim=0)
        g = torch.from_numpy(got[k]).cuda()
        if qp:
            err = ((f[1] - f[-1]) / (2 * h) - g).abs() / scale
            ok = err <= tol
        else:
            # as test_vjp_on_host.fd_check: the fourth-order quotient at h, or a central one at h/100 or h/1000
            err = ((8 * (f[1] - f[-1]) - (f[2] - f[-2])) / (12 * h) - g).abs() / scale
            ok = err <= tol
            for r in (0.01, 0.001):
                ok |= ((f[r] - f[-r]) / (2 * r * h) - g).abs() / scale <= tol
        if bool(same.any()):
            worst = max(worst, float(err[same].max()))
            bad = torch.nonzero(same & ~ok).flatten()
            assert bad.numel() == 0, (key, row, bad[:5].tolist(), err[bad[:5]].tolist())
        counted += int((same & (err <= tol)).sum())
    print("%s: %d stable (instance, theta entry) pairs of %d, largest relative deviation %.2e"
          % (name, counted, N * len(rows), worst))
    assert counted >= N * len(rows) // 4


@pytest.mark.parametrize("name", ALL)
def test_autograd_gradients_equal_vjp_batch(name):
    torch = _torch()
    N = 4096
    sc, ctrl, inp = _setup(name, N, seed=23)
    t, q, x, y = _dev_inputs(ctrl, inp)
    ts = t.clone().requires_grad_(True)
    qs = q.clone().requires_grad_(True)
    ys = y.clone().requires_grad_(True) if y is not None else None
    xs = x.clone().requires_grad_(True) if x is not None else None
    w = torch.rand((ctrl._qn, N), dtype=torch.float64, device="cuda")
    sol, status, active = ctrl.solve_batch_differentiable(ts, qs, xs, ys)[:3]
    assert not status.requires_grad and not active.requires_grad
    assert torch.equal(sol, ctrl.solve_batch(t, q, x, y)[0])
    for weight in (torch.ones_like(w), w):
        for a in (ts, qs, xs, ys):
            if a is not None:
                a.grad = None
        sol = ctrl.solve_batch_differentiable(ts, qs, xs, ys)[0]
        (sol * weight).sum().backward()
        ref = ctrl.vjp_batch(t, q, x, y, sol.detach(), status, active, weight.contiguous())
        assert torch.equal(ts.grad, ref[0]) and torch.equal(qs.grad, ref[1])
        if ys is not None:
            assert torch.equal(ys.grad, ref[3])
    # a shared (0-d) t gets the summed t_bar
    t0 = torch.tensor(float(inp["t"][0]), dtype=torch.float64, device="cuda", requires_grad=True)
    sol = ctrl.solve_batch_differentiable(t0, q, x, y)[0]
    sol.sum().backward()
    out = ctrl.solve_batch(t0.detach(), q, x, y)
    ref = ctrl.vjp_batch(t0.detach(), q, x, y, out[0], out[1], out[2], torch.ones_like(out[0]))
    assert torch.allclose(t0.grad, ref[0].sum(), rtol=1e-12, atol=0)


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed"])
def test_gradcheck_on_stable_instances(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 64, seed=24)
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    qp = name in QP_SCENARIOS
    eps = 1e-6 if qp else 1e-4
    # instances whose working set stays the same under gradcheck's perturbations of q
    keep = status == 0
    for j in range(q.shape[0]):
        for s in (-eps, eps):
            q2 = q.clone()
            q2[j] += s
            s2, st2, a2 = ctrl.solve_batch(t, q2, x, y)[:3]
            keep &= (st2 == 0) & torch.all(a2 == active, dim=0)
    idx = torch.nonzero(keep).flatten()[:6]
    assert idx.numel() >= 3
    qk = q[:, idx].contiguous().requires_grad_(True)
    tk = t[idx].contiguous()
    yk = y[:, idx].contiguous() if y is not None else None

    def f(qv):
        return ctrl.solve_batch_differentiable(tk, qv, None, yk)[0]
    assert torch.autograd.gradcheck(f, (qk,), eps=eps, atol=1e-5 if qp else 1e-4, rtol=1e-4)


@pytest.mark.parametrize("name", ALL)
def test_step_and_multipliers_unchanged_by_the_vjp_image(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 15, seed=25)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    t, q, x, y = _dev_inputs(ctrl, inp)
    before = [a.clone() for a in ctrl.solve_batch(t, q, x, y)]
    lam0 = ctrl.multipliers_batch(t, q, x, y, *before[:3])
    ctrl.vjp_batch(t, q, x, y, before[0], before[1], before[2], torch.ones_like(before[0]))
    after = ctrl.solve_batch(t, q, x, y)
    for a, b in zip(before, after):
        assert torch.equal(a, b)
    # the same step and multipliers from the VJP image's own kernels
    vsk = ctrl._vjp["skills"][q.device.index]
    lib = runtime.load_library()
    stream = torch.cuda.current_stream().cuda_stream
    N = q.shape[1]
    sol, status, active = torch.empty_like(before[0]), torch.empty_like(before[1]), torch.empty_like(before[2])
    ptr = lambda a: None if a is None else a.data_ptr()  # noqa: E731
    tp, qp, xp, yp = ptr(t), ptr(q), ptr(x), ptr(y)
    if kind == "qp":
        runtime.check(lib.clik_qp_step(vsk.handle, N, tp, 1, qp, xp, yp, None, None, sol.data_ptr(),
                                       status.data_ptr(), active.data_ptr(), 0, stream))
    else:
        iters = torch.empty_like(before[3])
        runtime.check(lib.clik_nlp_step(vsk.handle, N, tp, 1, qp, xp, yp, None, sol.data_ptr(), status.data_ptr(),
                                        iters.data_ptr(), active.data_ptr(), ctrl._max_iter(None), stream))
    lam = torch.empty_like(lam0)
    runtime.check(getattr(lib, "clik_%s_duals" % kind)(vsk.handle, N, tp, 1, qp, xp, yp, sol.data_ptr(),
                                                        status.data_ptr(), active.data_ptr(), lam.data_ptr(), stream))
    torch.cuda.synchronize()
    assert torch.equal(sol, before[0]) and torch.equal(status, before[1]) and torch.equal(active, before[2])
    assert torch.equal(lam.nan_to_num(7.0), lam0.nan_to_num(7.0))


def test_validation_and_images_without_the_kernel():
    torch = _torch()
    sc, ctrl, inp = _setup("ur5_qp", 64, seed=26)
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)
    sb = torch.ones_like(sol)
    N = 64
    bad_sol_bar = [sb[:, :-1].contiguous(), sb.float(), sb.t().contiguous().t(), sb.cpu()]
    for b in bad_sol_bar:
        with pytest.raises((runtime.ClikError, ValueError)):
            ctrl.vjp_batch(t, q, x, y, sol, status, active, b)
    good = [torch.empty(N, dtype=torch.float64, device="cuda"), torch.empty((6, N), dtype=torch.float64, device="cuda"),
            None, torch.empty((ctrl._ny, N), dtype=torch.float64, device="cuda")]
    out = ctrl.vjp_batch(t, q, x, y, sol, status, active, sb, out=good)
    assert all(a is b for a, b in zip(out, good))
    for k, bad in ((0, torch.empty(N + 1, dtype=torch.float64, device="cuda")),
                   (1, torch.empty((6, N), dtype=torch.float32, device="cuda")),
                   (1, torch.empty((N, 6), dtype=torch.float64, device="cuda").t()),
                   (3, torch.empty((ctrl._ny, N), dtype=torch.float64)),
                   (1, None)):
        o = list(good)
        o[k] = bad
        with pytest.raises(runtime.ClikError):
            ctrl.vjp_batch(t, q, x, y, sol, status, active, sb, out=o)
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.vjp_batch(inp["t"], inp["q"], None, inp["y"], sol.cpu().numpy(), status.cpu().numpy(),
                       active.cpu().numpy(), sb.cpu().numpy())
    # the default image has no VJP kernel: the ABI call fails, nothing is launched
    lib = runtime.load_library()
    sk = ctrl._skill(q.device.index)
    st = lib.clik_qp_vjp(sk.handle, N, t.data_ptr(), 1, q.data_ptr(), None, y.data_ptr(), sol.data_ptr(),
                         status.data_ptr(), active.data_ptr(), sb.data_ptr(), good[0].data_ptr(), good[1].data_ptr(),
                         None, good[3].data_ptr(), None)
    assert st == 1 and b"no QP VJP kernel" in lib.clik_last_error()
    vsk = ctrl._vjp["skills"][q.device.index]
    st = lib.clik_nlp_vjp(vsk.handle, N, t.data_ptr(), 1, q.data_ptr(), None, y.data_ptr(), sol.data_ptr(),
                          status.data_ptr(), active.data_ptr(), sb.data_ptr(), good[0].data_ptr(), good[1].data_ptr(),
                          None, good[3].data_ptr(), None)
    assert st == 1 and b"no NLP VJP kernel" in lib.clik_last_error()
