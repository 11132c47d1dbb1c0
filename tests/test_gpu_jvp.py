"""Forward-mode derivative and Jacobian of the QP and NLP steps on the GPU (jvp_batch, jacobian_batch, torch forward
AD through solve_batch_differentiable): against the host build of the same kernel source, against directional finite
differences of the device step at 2^16 instances, against vjp_batch through the adjoint identity at 2^18, and with
the step and VJP outputs unchanged by the JVP image."""
import numpy as np
import pytest

from casclik_b200 import scenarios
from test_face_reference_on_host import family_sub
from test_gpu_vjp import ALL, QP_SCENARIOS, _dev_inputs, _setup, _theta_bar, _torch, _up
from test_jvp_on_host import _split, host_jac, host_jvp, jvp_library, tangents
from test_vjp_on_host import theta_rows

pytestmark = pytest.mark.gpu


def _tangent_tensors(ctrl, td):
    return [_up(a) if a is not None else None for a in _split(ctrl, td)]


@pytest.mark.parametrize("name", ALL)
def test_device_jvp_and_jacobian_agree_with_the_host_build(name, tmp_path):
    sc, ctrl, inp = _setup(name, 512, seed=41)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    td = tangents(ctrl, inp, 5)
    td[:, 7] = 0.0
    tdt = _tangent_tensors(ctrl, td)
    dev = ctrl.jvp_batch(t, q, x, y, sol, status, active, *tdt).cpu().numpy()
    djac = ctrl.jacobian_batch(t, q, x, y, sol, status, active).cpu().numpy()
    hc = sc.make_controller()
    lib = jvp_library(hc, tmp_path)
    _, full = theta_rows(hc, inp)
    hs, hst, hact = sol.cpu().numpy(), status.cpu().numpy(), active.cpu().numpy().astype(np.uint32)
    host = host_jvp(lib, hc, kind, full, hs, hst, hact, td)
    hjac = host_jac(lib, hc, kind, full, hs, hst, hact)
    assert np.all(hst == 0) and np.all(dev[:, 7] == 0.0)
    err = np.abs(dev - host).max(axis=0) / (1 + np.abs(host).max(axis=0))
    ejac = np.abs(djac - hjac).max(axis=(0, 1)) / (1 + np.abs(hjac).max(axis=(0, 1)))
    print("%s: max relative deviation device vs host: JVP %.2e, Jacobian %.2e" % (name, err.max(), ejac.max()))
    assert err.max() <= 1e-12 and ejac.max() <= 1e-12


@pytest.mark.parametrize("name", ALL)
def test_device_directional_finite_differences_at_2_16(name):
    torch = _torch()
    N = 1 << 16
    sc, ctrl, inp = _setup(name, N, seed=42)
    qp = name in QP_SCENARIOS
    rel, tol = (1e-6, 1e-6) if qp else (1e-4, 1e-4)     # the steps and stencils of test_vjp_on_host.fd_check
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    # direction: each entry of theta moves by at most the step of fd_check, rel max(1, |theta_k|)
    theta = np.vstack([inp["t"][None]] + [inp[k] for k in "qxy" if k in inp])
    td = tangents(ctrl, inp, 6)
    td = td / np.abs(td).max(axis=0) * np.maximum(1.0, np.abs(theta))
    tdt = _tangent_tensors(ctrl, td)
    got = ctrl.jvp_batch(t, q, x, y, sol, status, active, *tdt)
    scale = 1 + got.abs().amax(dim=0)
    base = [t, q, x, y]
    h = rel
    same = status == 0
    f = {}
    for step in ((1, -1) if qp else (1, -1, 2, -2, 0.01, -0.01, 0.001, -0.001)):
        moved = [None if a is None else a + step * h * d for a, d in zip(base, tdt)]
        sp, stp, ap = ctrl.solve_batch(*moved)[:3]
        same &= (stp == 0) & torch.all(ap == active, dim=0)
        f[step] = sp
    if qp:
        err = ((f[1] - f[-1]) / (2 * h) - got).abs().amax(dim=0) / scale
        ok = err <= tol
    else:
        err = ((8 * (f[1] - f[-1]) - (f[2] - f[-2])) / (12 * h) - got).abs().amax(dim=0) / scale
        ok = err <= tol
        for r in (0.01, 0.001):
            ok |= ((f[r] - f[-r]) / (2 * r * h) - got).abs().amax(dim=0) / scale <= tol
    bad = torch.nonzero(same & ~ok).flatten()
    print("%s: %d stable instances of %d, largest relative deviation %.2e"
          % (name, int(same.sum()), N, float(err[same].max())))
    assert bad.numel() == 0, (bad[:5].tolist(), err[bad[:5]].tolist())
    assert int(same.sum()) >= N // 4


@pytest.mark.parametrize("name", ALL)
def test_adjoint_identity_against_vjp_batch_at_2_18(name):
    torch = _torch()
    N = 1 << 18
    sc, ctrl, inp = _setup(name, N, seed=43)
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    g = torch.Generator("cuda").manual_seed(7)
    td = torch.randn((len(theta_rows(ctrl, {k: v[..., :1] for k, v in inp.items()})[0]), N), dtype=torch.float64,
                     device="cuda", generator=g)
    xb = torch.randn((ctrl._qn, N), dtype=torch.float64, device="cuda", generator=g)
    nq = q.shape[0]
    parts = [td[0].contiguous(), td[1:1 + nq].contiguous(), td[1 + nq:1 + nq + ctrl._nxv].contiguous() if ctrl._nxv
             else None, td[1 + nq + ctrl._nxv:].contiguous() if ctrl._ny else None]
    xd = ctrl.jvp_batch(t, q, x, y, sol, status, active, *parts)
    tb = torch.from_numpy(_theta_bar(ctrl.vjp_batch(t, q, x, y, sol, status, active, xb))).cuda()
    fin = torch.isfinite(xd).all(dim=0)
    assert torch.equal(fin, torch.isfinite(tb).all(dim=0))
    lhs, rhs = (xb * xd).sum(dim=0)[fin], (tb * td).sum(dim=0)[fin]
    scale = (xb.norm(dim=0) * xd.norm(dim=0) + tb.norm(dim=0) * td.norm(dim=0))[fin]
    gap = (lhs - rhs).abs() / torch.where(scale > 0, scale, torch.ones_like(scale))
    print("%s: %d finite instances, largest adjoint gap %.2e" % (name, int(fin.sum()), float(gap.max())))
    assert float(gap.max()) <= 1e-12 and int(fin.sum()) >= N // 2


@pytest.mark.parametrize("name", ALL)
def test_forward_ad_equals_jvp_batch(name):
    torch = _torch()
    import torch.autograd.forward_ad as fwAD
    N = 4096
    sc, ctrl, inp = _setup(name, N, seed=44)
    t, q, x, y = _dev_inputs(ctrl, inp)
    g = torch.Generator("cuda").manual_seed(9)
    qd = torch.randn(q.shape, dtype=torch.float64, device="cuda", generator=g)
    yd = torch.randn(y.shape, dtype=torch.float64, device="cuda", generator=g) if y is not None else None
    t0 = torch.tensor(float(inp["t"][0]), dtype=torch.float64, device="cuda")
    for tt, tdot in ((t, torch.randn(t.shape, dtype=torch.float64, device="cuda", generator=g)),
                     (t0, torch.tensor(0.3, dtype=torch.float64, device="cuda"))):
        with fwAD.dual_level():
            outs = ctrl.solve_batch_differentiable(fwAD.make_dual(tt, tdot), fwAD.make_dual(q, qd), x,
                                                   None if y is None else fwAD.make_dual(y, yd))
            sol_dot = fwAD.unpack_dual(outs[0]).tangent
            assert all(fwAD.unpack_dual(o).tangent is None for o in outs[1:])
            sol, status, active = [fwAD.unpack_dual(o).primal for o in outs[:3]]
        ref = ctrl.jvp_batch(tt, q, x, y, sol, status, active, t_dot=tdot, q_dot=qd, y_dot=yd)
        assert torch.equal(sol_dot.nan_to_num(7.0), ref.nan_to_num(7.0))


@pytest.mark.parametrize("name", ALL)
def test_step_and_vjp_unchanged_by_the_jvp_image(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 1 << 15, seed=45)
    t, q, x, y = _dev_inputs(ctrl, inp)
    before = [a.clone() for a in ctrl.solve_batch(t, q, x, y)]
    ones = torch.ones_like(before[0])
    vjp0 = [a.clone() if a is not None else None for a in ctrl.vjp_batch(t, q, x, y, *before[:3], ones)]
    ctrl.jacobian_batch(t, q, x, y, *before[:3])
    assert ctrl._jvp is not None
    after = ctrl.solve_batch(t, q, x, y)
    for a, b in zip(before, after):
        assert torch.equal(a, b)
    vjp1 = ctrl.vjp_batch(t, q, x, y, *before[:3], ones)
    for a, b in zip(vjp0, vjp1):
        assert (a is None and b is None) or torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0))


@pytest.mark.parametrize("name", ALL)
def test_face_reference_families_device_jacobian(name, tmp_path):
    """A strided subsample of the singular families: the device Jacobian equals the host build, whose Jacobian
    test_jvp_on_host checks against the 50-digit face derivative, within 1e-12, with the same NaN instances."""
    sc, ctrl, _ = _setup(name, 1, seed=0)
    kind = "qp" if name in QP_SCENARIOS else "nlp"
    inp, _ = family_sub(sc, 7)
    t, q, x, y = _dev_inputs(ctrl, inp)
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    djac = ctrl.jacobian_batch(t, q, x, y, sol, status, active).cpu().numpy()
    hc = sc.make_controller()
    lib = jvp_library(hc, tmp_path)
    _, full = theta_rows(hc, inp)
    hjac = host_jac(lib, hc, kind, full, sol.cpu().numpy(), status.cpu().numpy(),
                    active.cpu().numpy().astype(np.uint32))
    nan = np.isnan(hjac).any(axis=(0, 1))
    assert np.array_equal(nan, np.isnan(djac).any(axis=(0, 1)))
    err = np.abs(djac - hjac)[:, :, ~nan].max(axis=(0, 1)) / (1 + np.abs(hjac[:, :, ~nan]).max(axis=(0, 1)))
    print("%s: %d family instances, %d NaN, max relative deviation %.2e" % (name, nan.size, nan.sum(), err.max()))
    assert err.max() <= 1e-12


def test_one_step_closed_loop_jacobian():
    """q_{k+1} = q_k + dt qdot(q_k): I + dt dqdot/dq from jacobian_batch against a central difference of
    rollout_batch(steps=1) on instances that keep their working set and stay below the speed clip."""
    torch = _torch()
    N = 4096
    sc, ctrl, inp = _setup("ur5_qp", N, seed=46)
    t, q, x, y = _dev_inputs(ctrl, inp)
    dt, vmax, h = 0.008, 1e3, 1e-6
    sol, status, active = ctrl.solve_batch(t, q, x, y)[:3]
    jac = ctrl.jacobian_batch(t, q, x, y, sol, status, active)
    nq = q.shape[0]
    same = (status == 0) & (sol[:nq].abs() < vmax).all(dim=0)
    for j in range(nq):
        cols = []
        for s in (1, -1):
            q2 = q.clone()
            q2[j] += s * h
            st2, a2 = ctrl.solve_batch(t, q2, x, y)[1:3]
            same &= (st2 == 0) & torch.all(a2 == active, dim=0)
            qr = q2.clone()
            ctrl.rollout_batch(t, qr, steps=1, dt=dt, input_var=y, max_speed=vmax)
            cols.append(qr)
        fd = (cols[0] - cols[1]) / (2 * h)
        want = dt * jac[:nq, 1 + j, :]
        want[j] += 1.0
        err = (fd - want).abs().amax(dim=0)
        assert float(err[same].max()) <= 1e-6, float(err[same].max())
    assert int(same.sum()) >= N // 4
