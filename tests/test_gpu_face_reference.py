"""The sm_100a build of the NLP step, the multipliers and the QP / NLP VJP on the singular families: 2^14 draws of the
free joints per delta and family through solve_batch, multipliers_batch and vjp_batch.  Every output of the whole
batch must be written (finite, or NaN where the rules allow it), an all-zero cotangent must give exactly 0 everywhere,
and a strided subsample (one draw per delta and family) is checked against the 50-digit referee with the criteria of
tests/test_face_reference_on_host.py.  On one family batch, solve_batch_differentiable(...).backward() must equal
vjp_batch bit for bit."""
import numpy as np
import pytest

from test_face_reference_on_host import EPS, OBSERVED, check_outputs, make_case
from test_singular_on_host import family_batch

pytestmark = pytest.mark.gpu
DRAWS = 1 << 14
SENTINEL = 12345.678
COUNTS = {}


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _dev(ctrl, inp):
    torch = _torch()
    up = (lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda())
    x = inp.get("x")
    if ctrl._nxv and x is None:
        x = np.zeros((ctrl._nxv, inp["q"].shape[1]))
    return up(inp["t"]), up(inp["q"]), up(x), up(inp.get("y") if ctrl._ny else None)


def _theta_bar(out):
    return np.vstack([out[0].cpu().numpy()[None]] + [a.cpu().numpy() for a in out[1:] if a is not None])


CASES = ["ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic", "moe2016_taskspeed", "quartic_offset",
         "offaxis_eps_0"] + ["eps_%g" % e for e in EPS]
SINGULAR_HESSIAN = ("eps_0", "offaxis_eps_0")     # lambda_min(grad^2 F) = 0 on every instance: the band requires NaN


@pytest.mark.parametrize("name", CASES)
def test_face_reference_on_the_gpu(name):
    torch = _torch()
    kind, sc, ctrl = make_case(name)
    ctrl.setup_solver()
    inp, _ = family_batch(sc, DRAWS, seed=11)
    inp = {k: v for k, v in inp.items() if v is not None and k != "delta"}
    t, q, x, y = _dev(ctrl, inp)
    out = ctrl.solve_batch(t, q, x, y)
    sol, status, active = out[0], out[1], out[2]
    N = sol.shape[1]
    lam = ctrl.multipliers_batch(t, q, x, y, sol, status, active,
                                 out=torch.full((ctrl._qm, N), SENTINEL, dtype=torch.float64, device="cuda"))
    xb = torch.randn(sol.shape, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    rows = (1, q.shape[0], ctrl._nxv, ctrl._ny)
    bufs = [torch.full((r, N), SENTINEL, dtype=torch.float64, device="cuda") if r else None for r in rows]
    bufs[0] = bufs[0][0]
    tb = _theta_bar(ctrl.vjp_batch(t, q, x, y, sol, status, active, xb, out=bufs))
    zero = _theta_bar(ctrl.vjp_batch(t, q, x, y, sol, status, active, torch.zeros_like(sol)))
    torch.cuda.synchronize()
    sol, status, active, lam = sol.cpu().numpy(), status.cpu().numpy(), active.cpu().numpy(), lam.cpu().numpy()
    assert not (lam == SENTINEL).any() and not (tb == SENTINEL).any(), "outputs not written"
    assert np.all(zero == 0.0), "an all-zero cotangent must give exactly 0"
    assert np.all(np.isin(status, (0, 1, 2, 4, 5)))
    ok = status == 0
    assert np.isfinite(sol[:, ok]).all()
    for a in (lam, tb):        # per instance: finite, or NaN in every entry; NaN wherever the step is not solved
        col_nan = np.isnan(a).any(axis=0)
        assert np.all(col_nan == np.isnan(a).all(axis=0)) and np.isfinite(a[:, ~col_nan]).all()
        assert col_nan[~ok].all()
    if name in SINGULAR_HESSIAN:
        assert np.isnan(tb[:, ok]).all(), "finite theta_bar on a singular Hessian"
    COUNTS[name] = "%d solved of %d, NaN theta_bar on %d of them" % (ok.sum(), N, np.isnan(tb[:, ok]).any(axis=0).sum())
    idx = np.nonzero(np.arange(N) % DRAWS == 0)[0]
    if name.startswith(("eps_", "offaxis")):
        idx = idx[::4]
    sub = {k: (v[..., idx] if k != "t" else v[idx]) for k, v in inp.items()}
    sl = np.ascontiguousarray
    check_outputs("gpu " + name, kind, ctrl, sub, sl(sol[:, idx]), sl(status[idx]), sl(active[:, idx]),
                  sl(lam[:, idx]), xb.cpu().numpy()[:, idx], sl(tb[:, idx]))


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_taskspeed"])
def test_autograd_equals_vjp_batch_on_a_family_batch(name):
    torch = _torch()
    kind, sc, ctrl = make_case(name)
    ctrl.setup_solver()
    inp, _ = family_batch(sc, 1 << 10, seed=12)
    inp = {k: v for k, v in inp.items() if v is not None and k != "delta"}
    t, q, x, y = _dev(ctrl, inp)
    qs, ys = q.clone().requires_grad_(True), y.clone().requires_grad_(True)
    ts = t.clone().requires_grad_(True)
    sol, status, active = ctrl.solve_batch_differentiable(ts, qs, None, ys)[:3]
    w = torch.rand(sol.shape, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    w[:, ::7] = 0.0                           # masked instances, solved or not, contribute exactly 0
    (sol * w).sum().backward()
    ref = ctrl.vjp_batch(t, q, x, y, sol.detach(), status, active, w.contiguous())
    torch.cuda.synchronize()
    for got, want in ((ts.grad, ref[0]), (qs.grad, ref[1]), (ys.grad, ref[3])):
        assert torch.equal(got.nan_to_num(7.0), want.nan_to_num(7.0))
        assert torch.equal(torch.isnan(got), torch.isnan(want))


def test_report_observed_maxima_gpu():
    """Runs last in this module: the largest ratios of error to bound, and the instance counts."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items()) if "gpu" in k})
    print("instances:", COUNTS)
