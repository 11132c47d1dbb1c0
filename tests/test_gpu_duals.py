"""Constraint multipliers on the GPU (clik_qp_duals / clik_nlp_duals and their host and single-instance forms):
between the entry points, against the host build of the same kernel source, and at scale against the
first-order conditions."""
import numpy as np
import pytest

from casclik_b200 import scenarios
from casclik_b200.sym import dag
from nlp_oracle import _inputs_map, constraint_rows
from test_duals_on_host import host_duals
from test_kernel_code_on_host import _host_library

pytestmark = pytest.mark.gpu

QP_SCENARIOS = ("ur5_qp", "ur5_moe2016_qp")
ALL = QP_SCENARIOS + ("ur5_nlp_taskspeed", "ur5_nlp_quartic")


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _setup(name, N, seed):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    inp = {k: v for k, v in sc.sample(N, seed=seed).items() if v is not None}
    return sc, ctrl, inp


def _up(a):
    torch = _torch()
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _device_step(ctrl, inp):
    """solve_batch + multipliers_batch on CUDA tensors -> NumPy (sol, status, active, lam)."""
    torch = _torch()
    t, q, y = _up(inp["t"]), _up(inp["q"]), _up(inp.get("y"))
    out = ctrl.solve_batch(t, q, None, y)
    sol, status, active = out[0], out[1], out[2]
    lam = ctrl.multipliers_batch(t, q, None, y, sol, status, active)
    torch.cuda.synchronize()
    return (sol.cpu().numpy(), status.cpu().numpy(), active.cpu().numpy().astype(np.uint32), lam.cpu().numpy())


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_device_host_pinned_and_single_instance_agree_bit_for_bit(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 5000, seed=4)
    sol, status, active, lam = _device_step(ctrl, inp)
    assert np.all(status == 0) and np.isfinite(lam).all()
    y = inp.get("y")
    hl = ctrl.multipliers_batch(inp["t"], inp["q"], None, y, sol, status, active.view(np.int32))   # pageable
    assert np.array_equal(hl, lam)
    pin = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    out = pin(np.zeros_like(lam))
    pl = ctrl.multipliers_batch(pin(inp["t"]), pin(inp["q"]), None, pin(y), pin(sol), pin(status),
                                pin(active.view(np.int32)), out=out)                               # page-locked
    assert pl is out and np.array_equal(pl, lam)
    key = "lam_a" if name in QP_SCENARIOS else "lam_g"
    for i in (0, 17, 4999):
        kw = {} if y is None else {"input_var": y[:, i]}
        ctrl.solve(float(inp["t"][i]), inp["q"][:, i], **kw)
        assert np.array_equal(ctrl.res[key].toarray().ravel(), lam[:, i]), i
        assert ctrl.res["lam_x"].shape == (ctrl._qn, 1)


@pytest.mark.parametrize("name", ALL)
def test_gpu_matches_the_host_build_of_the_kernel_source(name, tmp_path):
    sc, ctrl, inp = _setup(name, 512, seed=7)
    sol, status, active, lam = _device_step(ctrl, inp)
    lib = _host_library(ctrl, tmp_path)
    kernel = "clik_qp_duals_kernel" if name in QP_SCENARIOS else "clik_nlp_duals_kernel"
    hl = host_duals(lib, ctrl, inp, sol, status, active, kernel)
    assert np.array_equal(np.isnan(hl), np.isnan(lam))
    ok = ~np.isnan(hl)
    scale = 1.0 + np.abs(np.where(ok, hl, 0.0)).max(axis=0)
    assert (np.abs(np.where(ok, lam - hl, 0.0)).max(axis=0) <= 1e-9 * scale).all()


def _gradients(ctrl, inp, sol):
    """(g (N, n), A (N, m, n), lb, ub) of every instance: H x for the QP, grad F for the NLP, evaluated by the
    expression interpreter over the whole batch."""
    qp = not hasattr(ctrl, "_prog")
    prog = ctrl._program() if qp else ctrl._prog
    A, lb, ub = constraint_rows(prog, inp)
    vals = _inputs_map(prog, inp)
    N = sol.shape[1]
    if qp:
        h = np.stack([np.broadcast_to(np.asarray(v, dtype=np.float64), (N,)) for v in dag.evaluate(prog.h, vals)], 1)
        return h * sol.T, A, lb, ub
    vals.update({n.id: sol[j] for j, n in enumerate(prog.dec)})
    g = np.stack([np.broadcast_to(np.asarray(v, dtype=np.float64), (N,)) for v in dag.evaluate(list(prog.g), vals)], 1)
    return g, A, lb, ub


@pytest.mark.parametrize("name", ALL)
def test_every_solved_instance_at_scale_satisfies_the_first_order_conditions(name):
    N = 1 << 18
    sc, ctrl, inp = _setup(name, N, seed=0)
    sol, status, active, lam = _device_step(ctrl, inp)
    solved = status == 0
    assert solved.sum() > 0.99 * N
    assert np.isnan(lam[:, ~solved]).all()
    g, A, lb, ub = _gradients(ctrl, inp, sol)
    L = lam.T
    assert np.isfinite(L[solved]).all()
    res = np.abs(g + np.einsum("imn,im->in", A, L)).max(axis=1)
    tol = (1e-9 if name in QP_SCENARIOS else 1e-6) * (1.0 + np.abs(g).max(axis=1))
    bad = solved & ~(res <= tol)
    assert not bad.any(), (np.nonzero(bad)[0][:5], res[bad][:5])
    m = lam.shape[0]
    bits = np.arange(m, dtype=np.uint32)
    up = ((active[0][:, None] >> bits) & 1).astype(bool)
    lo = ((active[1][:, None] >> bits) & 1).astype(bool)
    assert np.all(L[solved][~(up | lo)[solved]] == 0.0)
    eq = lb == ub
    slack = 1e-9 * (1.0 + np.abs(np.nan_to_num(L)).max(axis=1, keepdims=True))
    assert np.all((L >= -slack)[solved][(up & ~eq)[solved]])
    assert np.all((L <= slack)[solved][(lo & ~eq)[solved]])


@pytest.mark.parametrize("name", ["ur5_moe2016_qp", "ur5_nlp_taskspeed"])
def test_solve_batch_is_unchanged_by_a_multipliers_call(name):
    torch = _torch()
    sc, ctrl, inp = _setup(name, 70001, seed=5)
    t, q, y = _up(inp["t"]), _up(inp["q"]), _up(inp.get("y"))
    first = [a.clone() for a in ctrl.solve_batch(t, q, None, y)]
    keep = [a.clone() for a in first[:3]]
    ctrl.multipliers_batch(t, q, None, y, first[0], first[1], first[2])
    again = ctrl.solve_batch(t, q, None, y)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(first, again))
    assert all(torch.equal(a, b) for a, b in zip(first[:3], keep))      # the step's outputs are only read
