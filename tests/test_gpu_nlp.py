"""The reactive-NLP controller on the GPU (sm_100a kernels through the C ABI): against the host build of the
same kernel source, between its own entry points, and at scale against the first-order certificate."""
import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import scenarios
from nlp_oracle import Instance, constraint_rows, nlp_kkt_residuals
from test_golden_controllers import QP, load_case
from test_kernel_code_on_host import _host_library
from test_nlp_kernel_on_host import qp_equivalent_cost, random_convex_cost, run_step

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _device_step(ctrl, inp, warm=None, max_iter=None):
    torch = _torch()
    up = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    sol, status, active, iters = ctrl.solve_batch(up(inp["t"]), up(inp["q"]), up(inp.get("x")), up(inp.get("y")),
                                                  warmstart=up(warm), max_iter=max_iter)
    torch.cuda.synchronize()
    return (sol.cpu().numpy(), status.cpu().numpy(), active.cpu().numpy().astype(np.uint32),
            iters.cpu().numpy())


def _cases():
    out = [("qp:" + n) for n in QP] + ["sc:" + n for n in sorted(scenarios.NLP_REGISTRY)] + ["fuzz:0", "fuzz:2", "cost:ytrack", "cost:qweight"]
    return out


def _build(case):
    kind, name = case.split(":")
    if kind == "qp":
        spec, inp, kwargs, _ = load_case(name)
        qc = cc.ReactiveQPController(spec, **kwargs)
        return cc.ReactiveNLPController(spec, qp_equivalent_cost(spec, qc), slack_var_weights=qc.slack_var_weights), inp
    if kind == "sc":
        sc = scenarios.get(name)
        return sc.make_controller(), {k: v for k, v in sc.sample(64, seed=0).items() if v is not None}
    if kind == "cost":                                  # costs that read t / q / y directly
        from test_nlp_costs_on_host import _ur5
        sc, ctrl = _ur5(name)
        inp = {k: v for k, v in sc.sample(64, seed=11).items() if v is not None}
        inp["t"] = np.random.default_rng(12).uniform(-0.5, 0.5, 64)
        return ctrl, inp
    from fuzz_skills import make_qp_skill
    spec, _, inp = make_qp_skill(int(name))
    ctrl = cc.ReactiveNLPController(spec, random_convex_cost(spec, int(name)))
    if spec.virtual_var is not None and spec.n_virtual_var and "x" not in inp:
        inp = dict(inp, x=np.zeros((spec.n_virtual_var, inp["q"].shape[1])))
    return ctrl, inp


@pytest.mark.parametrize("case", _cases())
def test_gpu_matches_the_host_build_of_the_kernel_source(case, tmp_path):
    ctrl, inp = _build(case)
    lib = _host_library(ctrl, tmp_path)
    hs, hst, hit, hact = run_step(lib, ctrl, inp)
    ctrl.setup_problem_functions()                      # the sm_100a build of the same source
    ds, dst, dact, dit = _device_step(ctrl, inp)
    assert np.array_equal(dst, hst)
    ok = hst == 0
    scale = 1.0 + np.abs(hs[:, ok]).max(axis=0) if ok.any() else 1.0
    assert (np.abs(ds[:, ok] - hs[:, ok]).max(axis=0) <= 1e-9 * scale).all()


def test_device_host_and_single_instance_entry_points_agree_bit_for_bit():
    sc = scenarios.get("ur5_nlp_quartic")
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    inp = {k: v for k, v in sc.sample(5000, seed=4).items() if v is not None}
    ds, dst, dact, dit = _device_step(ctrl, inp)
    hs, hst, hact, hit = ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"])
    assert np.array_equal(ds, hs) and np.array_equal(dst, hst) and np.array_equal(dit, hit)
    assert np.array_equal(dact, hact.astype(np.uint32))
    assert np.all(dst == 0)
    for i in (0, 17, 4999):
        rv, vv, sl = ctrl.solve(inp["t"][i], inp["q"][:, i], input_var=inp["y"][:, i])
        got = np.concatenate([rv.toarray().ravel(), sl.toarray().ravel()])
        assert vv is None and np.array_equal(got, ds[:, i])
        assert ctrl.res["status"] == 0 and ctrl.res["iterations"] == dit[i]
        F, _ = Instance(ctrl._prog, inp, i).fg(ds[:, i])
        assert abs(ctrl.res["f"] - F) <= 1e-12 * (1 + abs(F))


def test_rollout_matches_a_loop_of_solve_batch():
    torch = _torch()
    sc = scenarios.get("ur5_nlp_quartic")
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    n, steps, dt, vmax = 512, 12, 0.01, 0.5
    inp = {k: v for k, v in sc.sample(n, seed=6).items() if v is not None}
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    q, y, t0 = dev(inp["q"]), dev(inp["y"]), dev(inp["t"])
    ql, warm, failed = q.clone(), torch.zeros((ctrl._qn, n), dtype=torch.float64, device="cuda"), 0
    for k in range(steps):
        sol, status, _, _ = ctrl.solve_batch(t0 + dt * k, ql, None, y, warmstart=warm)
        bad = status != 0
        failed = failed + bad.to(torch.int32)
        sol[:, bad] = 0.0
        warm = sol.clone()
        ql = ql + torch.clamp(sol[:6], -vmax, vmax) * dt
    qr = q.clone()
    res = ctrl.rollout_batch(t0, qr, steps, dt, input_var=y, max_speed=vmax)
    torch.cuda.synchronize()
    assert torch.equal(res["n_failed"], failed if torch.is_tensor(failed) else torch.zeros_like(res["n_failed"]))
    assert (qr - ql).abs().max().item() <= 1e-9 * (1 + ql.abs().max().item())


@pytest.mark.parametrize("name", sorted(scenarios.NLP_REGISTRY))
def test_scenarios_at_scale(name):
    torch = _torch()
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    N = 1 << 18
    inp = {k: v for k, v in sc.sample(N, seed=0).items() if v is not None}
    sol, status, _, iters = _device_step(ctrl, inp)
    assert np.bincount(status, minlength=6).tolist() == [N, 0, 0, 0, 0, 0]
    idx = np.arange(0, N, 4099)
    sub = {k: (v[..., idx] if k != "t" else v[idx]) for k, v in inp.items()}
    A, lb, ub = constraint_rows(ctrl._prog, sub)
    for k, i in enumerate(idx):
        x = sol[:, i]
        _, g = Instance(ctrl._prog, sub, k).fg(x)
        kk = nlp_kkt_residuals(g, A[k], lb[k], ub[k], x)
        gs = 1.0 + np.abs(g).max()
        assert kk["primal"] < 1e-8 * (1 + np.abs(A[k] @ x).max()), (i, kk)
        assert kk["stationarity"] < 1e-8 * gs and kk["sign"] < 1e-8 * gs, (i, kk)
    if name == "ur5_nlp_taskspeed":
        assert np.all(iters == 1)
    del torch
