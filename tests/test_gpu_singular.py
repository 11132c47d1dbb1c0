"""The sm_100a build of the controller steps at and near kinematic singularities: the families of
tests/mp_reference.py with 2^14 draws of the free joints per delta (2^12 for the iiwa, which has seven
families), every instance checked for written outputs and the routes checked against each other, and a
strided subsample (two draws per delta and family) checked against the 50-digit referee with the criterion
of tests/test_singular_on_host.py."""
import numpy as np
import pytest

from casclik_b200 import scenarios
import mp_reference as mr
from test_singular_on_host import OBSERVED, PINV_OPTIONS, check_pinv, check_qp, family_batch

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _dev(inp):
    torch = _torch()
    return {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda())
            for k, v in inp.items() if k != "delta"}


def _sub(inp, draws):
    """Two draws per delta and family: indices and the sub-batch."""
    N = inp["q"].shape[1]
    idx = np.nonzero(np.isin(np.arange(N) % draws, (0, draws // 2)))[0]
    return idx, {k: (None if v is None else v[..., idx]) for k, v in inp.items()}


def _pinv_ref(sc, sub, opts):
    blocks, n = mr.mp_blocks(sc.spec, sub)
    return mr.pinv_reference(blocks, n, opts)


@pytest.mark.parametrize("route", ["split", "one_kernel", "group_all"])
@pytest.mark.parametrize("name", ["ur5_track", "iiwa_multitask"])
def test_pinv_routes_near_singularities_on_the_gpu(name, route, monkeypatch):
    """The routes of test_mode_search_routes_agree_on_the_gpu (fast + group pass, one kernel, sub-warp group
    kernel for everything) at damping 1e-7 and 1e-12: every mode flag in range and every velocity finite on
    the whole batch, and the subsample against the referee.  Each route is checked against the referee, not
    against the other routes: their velocities may differ in the last bits."""
    torch = _torch()
    if route == "one_kernel":
        monkeypatch.setenv("CLIK_PINV_SPLIT", "0")
    if route == "group_all":
        monkeypatch.setenv("CLIK_PINV_GROUP", "1")
    if name == "iiwa_multitask":
        monkeypatch.setenv("CLIK_UNIT_SETS", "0")      # the run-time mode tail, where the routes differ
    sc = scenarios.get(name)
    draws = 1 << (14 if name == "ur5_track" else 12)
    inp, _ = family_batch(sc, draws, seed=5)
    dev = _dev(inp)
    idx, sub = _sub(inp, draws)
    for opts_key in ("lam_1e-7", "lam_1e-12"):
        opts = dict(sc.options or {}, **PINV_OPTIONS[opts_key])
        ctrl = scenarios.get(name).make_controller()
        ctrl.options.update(opts)
        ctrl.setup_solver()
        v, _, mode = ctrl.solve_batch(dev["t"], dev["q"], None, dev["y"])
        torch.cuda.synchronize()
        v, mode = v.cpu().numpy(), mode.cpu().numpy()
        assert np.all((mode >= -1) & (mode < ctrl.n_modes)) and np.isfinite(v).all()
        check_pinv(v[:, idx], mode[idx], _pinv_ref(sc, sub, opts), "gpu %s %s %s" % (name, route, opts_key),
                   ctrl.n_modes)


def test_staged_pinv_kernel_near_singularities_on_the_gpu():
    """The TMA-staged persistent kernel gives the bits of the plain kernel on the singular families."""
    torch = _torch()
    sc = scenarios.get("ur5_track")
    draws = 1 << 14
    inp, _ = family_batch(sc, draws, seed=6)
    dev = _dev(inp)
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    plain = [a.clone() for a in ctrl.solve_batch(dev["t"], dev["q"], None, dev["y"]) if a is not None]
    ctrl.set_input_staging(True)
    staged = [a.clone() for a in ctrl.solve_batch(dev["t"], dev["q"], None, dev["y"]) if a is not None]
    torch.cuda.synchronize()
    for a, b in zip(plain, staged):
        assert torch.equal(a, b)
    idx, sub = _sub(inp, draws)
    check_pinv(staged[0].cpu().numpy()[:, idx], staged[1].cpu().numpy()[idx], _pinv_ref(sc, sub, sc.options),
               "gpu ur5_track staged", ctrl.n_modes)


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_qp_split_and_tail_kernels_near_singularities_on_the_gpu(name, monkeypatch):
    """CLIK_QP_SPLIT 0 / 1 and both tail allocations (CLIK_QP_TAIL_PICK 0 / 1) give the same bits on the
    whole batch; the subsample's minimisers, masks and status against the 50-digit face solution."""
    torch = _torch()
    sc = scenarios.get(name)
    draws = 1 << 14
    inp, _ = family_batch(sc, draws, seed=7)
    dev = _dev(inp)
    outs = {}
    for split, pick in (("1", "0"), ("1", "1"), ("0", "0")):
        monkeypatch.setenv("CLIK_QP_SPLIT", split)
        monkeypatch.setenv("CLIK_QP_TAIL_PICK", pick)
        ctrl = sc.make_controller()
        ctrl.setup_solver()
        outs[split + pick] = [t.clone() for t in ctrl.solve_batch(dev["t"], dev["q"], dev.get("x"), dev.get("y"))]
    torch.cuda.synchronize()
    ref = outs["10"]
    for k, o in outs.items():
        for a, b in zip(ref, o):
            assert torch.equal(a, b), k
    sol, status, active = (t.cpu().numpy() for t in ref[:3])
    assert np.all(status >= 0) and np.isfinite(sol[:, status == 0]).all()
    idx, sub = _sub(inp, draws)
    refs = mr.qp_reference(sc.spec, sub)
    h = mr.qp_mp_problem(sc.spec, {k: (None if v is None else v[..., :1]) for k, v in sub.items()})[0]
    check_qp(sol[:, idx], status[idx], active[:, idx], refs, np.asarray(h, dtype=float), "gpu " + name)


def test_rollout_toward_an_unreachable_target_on_the_gpu():
    """ur5_track chasing targets outside the workspace drives the arm into the stretched (singular) set:
    every instance ends with a finite q, and the device rollout equals a loop of solve_batch bit for bit."""
    torch = _torch()
    sc = scenarios.get("ur5_track")
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    N, K, dt, vmax = 1 << 14, 1000, 0.01, np.pi / 5
    inp = sc.sample(N, seed=8)
    y = torch.from_numpy(np.ascontiguousarray(inp["y"] * 2.5)).cuda()
    q0 = torch.from_numpy(np.ascontiguousarray(inp["q"])).cuda()
    q_roll = q0.clone()
    out = ctrl.rollout_batch(0.0, q_roll, K, dt, input_var=y, max_speed=vmax)
    q_loop = q0.clone()
    for k in range(K):
        v, _, mode = ctrl.solve_batch(dt * k, q_loop, None, y)
        v = torch.clamp(v, -vmax, vmax)          # the rollout reports the clipped command
        q_loop = q_loop + v * dt
    torch.cuda.synchronize()
    assert torch.isfinite(q_roll).all()
    assert torch.equal(q_roll, q_loop) and torch.equal(out["robot_vel"], v) and torch.equal(out["mode"], mode)
    # the arm did stretch: the 50-digit kappa of the position Jacobian at the end is far above the start's
    blocks, _ = mr.mp_blocks(sc.spec, {"t": np.zeros(64), "q": q_roll[:, :64].cpu().numpy(), "y": inp["y"][:, :64] * 2.5})
    b0, _ = mr.mp_blocks(sc.spec, {"t": np.zeros(64), "q": inp["q"][:, :64], "y": inp["y"][:, :64] * 2.5})
    assert np.median(mr.family_kappa(blocks)) > 100 * np.median(mr.family_kappa(b0))


def test_report_observed_maxima_gpu():
    """Runs last in this module: the largest ratios of error to bound, and the instance counts."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items()) if "gpu" in k})
