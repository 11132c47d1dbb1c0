"""Host-array routes of every step kind give the bits of the device-resident call on the same inputs.

Routes: pageable arrays (chunked copy pipeline), every array page-locked (zero copy), page-locked inputs with
pageable outputs (back to the pipeline), two handles of one cubin on device 0 through clik_*_step_host_multi,
optional outputs omitted, QP host warm starts, and multipliers_batch on host arrays.  The pinv and QP batches span
five pipeline chunks (4 * 2^17 + 4321 instances), so a scratch slot is reused and the last chunk is ragged."""
import ctypes

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import cs, runtime, scenarios

pytestmark = pytest.mark.gpu
vp = ctypes.c_void_p

N_CHUNKS = 4 * (1 << 17) + 4321
N_NLP = (1 << 18) + 4321


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _up(a):
    return None if a is None else _torch().from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _down(a):
    return None if a is None else a.cpu().numpy()


def _pin(a):
    return None if a is None else _torch().from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def _ptr(a):
    return None if a is None else vp(a.ctypes.data)


def _same(a, b):
    assert len(a) == len(b)
    return all((x is None and y is None) or np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True)
               for x, y in zip(a, b))


def _cart_spec(velocity_row=True):
    """Cart path-following skill of the notebooks (virtual path variable x), as in test_gpu_pinv.  The QP variant
    leaves out the hard velocity equality: with it, every sampled instance is infeasible."""
    t, p, dp = cs.MX.sym("t"), cs.MX.sym("p"), cs.MX.sym("dp")
    x, dx = cs.MX.sym("x"), cs.MX.sym("dx")
    up = cc.EqualityConstraint("move_up_path_cnstr", 300 - x, gain=1.0, priority=1)
    lim = cc.SetConstraint("cart_limit_cnstr", p, gain=1.0, set_min=0.0, set_max=1.0, priority=1)
    dist = cc.EqualityConstraint("min_dist_cnstr", 0.4 * cs.sin(0.3 * x) - p, gain=1.0,
                                 constraint_type="soft", priority=3)
    cons = [up, dist, lim]
    if velocity_row:
        cons.append(cc.VelocityEqualityConstraint("drift", p + 0.1 * x, target=0.05, priority=4))
    return cc.SkillSpecification("path", t, p, robot_vel_var=dp, virtual_var=x, virtual_vel_var=dx, constraints=cons)


def _cart_inputs(N, seed):
    rng = np.random.default_rng(seed)
    return {"t": rng.uniform(0, 1, N), "q": rng.uniform(-0.2, 1.2, (1, N)), "x": rng.uniform(0, 20, (1, N)),
            "y": None}


# (case, kind, N): scenarios by name; "cart_*" is the inline skill with a virtual variable
CASES = [("ur5_track", "pinv", N_CHUNKS), ("ur5_moe2016_pinv", "pinv", N_CHUNKS), ("ur5_qp", "qp", N_CHUNKS),
         ("ur5_nlp_quartic", "nlp", N_NLP), ("cart_pinv", "pinv", 100003), ("cart_qp", "qp", 100003)]


def _setup(case, N, seed=3):
    if case.startswith("cart_"):
        pinv = case == "cart_pinv"
        ctrl = cc.PseudoInverseController(_cart_spec()) if pinv else cc.ReactiveQPController(_cart_spec(False))
        inp = _cart_inputs(N, seed)
    else:
        sc = scenarios.get(case)
        ctrl = sc.make_controller()
        inp = sc.sample(N, seed=seed)
    ctrl.setup_solver()
    if case == "ur5_moe2016_pinv":
        inp["t"] = np.array([0.37])          # one time value shared by every instance (t_stride 0)
    return ctrl, inp


def _n_virtual(ctrl):
    return ctrl._nx if isinstance(ctrl, cc.PseudoInverseController) else ctrl._nxv


def _out_shapes(ctrl, kind, N):
    """(shape, dtype) of each solve_batch output; None for an output the skill does not have."""
    if kind == "pinv":
        nx = _n_virtual(ctrl)
        return [((ctrl.skill_spec.n_robot_var, N), np.float64), ((nx, N), np.float64) if nx else None,
                ((N,), np.int32)]
    shapes = [((ctrl._qn, N), np.float64), ((N,), np.int32), ((2, N), np.int32)]
    return shapes + [((N,), np.int32)] if kind == "nlp" else shapes


OPTIONAL = {"pinv": (2,), "qp": (1, 2), "nlp": (1, 2, 3)}     # mode / status, active / status, active, iterations


def _outs(ctrl, kind, N, pinned, omit=()):
    outs = []
    for k, spec in enumerate(_out_shapes(ctrl, kind, N)):
        if spec is None or k in omit:
            outs.append(None)
            continue
        a = np.empty(spec[0], dtype=spec[1])
        a = _pin(a) if pinned else a
        a[...] = np.nan if spec[1] == np.float64 else -7
        outs.append(a)
    return tuple(outs)


def _warm(ctrl, N, seed=5):
    return {"warmstart": np.random.default_rng(seed).uniform(-0.05, 0.05, (ctrl._qn, N))}


def _inputs(inp, conv):
    return tuple(conv(inp[k]) if inp[k] is not None else None for k in ("t", "q", "x", "y"))


def _host(ctrl, inp, out, conv=np.ascontiguousarray, **kw):
    res = ctrl.solve_batch(*_inputs(inp, conv), out=out, **{k: conv(v) for k, v in kw.items()})
    assert all(r is o for r, o in zip(res, out))
    return tuple(None if o is None else o.copy() for o in out)


def _device(ctrl, inp, **kw):
    res = ctrl.solve_batch(*_inputs(inp, _up), **{k: _up(v) for k, v in kw.items()})
    _torch().cuda.synchronize()
    return tuple(_down(r) for r in res)


def _multi(ctrl, kind, handles, inp, out, conv, warm):
    """clik_<kind>_step_host_multi with the given handles, straight through the C ABI."""
    lib = runtime.load_library()
    t, q, x, y = _inputs(inp, conv)
    arr = (vp * len(handles))(*handles)
    head = (arr, len(handles), q.shape[1], _ptr(t), 0 if t.size == 1 else 1, _ptr(q), _ptr(x), _ptr(y))
    p = [_ptr(o) for o in out]
    if kind == "pinv":
        runtime.check(lib.clik_pinv_step_host_multi(*head, *p))
        return
    w = conv(warm["warmstart"]) if warm else None       # kept alive through the call
    x0 = _ptr(w)
    if kind == "qp":
        mi = int(ctrl.options.get("max_iter", 0) or 0)
        runtime.check(lib.clik_qp_step_host_multi(*head, x0, None, p[0], p[1], p[2], mi))
    else:
        runtime.check(lib.clik_nlp_step_host_multi(*head, x0, p[0], p[1], p[3], p[2], ctrl._max_iter(None)))


@pytest.mark.parametrize("case,kind,N", CASES, ids=[c[0] for c in CASES])
def test_host_routes_give_the_device_bits(case, kind, N):
    ctrl, inp = _setup(case, N)
    warm = _warm(ctrl, N) if kind == "nlp" else {}
    ref = _device(ctrl, inp, **warm)
    if kind != "pinv":
        assert (ref[1] == 0).mean() > 0.5, case                 # most instances solved: the bits mean something
    # (a) pageable, (b) everything page-locked (zero copy), (c) page-locked inputs, pageable outputs (pipeline)
    for in_pinned, out_pinned in ((False, False), (True, True), (True, False)):
        conv = _pin if in_pinned else np.ascontiguousarray
        got = _host(ctrl, inp, _outs(ctrl, kind, N, out_pinned), conv, **warm)
        assert _same(got, ref), (case, in_pinned, out_pinned)
    # (d) two handles of the same cubin on device 0 (two shards from two host threads), pageable and pinned
    extra = runtime.CompiledSkill(ctrl._cubin, ctrl.kernel_meta, n_slack=ctrl.skill_spec.n_slack_var, device=0)
    handles = [ctrl._skill(0).handle.value, extra.handle.value]
    for pinned in (False, True):
        out = _outs(ctrl, kind, N, pinned)
        _multi(ctrl, kind, handles, inp, out, _pin if pinned else np.ascontiguousarray, warm)
        assert _same(out, ref), (case, pinned, "two handles")
    # (e) optional outputs omitted: the others are unchanged, on both routes
    omit = OPTIONAL[kind]
    ref_e = tuple(None if k in omit else r for k, r in enumerate(ref))
    for pinned in (False, True):
        conv = _pin if pinned else np.ascontiguousarray
        got = _host(ctrl, inp, _outs(ctrl, kind, N, pinned, omit=omit), conv, **warm)
        assert _same(got, ref_e), (case, pinned, "optional outputs omitted")


@pytest.mark.parametrize("case", ["ur5_qp", "cart_qp"])
def test_qp_host_warm_start_and_working_set(case):
    """(f) warmstart and warm_active as host arrays, pageable and page-locked, give the device bits."""
    N = N_CHUNKS if case == "ur5_qp" else 100003
    ctrl, inp = _setup(case, N)
    cold = _device(ctrl, inp)
    rng = np.random.default_rng(11)
    warm = {"warmstart": cold[0] + rng.uniform(-1e-3, 1e-3, cold[0].shape),
            "warm_active": np.ascontiguousarray(cold[2])}
    ref = _device(ctrl, inp, **warm)
    for pinned in (False, True):
        conv = _pin if pinned else np.ascontiguousarray
        got = _host(ctrl, inp, _outs(ctrl, "qp", N, pinned), conv, **warm)
        assert _same(got, ref), (case, pinned)


@pytest.mark.parametrize("name,N", [("ur5_qp", N_CHUNKS), ("ur5_nlp_quartic", N_NLP)])
def test_multipliers_on_host_arrays_give_the_device_bits(name, N):
    ctrl, inp = _setup(name, N)
    step = _device(ctrl, inp)
    sol, status, active = step[:3]
    torch = _torch()
    ref = _down(ctrl.multipliers_batch(*_inputs(inp, _up), _up(sol), _up(status), _up(active)))
    torch.cuda.synchronize()
    assert np.isfinite(ref[:, status == 0]).all()
    got = ctrl.multipliers_batch(*_inputs(inp, np.ascontiguousarray), sol, status, active)
    assert np.array_equal(got, ref, equal_nan=True), (name, "pageable")
    lam = _pin(np.full((ctrl._qm, N), np.nan))
    res = ctrl.multipliers_batch(*_inputs(inp, _pin), _pin(sol), _pin(status), _pin(active), out=lam)
    assert res is lam and np.array_equal(lam, ref, equal_nan=True), (name, "page-locked")
