"""The NLP controller's shard entry points on the GPU: a shard solved in place with the row stride of the whole
batch (clik_nlp_step_ld), one host batch cut over several skill handles (clik_nlp_step_host_multi) on one device
and on two, and solve_batch(..., devices=) — every form gives the bits of the single-device call."""
import ctypes

import numpy as np
import pytest

from casclik_b200 import runtime, scenarios

pytestmark = pytest.mark.gpu
vp = ctypes.c_void_p


def _torch():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _up(a, dev=0):
    return None if a is None else _torch().from_numpy(np.ascontiguousarray(a)).to("cuda:%d" % dev)


def _pin(a):
    return None if a is None else _torch().from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def _ptr(a):
    return None if a is None else vp(a.ctypes.data)


def _outs(ctrl, N, pinned):
    """(sol, status, active, iters) host buffers, page-locked or pageable, filled with sentinels."""
    shapes = (((ctrl._qn, N), np.float64, np.nan), ((N,), np.int32, -7), ((2, N), np.int32, -7), ((N,), np.int32, -7))
    outs = []
    for shape, dtype, fill in shapes:
        a = _pin(np.empty(shape, dtype=dtype)) if pinned else np.empty(shape, dtype=dtype)
        a[...] = fill
        outs.append(a)
    return tuple(outs)


def _setup(name, N, seed):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    ctrl.setup_solver()
    inp = sc.sample(N, seed=seed)
    warm = np.random.default_rng(seed + 1).uniform(-0.05, 0.05, (ctrl._qn, N))
    return ctrl, inp, warm


def _same(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True) for x, y in zip(a, b))


def _device_step(ctrl, inp, warm):
    torch = _torch()
    res = ctrl.solve_batch(_up(inp["t"]), _up(inp["q"]), None, _up(inp["y"]), warmstart=_up(warm))
    torch.cuda.synchronize()
    return tuple(r.cpu().numpy() for r in res)


def test_nlp_shard_in_place_with_row_stride_on_one_device():
    """clik_nlp_step_ld on [lo, hi) of a resident batch (pointers advanced by lo, ld = N) writes the bits of the
    whole-batch clik_nlp_step into the shard and nothing outside it; the warm start is read through x0."""
    torch = _torch()
    lib = runtime.load_library()
    N, lo, hi = 100003, 33333, 77778
    ctrl, inp, warm = _setup("ur5_nlp_quartic", N, seed=31)
    t, q, y, x0 = _up(inp["t"]), _up(inp["q"]), _up(inp["y"]), _up(warm)
    sol, status, active, iters = ctrl.solve_batch(t, q, None, y, warmstart=x0)
    cold = ctrl.solve_batch(t, q, None, y)
    torch.cuda.synchronize()
    assert not (torch.equal(cold[0], sol) and torch.equal(cold[3], iters))      # the warm start matters
    sol2, st2 = torch.full_like(sol, float("nan")), torch.full_like(status, -7)
    act2, it2 = torch.full_like(active, -7), torch.full_like(iters, -7)
    handle = ctrl._skill(0).handle
    mi = ctrl._max_iter(None)

    def at(x, lo, size):
        return vp(x.data_ptr() + size * lo)

    runtime.check(lib.clik_nlp_step_ld(handle, hi - lo, N, at(t, lo, 8), 1, at(q, lo, 8), None, at(y, lo, 8),
                                       at(x0, lo, 8), at(sol2, lo, 8), at(st2, lo, 4), at(it2, lo, 4),
                                       at(act2, lo, 4), mi, None))
    torch.cuda.synchronize()
    assert torch.equal(sol2[:, lo:hi], sol[:, lo:hi]) and torch.equal(st2[lo:hi], status[lo:hi])
    assert torch.equal(it2[lo:hi], iters[lo:hi]) and torch.equal(act2[:, lo:hi], active[:, lo:hi])
    assert bool(torch.isnan(sol2[:, :lo]).all()) and bool(torch.isnan(sol2[:, hi:]).all())
    for a in (st2, it2):
        assert bool((a[:lo] == -7).all()) and bool((a[hi:] == -7).all())
    assert bool((act2[:, :lo] == -7).all()) and bool((act2[:, hi:] == -7).all())
    # a row stride shorter than the shard is refused
    assert lib.clik_nlp_step_ld(handle, N, N - 1, vp(t.data_ptr()), 1, vp(q.data_ptr()), None, vp(y.data_ptr()),
                                None, vp(sol2.data_ptr()), None, None, None, mi, None) == 1
    assert b"row stride" in lib.clik_last_error()
    # a NULL handle behind a loaded one is named by its shard index
    small = {k: (None if v is None else np.ascontiguousarray(v[..., :16])) for k, v in inp.items()}
    out = _outs(ctrl, 16, pinned=False)
    arr = (vp * 2)(handle.value, None)
    assert lib.clik_nlp_step_host_multi(arr, 2, 16, _ptr(small["t"]), 1, _ptr(small["q"]), None, _ptr(small["y"]),
                                        None, *[_ptr(o) for o in (out[0], out[1], out[3], out[2])], mi) == 1
    assert b"skill handle 1 is NULL" in lib.clik_last_error()


def _host_multi(handles, ctrl, inp, warm, pinned):
    lib = runtime.load_library()
    conv = _pin if pinned else np.ascontiguousarray
    t, q, y, x0 = conv(inp["t"]), conv(inp["q"]), conv(inp["y"]), conv(warm)
    sol, status, active, iters = _outs(ctrl, q.shape[1], pinned)
    arr = (vp * len(handles))(*handles)
    runtime.check(lib.clik_nlp_step_host_multi(arr, len(handles), q.shape[1], _ptr(t), 1, _ptr(q), None, _ptr(y),
                                               _ptr(x0), _ptr(sol), _ptr(status), _ptr(iters), _ptr(active),
                                               ctrl._max_iter(None)))
    return sol.copy(), status.copy(), active.copy(), iters.copy()


@pytest.mark.parametrize("name", sorted(scenarios.NLP_REGISTRY))
def test_two_handles_on_one_device_give_the_single_handle_bits(name):
    """The skill loaded twice on device 0: clik_nlp_step_host_multi runs two shards from two host threads, on
    pageable (staged pipeline) and page-locked (zero-copy) arrays; N = 1 and 3 (fewer / more instances than
    handles, odd) and 300001 (shards longer than one pipeline chunk)."""
    for N in (1, 3, 300001):
        ctrl, inp, warm = _setup(name, N, seed=40 + N % 7)
        extra = runtime.CompiledSkill(ctrl._cubin, ctrl.kernel_meta, n_slack=ctrl.skill_spec.n_slack_var, device=0)
        handles = [ctrl._skill(0).handle.value, extra.handle.value]
        one = ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"], warmstart=warm)
        dev = _device_step(ctrl, inp, warm)
        assert _same(one, dev), (name, N)
        for pinned in (False, True):
            assert _same(_host_multi(handles[:1], ctrl, inp, warm, pinned), one), (name, N, pinned, "one handle")
            got = _host_multi(handles, ctrl, inp, warm, pinned)
            assert _same(got, one), (name, N, pinned)


def test_devices_on_one_gpu_through_the_python_api():
    """devices=[0] and devices=1 are today's host call (devices=None), with warmstart and out=; CUDA tensors
    refuse devices=."""
    N = 50001
    ctrl, inp, warm = _setup("ur5_nlp_quartic", N, seed=51)
    ref = ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"], warmstart=warm)
    for devices in ([0], 1):
        got = ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"], warmstart=warm, devices=devices)
        assert _same(got, ref), devices
        for pinned in (False, True):
            out = _outs(ctrl, N, pinned)
            res = ctrl.solve_batch(_pin(inp["t"]) if pinned else inp["t"], _pin(inp["q"]) if pinned else inp["q"],
                                   None, _pin(inp["y"]) if pinned else inp["y"],
                                   warmstart=_pin(warm) if pinned else warm, out=out, devices=devices)
            assert all(r is o for r, o in zip(res, out))
            assert _same(out, ref), (devices, pinned)
    with pytest.raises(ValueError, match="host arrays"):
        ctrl.solve_batch(_up(inp["t"]), _up(inp["q"]), None, _up(inp["y"]), devices=[0])


def test_two_physical_devices_give_the_single_gpu_bits():
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    N = 300001
    for name in sorted(scenarios.NLP_REGISTRY):
        ctrl, inp, warm = _setup(name, N, seed=61)
        ref = ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"], warmstart=warm)
        for devices in (2, "all"):
            got = ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"], warmstart=warm, devices=devices)
            assert _same(got, ref), (name, devices, "staged shards")
            out = _outs(ctrl, N, pinned=True)
            ctrl.solve_batch(_pin(inp["t"]), _pin(inp["q"]), None, _pin(inp["y"]), warmstart=_pin(warm), out=out,
                             devices=devices)
            assert _same(out, ref), (name, devices, "zero-copy shards")
        assert sorted(ctrl._compiled) == list(range(torch.cuda.device_count()))
