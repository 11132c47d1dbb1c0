"""The NLP controller's shard entry points (clik_nlp_step_ld, clik_nlp_step_host_multi) and the devices= argument
of ReactiveNLPController.solve_batch: argument errors are reported without a device."""
import ctypes

import numpy as np
import pytest

from casclik_b200 import runtime, scenarios


def test_host_multi_without_handles_is_invalid():
    lib = runtime.load_library()
    vp = ctypes.c_void_p
    N = 4
    t, q, y, sol = np.zeros(N), np.zeros((6, N)), np.zeros((3, N)), np.empty((9, N))
    p = lambda a: vp(a.ctypes.data)  # noqa: E731
    args = (N, p(t), 1, p(q), None, p(y), None, p(sol), None, None, None, 0)
    assert lib.clik_nlp_step_host_multi(None, 1, *args) == 1                   # CLIK_ERR_INVALID
    assert b"no skill handles" in lib.clik_last_error()
    one = (vp * 1)(None)
    assert lib.clik_nlp_step_host_multi(one, 0, *args) == 1
    assert b"no skill handles" in lib.clik_last_error()
    assert lib.clik_nlp_step_host_multi(one, 1, *args) == 1
    assert b"no skill handles" in lib.clik_last_error()
    two = (vp * 2)(None, None)
    assert lib.clik_nlp_step_host_multi(two, 2, *args) == 1
    assert b"no skill handles" in lib.clik_last_error()
    assert lib.clik_nlp_step_host(None, *args) == 1                            # the one-handle multi call
    assert b"no skill handles" in lib.clik_last_error()


def test_ld_with_a_null_skill_is_invalid():
    lib = runtime.load_library()
    assert lib.clik_nlp_step_ld(None, 4, 4, None, 0, None, None, None, None, None, None, None, None, 0, None) == 1
    assert b"skill is NULL" in lib.clik_last_error()


@pytest.mark.parametrize("devices", ["bogus", 0, [0, 0], (1, 1)])
def test_solve_batch_rejects_bad_devices(devices):
    """Rejected before any device is touched, whatever the number of visible GPUs."""
    sc = scenarios.get("ur5_nlp_quartic")
    ctrl = sc.make_controller()
    ctrl.setup_problem_functions(load=False)
    inp = sc.sample(8, seed=0)
    with pytest.raises(ValueError, match="devices"):
        ctrl.solve_batch(inp["t"], inp["q"], None, inp["y"], devices=devices)
