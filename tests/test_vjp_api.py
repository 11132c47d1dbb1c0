"""vjp_batch and solve_batch_differentiable without a device: the 32-row limit, NumPy inputs, the emitted manifest
line, and the ABI's refusal of a NULL skill."""
import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import build, cs, runtime, scenarios


def _setup_without_nvcc(ctrl, tmp_path):
    saved = (build.compile_cubin, build.kernel_registers)
    build.compile_cubin = lambda source, tag="skill", **kw: (b"", str(tmp_path / "skill.cubin"))
    build.kernel_registers = lambda *a, **kw: None
    try:
        ctrl.setup_problem_functions(load=False)
    finally:
        build.compile_cubin, build.kernel_registers = saved


def _wide_spec(rows):
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 3), cs.MX.sym("dq", 3)
    e = cs.vertcat(*[(1.0 + k) * q[k % 3] for k in range(rows)])
    cons = [cc.VelocitySetConstraint("box", e, set_min=-1.0, set_max=1.0)]
    return cc.SkillSpecification("wide%d" % rows, t, q, robot_vel_var=dq, constraints=cons)


def _ctrl(kind, spec):
    return cc.ReactiveQPController(spec) if kind == "qp" else cc.ReactiveNLPController(
        spec, cs.dot(spec.robot_vel_var, spec.robot_vel_var))


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_more_than_32_rows_raise_and_build_no_kernel(kind, tmp_path, monkeypatch):
    ctrl = _ctrl(kind, _wide_spec(33))
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._vjp_source()
    assert not meta["vjp"] and "vjp_kernel" not in source and "o[19]" not in source
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no VJP image may be built"))
    N = 4
    with pytest.raises(ValueError, match="at most 32 constraint rows"):
        ctrl.vjp_batch(np.zeros(N), np.zeros((3, N)), None, None, np.zeros((3, N)), np.zeros(N, np.int32),
                       np.zeros((2, N), np.int32), np.zeros((3, N)))
    assert ctrl._vjp is None


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_32_rows_get_the_kernel_and_the_manifest_line(kind, tmp_path):
    ctrl = _ctrl(kind, _wide_spec(32))
    _setup_without_nvcc(ctrl, tmp_path)
    source, meta = ctrl._vjp_source()
    assert meta["vjp"] and ("clik_%s_vjp_kernel(" % kind) in source
    assert ("o[19] = %d;" % (1 if kind == "qp" else 2)) in source
    assert "vjp" not in ctrl.kernel_source and "vjp_eval" in meta


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_nlp_quartic"])
def test_numpy_inputs_raise_without_building_the_image(name, tmp_path, monkeypatch):
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    monkeypatch.setattr(build, "compile_cubin", lambda *a, **kw: pytest.fail("no VJP image may be built"))
    N, n = 5, ctrl._qn
    inp = sc.sample(N, seed=0)
    args = (inp["t"], inp["q"], None, inp["y"], np.zeros((n, N)), np.zeros(N, np.int32), np.zeros((2, N), np.int32))
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.vjp_batch(*args, np.ones((n, N)))
    with pytest.raises(ValueError, match="CUDA"):
        ctrl.solve_batch_differentiable(inp["t"], inp["q"], None, inp["y"])
    assert ctrl._vjp is None
    nc = scenarios.get("ur5_nlp_taskspeed").make_controller()
    with pytest.raises(RuntimeError, match="setup"):
        nc.vjp_batch(*args, np.ones((n, N)))


def test_abi_rejects_a_null_skill():
    lib = runtime.load_library()
    for name in ("clik_qp_vjp", "clik_nlp_vjp"):
        assert getattr(lib, name)(None, 4, None, 0, *([None] * 12)) == 1
        assert b"skill is NULL" in lib.clik_last_error()
