"""multipliers_batch and the lam_* entries of solve()'s res: argument validation without a device, the 32-row
limit, and the emitted source (the multiplier kernel is appended; nothing emitted before it changes)."""
import ctypes
import hashlib
import os

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import build, cs, runtime, scenarios


def _setup_without_nvcc(ctrl, tmp_path):
    saved = (build.compile_cubin, build.kernel_registers)
    build.compile_cubin = lambda source, tag="skill", **kw: (b"", os.path.join(str(tmp_path), "skill.cubin"))
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


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_more_than_32_rows_has_no_multiplier_kernel(kind, tmp_path):
    spec = _wide_spec(33)
    ctrl = cc.ReactiveQPController(spec) if kind == "qp" else cc.ReactiveNLPController(
        spec, cs.dot(spec.robot_vel_var, spec.robot_vel_var))
    _setup_without_nvcc(ctrl, tmp_path)
    assert ctrl._qm == 33 and not ctrl.kernel_meta["duals"]
    assert "duals_kernel" not in ctrl.kernel_source and "o[18]" not in ctrl.kernel_source
    N = 4
    with pytest.raises(ValueError, match="at most 32 constraint rows"):
        ctrl.multipliers_batch(np.zeros(N), np.zeros((3, N)), None, None, np.zeros((3, N)),
                               np.zeros(N, np.int32), np.zeros((2, N), np.int32))


def test_32_rows_get_the_kernel(tmp_path):
    ctrl = cc.ReactiveQPController(_wide_spec(32))
    _setup_without_nvcc(ctrl, tmp_path)
    assert ctrl.kernel_meta["duals"] and "clik_qp_duals_kernel" in ctrl.kernel_source


def test_out_and_shapes_are_validated_without_a_device(tmp_path):
    sc = scenarios.get("ur5_qp")
    ctrl = sc.make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    N, n, m = 5, ctrl._qn, ctrl._qm
    inp = sc.sample(N, seed=0)
    t, q = inp["t"], inp["q"]
    sol, st, act = np.zeros((n, N)), np.zeros(N, np.int32), np.zeros((2, N), np.uint32)
    bad = [
        dict(out=np.zeros((m, N), np.float32)),              # dtype
        dict(out=np.zeros((m, N + 1))),                       # size
        dict(out=np.zeros((N, m)).T),                         # layout
        dict(sol=np.zeros((n, N + 1))),
        dict(status=np.zeros(N + 2, np.int32)),
        dict(active=np.zeros((1, N), np.int32)),
    ]
    for kw in bad:
        args = dict(sol=sol, status=st, active=act, out=None)
        args.update(kw)
        with pytest.raises(runtime.ClikError):
            ctrl.multipliers_batch(t, q, None, None, args["sol"], args["status"], args["active"], out=args["out"])
    with pytest.raises(ValueError, match="robot_var"):
        ctrl.multipliers_batch(t, q[:3], None, None, sol, st, act)
    with pytest.raises(ValueError, match="required"):
        ctrl.multipliers_batch(t, q, None, None, sol, None, act)
    nc = scenarios.get("ur5_nlp_quartic").make_controller()
    with pytest.raises(RuntimeError, match="setup"):
        nc.multipliers_batch(t, q, None, inp["y"], sol, st, act)


def test_abi_rejects_a_null_skill_and_missing_kernels():
    lib = runtime.load_library()
    for name in ("clik_qp_duals_host", "clik_nlp_duals_host"):
        assert getattr(lib, name)(None, 4, None, 0, None, None, None, None, None, None, None) == 1
        assert b"skill is NULL" in lib.clik_last_error()


class _FakeLib(object):
    """Stands in for the library behind solve(): writes recognisable values into the output pointers."""

    def __init__(self, n, m):
        self.n, self.m = n, m

    def _fill(self, sol, status, active, lam):
        ctypes.memmove(sol.value, np.arange(self.n, dtype=np.float64).ctypes.data, 8 * self.n)
        ctypes.memset(status.value, 0, 4)
        ctypes.memset(active.value, 0, 8)
        if lam is not None:
            ctypes.memmove(lam.value, (-1.0 - np.arange(self.m, dtype=np.float64)).ctypes.data, 8 * self.m)
        return 0

    def clik_qp_solve_one_lam(self, h, t, q, x, y, x0, sol, status, active, mi, lam):
        return self._fill(sol, status, active, lam)

    def clik_nlp_solve_one_lam(self, h, t, q, x, y, x0, sol, status, iters, active, mi, lam):
        ctypes.memset(iters.value, 0, 4)
        return self._fill(sol, status, active, lam)


class _FakeSkill(object):
    def __init__(self, n, m):
        self._lib = _FakeLib(n, m)
        self.handle = None


@pytest.mark.parametrize("kind", ["qp", "nlp"])
def test_solve_res_has_the_multiplier_entries(kind, tmp_path, monkeypatch):
    name = "ur5_qp" if kind == "qp" else "ur5_nlp_quartic"
    sc = scenarios.get(name)
    ctrl = sc.make_controller()
    _setup_without_nvcc(ctrl, tmp_path)
    n, m = ctrl._qn, ctrl._qm
    monkeypatch.setattr(ctrl, "_skill", lambda device=None: _FakeSkill(n, m))
    inp = sc.sample(1, seed=0)
    kw = {} if inp["y"] is None else {"input_var": inp["y"][:, 0]}
    ctrl.solve(float(inp["t"][0]), inp["q"][:, 0], **kw)
    key = "lam_a" if kind == "qp" else "lam_g"
    lam, lam_x = ctrl.res[key], ctrl.res["lam_x"]
    assert lam.shape == (m, 1) and lam_x.shape == (n, 1)
    assert np.array_equal(lam.toarray().ravel(), -1.0 - np.arange(m))
    assert not np.asarray(lam_x.toarray()).any()
    old = {"x", "status", "active_upper", "active_lower", "cost"} if kind == "qp" else {"x", "f", "status", "iterations"}
    assert set(ctrl.res) == old | {key, "lam_x"}


# sha256 of the sources the parent commit emitted for these skills (default environment, each skill built first in a
# fresh interpreter: the operand order of commutative nodes follows the order in which the process created them).
# The multiplier kernel is appended after the manifest kernel and announced by one line in it; nothing else changes.
PARENT_SOURCE_SHA256 = {
    "ur5_qp": "998a8b713678dae46e1b75c32468d3ec6edeb6feedadac052131622301e66ee7",
    "ur5_moe2016_qp": "d4e6d65064d85442fc26821d22d2c2772d8356fa41ec1bee0ed3f422f5e80d4c",
    "ur5_nlp_quartic": "01af1d69d3092961f239a474f4f880c67c0b29666ce82bfa8d0a71305829ba24",
    "ur5_nlp_taskspeed": "a13f130ee822f77e0fd2fa10fe8825c60b7479ff10fe4ffffd2793d14268b42d",
    "dense0": "65ca4c605183d1a3dc3f4fe0740e66cc4dffa5d464e8201742fb8cd4d5de347b",
    "fuzz1": "419ffcfac7504332e8ffae018f29df1a9928d804613614bbb5cdc23dede442db",
}


_EMIT = r"""
import json, sys
import casclik_b200 as cc
from casclik_b200 import scenarios
from casclik_b200.codegen import emit_skill
from fuzz_skills import make_dense_qp_skill, make_qp_skill
name = sys.argv[1]
if name in scenarios.NLP_REGISTRY:
    ctrl = scenarios.get(name).make_controller()
    src, meta = emit_skill(nlp=ctrl._prog, label=ctrl.skill_spec.label, nlp_tol=float(ctrl.options["tol"]))
else:
    if name in ("dense0", "fuzz1"):
        spec, w, _ = make_dense_qp_skill(0) if name == "dense0" else make_qp_skill(1)
        ctrl = cc.ReactiveQPController(spec, **w)
    else:
        ctrl = scenarios.get(name).make_controller()
    src, meta = emit_skill(qp=ctrl._program(), label=ctrl.skill_spec.label)
sys.stdout.write(json.dumps({"src": src, "duals": meta["duals"], "structured": bool(meta.get("qp_structured"))}))
"""


@pytest.mark.parametrize("name", sorted(PARENT_SOURCE_SHA256))
def test_emitted_source_only_gains_the_multiplier_kernel(name):
    import json
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    env = {k: v for k, v in os.environ.items() if not k.startswith("CLIK_")}
    env["PYTHONPATH"] = os.pathsep.join([os.path.dirname(here), here])
    out = subprocess.run([sys.executable, "-c", _EMIT, name], capture_output=True, text=True, env=env, check=True)
    res = json.loads(out.stdout)
    src = res["src"]
    assert res["duals"]
    head, sep, tail = src.partition("\n\n// ---- constraint multipliers of the step's output (clik_duals.cuh) ----\n")
    assert sep and tail.count("__global__") == 1 and "duals_kernel(" in tail
    lines = (head + "\n").split("\n")
    o18 = [ln for ln in lines if ln.lstrip().startswith("o[18] = ")]
    assert len(o18) == 1
    lines.remove(o18[0])
    assert hashlib.sha256("\n".join(lines).encode()).hexdigest() == PARENT_SOURCE_SHA256[name]
    assert ("struct SkillDuals : Skill" in tail) == res["structured"]
