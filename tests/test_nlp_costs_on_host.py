"""NLP costs that read the skill's inputs directly — a velocity target from input_var, a raw joint
coordinate as a weight, the time — through the host build of the emitted kernel source (as in
test_nlp_kernel_on_host.py), against SLSQP and the first-order certificate; and the emitted F, gradient and
Hessian against central finite differences of the emitted F and against the expression interpreter."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import cs, scenarios
from casclik_b200.sym import dag
from test_kernel_code_on_host import ROOT, SHIM, _host_library
from test_nlp_kernel_on_host import MU, _check_against_slsqp

PROBE = r'''
extern "C" double nlp_probe(double t, const double* q, const double* x, const double* y, const double* v,
                            double* g, double* H, double* f_only) {
  double qv[Skill::NQ > 0 ? Skill::NQ : 1] = {0}, xv[Skill::NX > 0 ? Skill::NX : 1] = {0};
  double yv[Skill::NY > 0 ? Skill::NY : 1] = {0}, vv[Skill::NN], gg[Skill::NN], HH[Skill::NN * (Skill::NN + 1) / 2];
  for (int j = 0; j < Skill::NQ; ++j) qv[j] = q[j];
  for (int j = 0; j < Skill::NX; ++j) xv[j] = x[j];
  for (int j = 0; j < Skill::NY; ++j) yv[j] = y[j];
  for (int j = 0; j < Skill::NN; ++j) vv[j] = v[j];
  clik::NlpData<Skill> d;
  Skill::eval_nlp_pre(t, qv, xv, yv, d);
  const double F = Skill::eval_nlp_fgH(d.P, vv, gg, HH);
  for (int j = 0; j < Skill::NN; ++j) g[j] = gg[j];
  for (int k = 0; k < Skill::NN * (Skill::NN + 1) / 2; ++k) H[k] = HH[k];
  *f_only = Skill::eval_nlp_f(d.P, vv);
  return F;
}
'''


def _ur5(cost_name):
    """ur5_qp's skill with a cost that feeds t, q or y straight into decision-dependent nodes."""
    sc = scenarios.get("ur5_qp")
    spec = sc.spec
    dq, q, y, t = spec.robot_vel_var, spec.robot_var, spec.input_var, spec.time_var
    quart = cs.sum1((dq * dq) * (dq * dq))
    e = dq[:3] - y
    cost = {
        # track a velocity target from the input (mu-weighted: F is small, the cost weakly curved)
        "ytrack": MU * (cs.dot(e, e) + cs.dot(dq, dq) + quart),
        # a raw joint coordinate as a weight (q_0 > 0 on the sampled range: convex)
        "qweight": q[0] * dq[0] * dq[0] + cs.dot(dq, dq) + 0.1 * quart,
        # the time as a velocity target
        "time": (dq[0] - t) * (dq[0] - t) + cs.dot(dq, dq) + quart,
    }[cost_name]
    return sc, cc.ReactiveNLPController(spec, cost)


@pytest.mark.parametrize("cost_name", ["ytrack", "qweight", "time"])
def test_costs_reading_inputs_directly(cost_name, tmp_path):
    sc, ctrl = _ur5(cost_name)
    lib = _host_library(ctrl, tmp_path)
    assert not ctrl.kernel_meta["nlp_quadratic"]
    src = ctrl.kernel_source
    body = src[src.index("eval_nlp_f("):src.index("static constexpr unsigned NLP_READ_T")]
    assert "q[" not in body and "y[" not in body and " t " not in body and "t)" not in body   # hoisted into P
    inp = {k: v for k, v in sc.sample(64, seed=11).items() if v is not None}
    inp["t"] = np.random.default_rng(12).uniform(-0.5, 0.5, 64)
    solved, iters = _check_against_slsqp(ctrl, lib, inp)
    assert solved == 64 and iters.max() > 1


def _probe_library(ctrl, tmp_path):
    _host_library(ctrl, tmp_path)                     # lowers + emits (kernel_source) without nvcc
    src = tmp_path / "probe.cpp"
    src.write_text(SHIM + ctrl.kernel_source + PROBE)
    so = tmp_path / "probe.so"
    subprocess.run(["g++", "-O0", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                    "-I", os.path.join(ROOT, "casclik_b200", "csrc"), "-o", str(so), str(src)], check=True)
    lib = ctypes.CDLL(str(so))
    lib.nlp_probe.restype = ctypes.c_double
    return lib


@pytest.mark.parametrize("name", ["ur5_nlp_quartic", "ur5_nlp_taskspeed", "qweight"])
def test_emitted_gradient_and_hessian_against_finite_differences(name, tmp_path):
    if name == "qweight":
        sc, ctrl = _ur5("qweight")
    else:
        sc = scenarios.get(name)
        ctrl = sc.make_controller()
    lib = _probe_library(ctrl, tmp_path)
    prog = ctrl._prog
    n = prog.nx
    nh = n * (n + 1) // 2
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    inp = sc.sample(4, seed=21)
    rng = np.random.default_rng(22)
    for i in range(4):
        t = np.array([0.3])
        q = np.ascontiguousarray(inp["q"][:, i])
        y = np.ascontiguousarray(inp["y"][:, i])
        x = np.zeros(1)
        v0 = rng.uniform(-0.5, 0.5, n)

        def fgh(v):
            g, H, fo = np.empty(n), np.empty(nh), np.empty(1)
            F = lib.nlp_probe(ctypes.c_double(t[0]), p(q), p(x), p(y), p(np.ascontiguousarray(v)), p(g), p(H), p(fo))
            Hf = np.zeros((n, n))
            Hf[np.tril_indices(n)] = H               # row-major packed lower triangle
            return F, g, Hf + np.tril(Hf, -1).T, fo[0]

        F, g, H, fo = fgh(v0)
        assert fo == F
        vals = {prog.syms.t[0].id: t[0]}
        vals.update({s.id: q[j] for j, s in enumerate(prog.syms.q)})
        vals.update({s.id: y[j] for j, s in enumerate(prog.syms.y)})
        vals.update({s.id: v0[j] for j, s in enumerate(prog.dec)})
        Fi = float(dag.evaluate([prog.F], vals)[0])  # the expression interpreter, not the emitted code
        assert abs(F - Fi) <= 1e-13 * (1 + abs(Fi))
        h = 1e-5
        gfd, Hfd = np.empty(n), np.empty((n, n))
        for j in range(n):
            e = np.zeros(n)
            e[j] = h
            Fp, gp, _, _ = fgh(v0 + e)
            Fm, gm, _, _ = fgh(v0 - e)
            gfd[j] = (Fp - Fm) / (2 * h)
            Hfd[:, j] = (gp - gm) / (2 * h)
        assert np.abs(g - gfd).max() <= 1e-6 * (1 + np.abs(g).max()), np.abs(g - gfd).max()
        assert np.abs(H - Hfd).max() <= 1e-6 * (1 + np.abs(H).max()), np.abs(H - Hfd).max()
