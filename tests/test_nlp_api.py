"""ReactiveNLPController's Python surface and cs.hessian (no GPU needed)."""
import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import cs, scenarios
from casclik_b200.sym import dag


def _ur5_qp_spec():
    return scenarios.get("ur5_qp").spec


def test_hessian_matches_a_hand_derived_case():
    x = cs.MX.sym("x", 2)
    f = x[0] ** 2 * x[1] + cs.sin(x[1])
    H, g = cs.hessian(f, x)
    assert H.size() == (2, 2) and g.size() == (2, 1)
    for a, b in ((0.3, -1.2), (2.0, 0.5)):
        vals = {x.nodes()[0].id: a, x.nodes()[1].id: b}
        hv = np.array(dag.evaluate(H.nodes(), vals), dtype=float).reshape(2, 2, order="F")
        gv = np.array(dag.evaluate(g.nodes(), vals), dtype=float)
        assert np.allclose(gv, [2 * a * b, a * a + np.cos(b)], rtol=0, atol=1e-14)
        assert np.allclose(hv, [[2 * b, 2 * a], [2 * a, -np.sin(b)]], rtol=0, atol=1e-14)


def test_constructor_validation():
    spec = _ur5_qp_spec()
    dq = spec.robot_vel_var
    with pytest.raises(ValueError, match="scalar"):
        cc.ReactiveNLPController(spec, dq * dq)
    foreign = cs.MX.sym("foreign_weight")
    with pytest.raises(ValueError, match="foreign_weight"):
        cc.ReactiveNLPController(spec, foreign * cs.dot(dq, dq))
    t, q, dq40 = cs.MX.sym("t"), cs.MX.sym("q", 40), cs.MX.sym("dq", 40)
    big = cc.SkillSpecification("big", t, q, robot_vel_var=dq40,
                                constraints=[cc.VelocitySetConstraint("spd", q, set_min=-np.ones(40), set_max=np.ones(40))])
    with pytest.raises(ValueError, match="at most 32"):
        cc.ReactiveNLPController(big, cs.dot(dq40, dq40))
    t, q2, dq2 = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    tall = cc.SkillSpecification("tall", t, q2, robot_vel_var=dq2,           # 2 variables, 65 rows
                                 constraints=[cc.VelocitySetConstraint("rows", cs.vertcat(*[q2[k % 2] * (1 + k) for k in range(65)]),
                                                                       set_min=-1.0, set_max=1.0)])
    with pytest.raises(ValueError, match="64 constraint rows"):
        cc.ReactiveNLPController(tall, cs.dot(dq2, dq2))
    with pytest.raises(ValueError):
        cc.ReactiveNLPController(spec, cs.dot(dq, dq), options={"tol": 0.0})


def test_option_defaults():
    spec = _ur5_qp_spec()
    ctrl = cc.ReactiveNLPController(spec, cs.dot(spec.robot_vel_var, spec.robot_vel_var))
    o = ctrl.options
    assert o["solver_name"] == "ipopt" and o["solver_opts"] == {} and o["function_opts"] == {}
    assert o["max_iter"] == 50 and o["tol"] == 1e-10
    assert ctrl.weight_shifter == 0.001
    kept = cc.ReactiveNLPController(spec, 0.0, options={"solver_name": "ipopt", "solver_opts": {"ipopt.print_level": 0},
                                                                  "max_iter": 7, "tol": 1e-8})
    assert kept.options["solver_opts"] == {"ipopt.print_level": 0} and kept.options["max_iter"] == 7


def test_cost_expression_is_the_stated_convention():
    spec = _ur5_qp_spec()
    dq, s = spec.robot_vel_var, spec.slack_var
    cost = cs.dot(dq, dq) * 3.0
    ctrl = cc.ReactiveNLPController(spec, cost, slack_var_weights=[2.0, 3.0, 4.0])
    F = ctrl.get_cost_expr()
    rng = np.random.default_rng(0)
    v = rng.normal(size=9)
    vals = {n.id: v[j] for j, n in enumerate(dq.nodes() + s.nodes())}
    got = float(dag.evaluate(F.nodes(), vals)[0])
    want = 3.0 * v[:6] @ v[:6] + sum((0.001 + w) * v[6 + k] ** 2 for k, w in enumerate((2.0, 3.0, 4.0)))
    assert abs(got - want) <= 1e-13 * abs(want)
    default = cc.ReactiveNLPController(spec, cost)          # slack weights: cnstr.slack_weight per soft row
    sw = spec.constraints[0].slack_weight
    got = float(dag.evaluate(default.get_cost_expr().nodes(), vals)[0])
    assert abs(got - (3.0 * v[:6] @ v[:6] + (0.001 + sw) * v[6:] @ v[6:])) <= 1e-13 * abs(got)
    A, lb, ub = ctrl.get_constraints_expr()
    qp = cc.ReactiveQPController(spec)
    Aq, lbq, ubq = qp.get_constraints_expr()
    assert [n.id for n in A.nodes()] == [n.id for n in Aq.nodes()]
    assert [n.id for n in lb.nodes()] == [n.id for n in lbq.nodes()]


def test_solve_before_setup_raises_and_the_initial_problem_is_scoped():
    spec = _ur5_qp_spec()
    ctrl = cc.ReactiveNLPController(spec, cs.dot(spec.robot_vel_var, spec.robot_vel_var))
    with pytest.raises(RuntimeError, match="setup"):
        ctrl.solve(0.0, [0.1] * 6, input_var=[0.3, 0.3, 0.3])
    ctrl.setup_initial_problem_solver()
    with pytest.raises(NotImplementedError, match="follow-up"):
        ctrl.solve_initial_problem(0.0, [0.1] * 6)
    t, q, dq = cs.MX.sym("t"), cs.MX.sym("q", 2), cs.MX.sym("dq", 2)
    plain = cc.SkillSpecification("plain", t, q, robot_vel_var=dq,
                                  constraints=[cc.VelocitySetConstraint("spd", q, set_min=-np.ones(2), set_max=np.ones(2))])
    p = cc.ReactiveNLPController(plain, cs.dot(dq, dq))
    p.setup_initial_problem_solver()
    assert p.solve_initial_problem(0.0, [0.0, 0.0]) == (None, None)


def test_emitted_image_and_manifest():
    sc = scenarios.get("ur5_nlp_taskspeed")
    ctrl = sc.make_controller()
    from casclik_b200 import build
    saved = build.compile_cubin
    build.compile_cubin = lambda source, tag="skill", **kw: (b"", "/nonexistent.cubin")
    try:
        ctrl.setup_problem_functions(load=False)
    finally:
        build.compile_cubin = saved
    src, meta = ctrl.kernel_source, ctrl.kernel_meta
    assert meta["has_nlp"] and not meta["has_pinv"] and not meta["has_qp"]
    assert (meta["qp_n"], meta["qp_m"]) == (9, 15) and meta["nlp_quadratic"]
    assert "o[7] = 256;" in src and "clik_nlp_kernel" in src and "clik_nlp_rollout_kernel" in src
    assert "clik_qp_kernel" not in src
    # the forward kinematics is evaluated once per step: the cost functions only read hoisted values
    f_body = src[src.index("eval_nlp_f("):src.index("eval_nlp_fgH(")]
    assert "sincos" not in f_body and "q[" not in f_body and "P[" in f_body
    assert set(meta["nlp_eval"]) == {"pre", "f", "fgH"} and meta["nlp_eval"]["fgH"]["flops"] > 0
    assert cc.ReactiveNLPController is type(ctrl)
