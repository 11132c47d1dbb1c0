"""The benchmark / parity scenarios of BASELINE.json (`configs`), built through the public API.

Each builder returns a `Scenario`: the SkillSpecification, the controller class and options, and
a seeded synthetic input sampler (SURVEY.md §8d gives the distributions).  Used by bench.py,
__graft_entry__.py and the tests, so all three measure and check exactly the same skills.

  ur5_track       configs[0], configs[1]: UR5 (URDF FK), one EqualityConstraint  e = p_fk(q) - y
  iiwa_multitask  configs[2]: 7 joint-limit SetConstraints + 4-row pose EqualityConstraint
  ur5_qp          configs[3]: soft position Eq (K = 50) + joint limits + joint speed limits
  ur5_moe2016     configs[4]: 3 scalar box sets (K = 500) + time-varying 3-row path Eq (K = 0.15)

NLP_REGISTRY holds the scenarios of ReactiveNLPController (no BASELINE config; tools/nlp_bench.py):

  ur5_nlp_taskspeed  ur5_qp's constraints, cost |J_p(q) dq|^2 + mu |dq|^2 (quadratic, q-dependent Hessian)
  ur5_nlp_quartic    ur5_qp's constraints, cost mu |dq|^2 + sum_j (dq_j / 0.3)^4 (convex, not quadratic)
"""
import math

import numpy as np

from . import sym as cs
from . import fk
from .constraints import EqualityConstraint, SetConstraint, VelocitySetConstraint
from .skill_specification import SkillSpecification
from .sym import dag


class Scenario(object):
    def __init__(self, name, spec, controller, options, sampler, description, cost_expr=None):
        self.name, self.spec, self.controller = name, spec, controller
        self.options, self.sampler, self.description = options, sampler, description
        self.cost_expr = cost_expr       # the NLP controller's cost

    def make_controller(self):
        from .controllers import PseudoInverseController, ReactiveQPController, ReactiveNLPController
        if self.controller == "nlp":
            return ReactiveNLPController(self.spec, self.cost_expr,
                                         options=dict(self.options) if self.options else None)
        cls = {"pinv": PseudoInverseController, "qp": ReactiveQPController}[self.controller]
        return cls(skill_spec=self.spec, options=dict(self.options) if self.options else None)

    def sample(self, N, seed=0):
        """-> dict(t (N,), q (nq, N), x or None, y (ny, N) or None), float64, coordinate-major."""
        return self.sampler(N, np.random.default_rng(seed))


def _eval_batch(func, q):
    """Evaluate a cs.Function of one vector argument for a batch q (n, N) -> (rows, N)."""
    ins = func.mx_in(0).nodes()
    outs = func.mx_out(0).nodes()
    vals = dag.evaluate(outs, {s.id: q[i] for i, s in enumerate(ins)})
    N = q.shape[1]
    return np.stack([np.broadcast_to(np.asarray(v, dtype=np.float64), (N,)) for v in vals])


def _ur5_q(N, rng):
    # the notebooks' own %%timeit distribution: 0.5*pi*rand + 0.25*pi
    return rng.uniform(0.25 * math.pi, 0.75 * math.pi, size=(6, N))


def ur5_track():
    d = fk.ur5()
    t = cs.MX.sym("t")
    q = cs.MX.sym("q", 6)
    y = cs.MX.sym("y", 3)
    p = d["T_fk"](q)[:3, 3]
    cnstr = EqualityConstraint(label="track_point", expression=p - y, gain=1.0)
    spec = SkillSpecification(label="ur5_track", time_var=t, robot_var=q, input_var=y,
                              constraints=[cnstr])
    p_fk = cs.Function("p_fk", [q], [p])

    def sampler(N, rng):
        qs = _ur5_q(N, rng)
        target = _eval_batch(p_fk, _ur5_q(N, rng))
        return {"t": np.zeros(N), "q": qs, "x": None, "y": np.ascontiguousarray(target[:3])}

    return Scenario("ur5_track", spec, "pinv", None, sampler,
                    "UR5 PseudoInverseController, one 3-row EqualityConstraint (EE position tracking)")


def iiwa_multitask(stress=False):
    d = fk.iiwa14()
    n = 7
    t = cs.MX.sym("t")
    q = cs.MX.sym("q", n)
    y = cs.MX.sym("y", 12)          # [vec(R_des) column-major ; p_des]
    lower, upper = np.array(d["lower"]), np.array(d["upper"])
    T = d["T_fk"](q)
    R, p = T[:3, :3], T[:3, 3]
    R_des = cs.reshape(y[:9], 3, 3)
    p_des = y[9:]
    limits = [SetConstraint(label="limit_q_%d" % i, expression=q[i], set_min=float(lower[i]),
                            set_max=float(upper[i]), priority=i) for i in range(n)]
    if stress:   # T_dist3: three-point form, 9 rows
        rows = [T[i, :3].T + p - R_des[i, :].T - p_des for i in range(3)]
        pose = cs.vertcat(*rows)
    else:        # T_dist2: position + || R_des' R - I ||_F, 4 rows
        pose = cs.vertcat(p - p_des, cs.norm_fro(cs.mtimes(R_des.T, R) - np.eye(3)))
    pose_c = EqualityConstraint(label="pose", expression=pose, gain=1.0, priority=n)
    spec = SkillSpecification(label="iiwa_multitask" + ("_stress" if stress else ""), time_var=t,
                              robot_var=q, input_var=y, constraints=limits + [pose_c])
    T_fk = cs.Function("T_flat", [q], [cs.vertcat(cs.vec(R), p)])

    def sampler(N, rng):
        rng_w = (upper - lower)[:, None]
        qs = rng.uniform(0.0, 1.0, size=(n, N)) * (1.1 * rng_w) + (lower[:, None] - 0.05 * rng_w)
        qd = rng.uniform(0.0, 1.0, size=(n, N)) * rng_w + lower[:, None]
        return {"t": np.zeros(N), "q": qs, "x": None, "y": np.ascontiguousarray(_eval_batch(T_fk, qd))}

    return Scenario(spec.label, spec, "pinv", None, sampler,
                    "KUKA iiwa 7-DOF: 7 joint-limit SetConstraints (128 modes) + %d-row pose "
                    "EqualityConstraint" % (9 if stress else 4))


def ur5_qp():
    d = fk.ur5()
    t = cs.MX.sym("t")
    q = cs.MX.sym("q", 6)
    dq = cs.MX.sym("dq", 6)
    y = cs.MX.sym("y", 3)
    p = d["T_fk"](q)[:3, 3]
    max_speed = math.pi / 5
    c_pos = EqualityConstraint(label="Minimize_point_error", expression=y - p, gain=50.,
                               constraint_type="soft")
    c_lim = SetConstraint(label="Joint_Limits", expression=q, set_min=np.array(d["lower"]),
                          set_max=np.array(d["upper"]))
    c_spd = VelocitySetConstraint(label="Joint_speed_limits", expression=q,
                                  set_min=-cs.vertcat([max_speed] * 6),
                                  set_max=cs.vertcat([max_speed] * 6))
    spec = SkillSpecification(label="ur5_qp", time_var=t, robot_var=q, robot_vel_var=dq,
                              input_var=y, constraints=[c_pos, c_lim, c_spd])
    p_fk = cs.Function("p_fk", [q], [p])

    def sampler(N, rng):
        qs = _ur5_q(N, rng)
        target = _eval_batch(p_fk, _ur5_q(N, rng))
        return {"t": np.zeros(N), "q": qs, "x": None, "y": np.ascontiguousarray(target[:3])}

    return Scenario("ur5_qp", spec, "qp", None, sampler,
                    "UR5 ReactiveQPController: soft 3-row position Eq (K=50) + 6 joint-limit rows + "
                    "6 joint-speed rows; 9 variables x 15 rows")


def _moe_constraints(t, q):
    d = fk.from_denavit_hartenberg(
        joint_angles=["s"] * 6,
        link_lengths=[0., -0.425, -0.392, 0., 0., 0.],
        link_offsets=[0.089, 0., 0., 0.109, 0.095, 0.082],
        link_twists=[math.pi / 2, 0., 0., math.pi / 2, -math.pi / 2, 0.])
    p = d["T_fk"](q)[:3, 3]
    omega = 0.1
    path = cs.vertcat(0.5 * cs.sin(omega * t) * cs.sin(omega * t) + 0.2,
                      0.5 * cs.cos(omega * t) + 0.25 * cs.sin(omega * t),
                      0.5 * cs.sin(omega * t) * cs.cos(omega * t) + 0.1)
    nj = 6
    cx = SetConstraint(label="colav_x", expression=p[0], set_min=0.1, set_max=0.6,
                       priority=nj + 2, gain=5e2)
    cy = SetConstraint(label="colav_y", expression=p[1], set_min=-0.5, set_max=0.4,
                       priority=nj + 1, gain=5e2)
    cz = SetConstraint(label="colav_z", expression=p[2], set_min=-0.3, set_max=0.25,
                       priority=nj + 3, gain=5e2)
    cp = EqualityConstraint(label="move_point2", expression=p - path, priority=nj + 4,
                            constraint_type="soft", gain=0.15)
    return [cx, cy, cz, cp]


def ur5_moe2016(controller="pinv"):
    t = cs.MX.sym("t")
    q = cs.MX.sym("q", 6)
    dq = cs.MX.sym("dq", 6)
    spec = SkillSpecification(label="box_move", time_var=t, robot_var=q, robot_vel_var=dq,
                              constraints=_moe_constraints(t, q))

    def sampler(N, rng):
        return {"t": rng.uniform(0.0, 80.0, size=N), "q": _ur5_q(N, rng), "x": None, "y": None}

    return Scenario("ur5_moe2016_" + controller, spec, controller, None, sampler,
                    "UR5 (DH FK) Moe-2016 example 2: 3 scalar box SetConstraints (K=500, 8 modes) + "
                    "time-varying 3-row path EqualityConstraint (K=0.15)")


def ur5_moe2016_multidim():
    """The notebook's `skill_multidim` (ur5_moe2016_example2.ipynb cell 8): one 3-row box
    SetConstraint + path Eq, run with options {"multidim_sets": True} (experimental in the reference)."""
    t = cs.MX.sym("t")
    q = cs.MX.sym("q", 6)
    dq = cs.MX.sym("dq", 6)
    cx, cy, cz, cp = _moe_constraints(t, q)
    p = cs.vertcat(cx.expression, cy.expression, cz.expression)
    box = SetConstraint(label="colav_box", expression=p, set_min=np.array([0.1, -0.5, -0.3]),
                        set_max=np.array([0.6, 0.4, 0.25]), priority=7, gain=5e2)
    spec = SkillSpecification(label="box_move_multidim", time_var=t, robot_var=q, robot_vel_var=dq,
                              constraints=[box, cp])

    def sampler(N, rng):
        return {"t": rng.uniform(0.0, 80.0, size=N), "q": _ur5_q(N, rng), "x": None, "y": None}

    return Scenario("ur5_moe2016_multidim", spec, "pinv", {"multidim_sets": True}, sampler,
                    "UR5 (DH FK) Moe-2016 example 2, multidim variant: one 3-row box SetConstraint "
                    "(2 modes, options multidim_sets=True) + time-varying 3-row path EqualityConstraint")


REGISTRY = {
    "ur5_track": ur5_track,
    "iiwa_multitask": iiwa_multitask,
    "iiwa_multitask_stress": lambda: iiwa_multitask(stress=True),
    "ur5_qp": ur5_qp,
    "ur5_moe2016_pinv": lambda: ur5_moe2016("pinv"),
    "ur5_moe2016_qp": lambda: ur5_moe2016("qp"),
    "ur5_moe2016_multidim": ur5_moe2016_multidim,
}


def ur5_nlp(cost):
    """ur5_qp's skill (9 variables x 15 rows) with a general cost of the NLP controller."""
    base = ur5_qp()
    spec = base.spec
    q, dq = spec.robot_var, spec.robot_vel_var
    mu = 0.001
    if cost == "taskspeed":
        J = cs.jacobian(fk.ur5()["T_fk"](q)[:3, 3], q)
        v = cs.mtimes(J, dq)
        expr = cs.dot(v, v) + mu * cs.dot(dq, dq)
        what = "|J_p(q) dq|^2 + mu |dq|^2 (quadratic, configuration-dependent Hessian)"
    else:
        u2 = (dq / 0.3) * (dq / 0.3)
        expr = mu * cs.dot(dq, dq) + cs.sum1(u2 * u2)
        what = "mu |dq|^2 + sum_j (dq_j / 0.3)^4 (convex, not quadratic)"
    return Scenario("ur5_nlp_" + cost, spec, "nlp", None, base.sampler,
                    "UR5 ReactiveNLPController on ur5_qp's constraints (9 variables x 15 rows), cost " + what,
                    cost_expr=expr)


NLP_REGISTRY = {
    "ur5_nlp_taskspeed": lambda: ur5_nlp("taskspeed"),
    "ur5_nlp_quartic": lambda: ur5_nlp("quartic"),
}


def get(name):
    return REGISTRY[name]() if name in REGISTRY else NLP_REGISTRY[name]()
