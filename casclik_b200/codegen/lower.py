"""Lower a SkillSpecification to the scalar programs the kernels need.

For the pseudo-inverse controller this mirrors the *inputs* of the reference's per-mode expression
builder (reference casclik/controllers/pseudo_inverse.py:274-321: Jt, Ji, cnstr_des per constraint)
and stops there — the mode algebra itself is the hand-written kernel (csrc/clik_pinv.cuh).
For the QP controller it mirrors get_cost_expr / get_constraints_expr
(reference casclik/controllers/reactive_qp.py:175-246): H diagonal, A, lb, ub.
"""
from .. import sym as cs
from ..sym import dag
from ..constraints import (EqualityConstraint, SetConstraint, VelocityEqualityConstraint,
                           VelocitySetConstraint)

KIND_EQ, KIND_SET, KIND_VELEQ, KIND_VELSET = 0, 1, 2, 3


def kind_of(cnstr):
    if isinstance(cnstr, EqualityConstraint):
        return KIND_EQ
    if isinstance(cnstr, SetConstraint):
        return KIND_SET
    if isinstance(cnstr, VelocityEqualityConstraint):
        return KIND_VELEQ
    if isinstance(cnstr, VelocitySetConstraint):
        return KIND_VELSET
    raise TypeError("unknown constraint class %r" % type(cnstr).__name__)


def _col(x, rows, what, label):
    """Coerce a bound / target to a column of `rows` nodes (scalars broadcast)."""
    m = x if isinstance(x, cs.GenericMatrixCommon) else cs.DM(x)
    nodes = m.nodes()
    if len(nodes) == 1 and rows > 1:
        nodes = nodes * rows
    if len(nodes) != rows:
        raise ValueError("%s of %s has %d entries, expression has %d rows"
                         % (what, label, len(nodes), rows))
    return nodes


class Symbols(object):
    """C names of the skill's free symbols."""

    def __init__(self, spec):
        self.t = spec.time_var.nodes()
        if len(self.t) != 1:
            raise ValueError("time_var must be a scalar symbol")
        self.q = spec.robot_var.nodes()
        self.x = spec.virtual_var.nodes() if spec.virtual_var is not None else []
        use_input = spec.input_var is not None and spec._has_input
        self.y = spec.input_var.nodes() if use_input else []
        self.names = {self.t[0].id: "t"}
        for i, n in enumerate(self.q):
            self.names[n.id] = "q[%d]" % i
        for i, n in enumerate(self.x):
            self.names[n.id] = "x[%d]" % i
        for i, n in enumerate(self.y):
            self.names[n.id] = "y[%d]" % i

    def check_closed(self, nodes, what):
        free = [s.name for s in dag.symbols_of(nodes) if s.id not in self.names]
        if free:
            raise ValueError("%s depends on symbols that are not time/robot/virtual/input "
                             "variables of the skill: %s" % (what, sorted(set(free))))


def _constraint_rows(spec, n_rob, n_virt, n_slack):
    """Rows of  lb <= A x <= ub  over x = [robot vel; virtual vel; slack], one per constraint row:
    [de/dq | de/dx | -1 on the row's own slack if soft]            reactive_qp.py:191-246.
    -> (A as lists of nodes, lb nodes, ub nodes, row labels)."""
    A, lbs, ubs, labels = [], [], [], []
    slack_ind = 0
    for c in spec.constraints:
        kind = kind_of(c)
        e = c.expression
        rows = e.size()[0]
        Jq = cs.jacobian(e, spec.robot_var)
        Jx = cs.jacobian(e, spec.virtual_var) if spec.virtual_var is not None else None
        Jt = cs.jacobian(e, spec.time_var)
        lb = -Jt
        ub = -Jt
        if kind == KIND_EQ:
            ke = c.gain_times(e)
            lb = lb + (-ke)
            ub = ub + (-ke)
        elif kind == KIND_SET:
            smin = cs.MX(cs.vertcat(*_col(c.set_min, rows, "set_min", c.label)))
            smax = cs.MX(cs.vertcat(*_col(c.set_max, rows, "set_max", c.label)))
            lb = lb + c.gain_times(smin - e)
            ub = ub + c.gain_times(smax - e)
        elif kind == KIND_VELEQ:
            tg = cs.MX(cs.vertcat(*_col(c.target, rows, "target", c.label)))
            lb = lb + tg
            ub = ub + tg
        else:
            lb = lb + cs.MX(cs.vertcat(*_col(c.set_min, rows, "set_min", c.label)))
            ub = ub + cs.MX(cs.vertcat(*_col(c.set_max, rows, "set_max", c.label)))
        soft = c.constraint_type == "soft"
        for r in range(rows):
            row = [Jq._a[r, k] for k in range(n_rob)]
            if Jx is not None:
                row += [Jx._a[r, k] for k in range(n_virt)]
            srow = [dag.ZERO] * n_slack
            if soft:
                srow[slack_ind + r] = dag.MINUS_ONE
            A.append(row + srow)
            labels.append("%s[%d]" % (c.label, r))
        if soft:
            slack_ind += rows
        lbs += lb.nodes()
        ubs += ub.nodes()
    return A, lbs, ubs, labels


def _classify_rows(A):
    """Row structure: a "unit" row has exactly one structural non-zero and it is a constant (bounds on
    a single variable: joint limits, speed limits); everything else is dense.
    -> ([(row, column, coefficient)], [dense row indices])."""
    unit_rows, dense_rows = [], []
    for r, row in enumerate(A):
        nz = [(j, n) for j, n in enumerate(row) if n is not dag.ZERO]
        if len(nz) == 1 and nz[0][1].is_const and nz[0][1].val != 0.0:
            unit_rows.append((r, nz[0][0], nz[0][1].val))
        else:
            dense_rows.append(r)
    return unit_rows, dense_rows


class PinvProgram(object):
    """Per-constraint numeric blocks for the pseudo-inverse controller."""

    def __init__(self, spec, options):
        self.syms = Symbols(spec)
        self.n_rob = spec.n_robot_var
        self.n_virt = spec.n_virtual_var if spec.virtual_var is not None else 0
        self.n_in = len(self.syms.y)
        self.ns = self.n_rob + self.n_virt
        state = spec.robot_var if spec.virtual_var is None else cs.vertcat(spec.robot_var,
                                                                         spec.virtual_var)
        ff = bool(options["feedforward"])
        self.multidim = bool(options["multidim_sets"])
        self.conv_last = bool(options["converge_final_set_to_max"])
        method = options["pinv_method"]
        if method not in ("damped", "standard"):
            raise ValueError("pinv_method must be 'damped' or 'standard'")
        self.damped = method == "damped"
        self.damping = float(options["damping_factor"])
        self.blocks = []
        row = 0
        set_idx = 0
        for c in spec.constraints:
            kind = kind_of(c)
            if kind == KIND_VELSET:
                continue  # no branch of the reference's loop matches it (Appendix A6)
            rows = c.expression.size()[0]
            if kind == KIND_SET and rows > 1 and not self.multidim:
                raise NotImplementedError(
                    "PseudoInverseController does not yet have guaranteed stable support for "
                    "multidimensional SetConstraints. Size(" + c.label + ")=" + str(rows)
                    + ". Set the multidim_sets field in options to True for experimental support.")
            e = c.expression
            J = cs.jacobian(e, state)
            Jt = cs.jacobian(e, spec.time_var)
            blk = {"kind": kind, "rows": rows, "row0": row, "label": c.label, "set_index": -1,
                   "e": e.nodes(), "jt": Jt.nodes(),
                   "J": [[J._a[r, k] for k in range(self.ns)] for r in range(rows)]}
            if kind == KIND_EQ:
                des = -c.gain_times(e)
                if ff:
                    des = des + (-Jt)
                blk["des"] = des.nodes()
            elif kind == KIND_VELEQ:
                des = cs.MX(cs.vertcat(*_col(c.target, rows, "target", c.label)))
                if ff:
                    des = des + (-Jt)
                blk["des"] = des.nodes()
            else:
                blk["smin"] = _col(c.set_min, rows, "set_min", c.label)
                blk["smax"] = _col(c.set_max, rows, "set_max", c.label)
                if self.multidim:
                    # S = diag(e - max > 0 or e - min < 0)              pseudo_inverse.py:289-298
                    blk["rmask"] = [dag.logic_or(dag.lt(dag.ZERO, dag.sub(en, mx)), dag.lt(dag.sub(en, mn), dag.ZERO))
                                    for en, mn, mx in zip(blk["e"], blk["smin"], blk["smax"])]
                blk["set_index"] = set_idx
                set_idx += 1
            self.blocks.append(blk)
            row += rows
        if not self.blocks:
            raise ValueError("skill has no constraint the pseudo-inverse controller can use")
        # converge_final_set_to_max (pseudo_inverse.py:337-356): when the LAST constraint is a
        # SetConstraint and it is active, it also drives its expression to set_max through the
        # null space of everything above it.  `is_last` in the reference refers to the full
        # constraint list, so a trailing VelocitySetConstraint switches the option off.
        last = spec.constraints[-1] if spec.constraints else None
        self.conv_last = (self.conv_last and last is not None and kind_of(last) == KIND_SET
                          and self.blocks[-1]["kind"] == KIND_SET)
        if self.conv_last:
            if not any(b["kind"] in (KIND_EQ, KIND_VELEQ) for b in self.blocks[:-1]):
                raise ValueError("converge_final_set_to_max needs an Equality / VelocityEquality constraint "
                                 "above the final set: with an empty active list the reference fails at "
                                 "setup (cs.vertcat(*[]), pseudo_inverse.py:343)")
            b = self.blocks[-1]
            c = last
            e = c.expression
            des = c.gain_times(cs.MX(cs.vertcat(*b["smax"])) - e)
            if ff:
                des = des + (-cs.jacobian(e, spec.time_var))
            b["des"] = des.nodes()
        self.m = row
        self.n_sets = set_idx
        self.max_rows = max(b["rows"] for b in self.blocks)
        # "unit sets": every SetConstraint bounds a single state coordinate with a constant
        # coefficient (joint limits: e = q_k), on distinct coordinates, and the only Eq / VelEq
        # constraint comes after all of them.  Then the stacked active-set Jacobian has
        # S S' = diag(c_k^2) and a mode's null-space projector is a per-coordinate scaling.
        self.unit_sets = None
        sets = [b for b in self.blocks if b["kind"] == KIND_SET]
        tasks = [b for b in self.blocks if b["kind"] in (KIND_EQ, KIND_VELEQ)]
        if sets and len(tasks) == 1 and self.blocks[-1] is tasks[0] and not self.multidim and not self.conv_last:
            info, cols = [], set()
            for b in sets:
                nz = [(j, n) for j, n in enumerate(b["J"][0]) if n is not dag.ZERO]
                if len(nz) == 1 and nz[0][1].is_const and nz[0][1].val != 0.0 and nz[0][0] not in cols:
                    cols.add(nz[0][0])
                    info.append((nz[0][0], nz[0][1].val))
                else:
                    info = None
                    break
            self.unit_sets = info
        for b in self.blocks:
            nodes = b["e"] + b["jt"] + [n for r in b["J"] for n in r]
            nodes += b.get("des", []) + b.get("smin", []) + b.get("smax", []) + b.get("rmask", [])
            self.syms.check_closed(nodes, "constraint " + b["label"])


class QpProgram(object):
    """H diagonal, A, lb, ub of the reactive QP (x = [robot vel; virtual vel; slack])."""

    def __init__(self, spec, w_rob, w_virt, w_slack, mu):
        self.syms = Symbols(spec)
        self.n_rob = spec.n_robot_var
        self.n_virt = spec.n_virtual_var if spec.virtual_var is not None else 0
        self.n_in = len(self.syms.y)
        self.n_slack = spec.n_slack_var
        self.nx = self.n_rob + self.n_virt + self.n_slack
        # cost: H = diag([mu*w_rob ; mu*w_virt ; mu + w_slack])        reactive_qp.py:175-189
        parts = [mu * w_rob]
        if self.n_virt > 0:
            parts.append(mu * w_virt)
        if self.n_slack > 0:
            parts.append(mu + w_slack)
        self.h = cs.vertcat(*parts).nodes()
        if len(self.h) != self.nx:
            raise ValueError("weights do not match the number of optimisation variables")
        self.A, self.lb, self.ub, self.labels = _constraint_rows(spec, self.n_rob, self.n_virt, self.n_slack)
        self.m = len(self.A)
        nodes = self.h + self.lb + self.ub + [n for r in self.A for n in r]
        self.syms.check_closed(nodes, "QP matrices")
        self.unit_rows, self.dense_rows = _classify_rows(self.A)


#: capacity of the in-kernel NLP solver (the tiers of the dense QP core it calls, clik_qp_dense)
NLP_MAX_NX, NLP_MAX_M = 32, 64


class NlpProgram(object):
    """Linearly constrained NLP of the reactive NLP controller over x = [robot vel; virtual vel; slack]:

        min F(x)   s.t.  lb <= A x <= ub

    with A, lb, ub exactly as QpProgram builds them.  `objective` is the whole scalar F, as
    ReactiveNLPController.get_cost_expr composes it (the one place that states the cost convention).
    Holds F, its gradient `g` and the lower triangle of H = d2F/dx2 (row-major packed:
    H[i*(i+1)/2 + j], j <= i) as scalar nodes over the decision symbols `dec` (robot_vel_var;
    virtual_vel_var; slack_var) and t, q, x, y; `quadratic` is true when no entry of H depends on a
    decision symbol."""

    def __init__(self, spec, objective):
        self.syms = Symbols(spec)
        self.n_rob = spec.n_robot_var
        self.n_virt = spec.n_virtual_var if spec.virtual_var is not None else 0
        self.n_slack = spec.n_slack_var
        self.nx = self.n_rob + self.n_virt + self.n_slack
        if not isinstance(objective, cs.GenericMatrixCommon):
            objective = cs.DM(objective)
        if tuple(objective.size()) != (1, 1):
            raise ValueError("the cost must be a scalar (1x1) expression, got %dx%d" % tuple(objective.size()))
        self.dec = list(spec.robot_vel_var.nodes())
        if self.n_virt > 0:
            self.dec += spec.virtual_vel_var.nodes()
        if self.n_slack > 0:
            self.dec += spec.slack_var.nodes()
        cost = objective.nodes()[0]
        # a cost that reads the input although no constraint does: the input rows become kernel inputs
        if spec.input_var is not None and not self.syms.y:
            yn = spec.input_var.nodes()
            if dag.depends_on([cost], yn):
                self.syms.y = yn
                for i, n in enumerate(yn):
                    self.syms.names[n.id] = "y[%d]" % i
        self.n_in = len(self.syms.y)
        dec_ids = {n.id for n in self.dec}
        free = [s.name for s in dag.symbols_of([cost]) if s.id not in self.syms.names and s.id not in dec_ids]
        if free:
            raise ValueError("the cost depends on symbols that are not time/robot/virtual/input variables or "
                             "decision variables (robot_vel_var, virtual_vel_var, slack_var) of the skill: %s"
                             % sorted(set(free)))
        self.A, self.lb, self.ub, self.labels = _constraint_rows(spec, self.n_rob, self.n_virt, self.n_slack)
        self.m = len(self.A)
        if self.nx > NLP_MAX_NX or self.m > NLP_MAX_M:
            raise ValueError("the NLP controller supports at most %d decision variables and %d constraint rows "
                             "(this skill: %d x %d)" % (NLP_MAX_NX, NLP_MAX_M, self.nx, self.m))
        self.syms.check_closed(self.lb + self.ub + [n for r in self.A for n in r], "NLP constraints")
        self.unit_rows, self.dense_rows = _classify_rows(self.A)
        self.F = cost
        self.g = dag.jacobian([cost], self.dec)[0]
        Hfull = dag.jacobian(self.g, self.dec)
        self.H = [Hfull[i][j] for i in range(self.nx) for j in range(i + 1)]
        self.quadratic = not dag.depends_on(self.H, self.dec)
