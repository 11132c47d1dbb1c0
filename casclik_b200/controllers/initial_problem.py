"""Initial-value problem of the reactive QP controller: choose virtual velocities and slack
for a given (fixed) robot velocity before the control loop starts.

Mirrors reference casclik/controllers/reactive_qp.py:300-459:
  variables  [virtual_vel ; slack],  H = diag([mu*w_virt ; (1+mu)*w_slack])           (:324-332)
  rows       only constraints that touch a virtual variable or own slack                 (:383-386)
  bounds     -de/dt - (de/dq) robot_vel + the usual per-type terms                       (:354-370)
`solve` (one instance, what the reference offers) evaluates the matrices on the host from the
expression graph and sends the QP through the dense CUDA QP entry point (clik_qp_dense).
`solve_batch` (N instances: every rollout of a batch needs its own initial slack / virtual velocity)
lowers the same expressions through the expression compiler into a fused QP kernel of their own:
the robot velocity is one more per-instance input, appended to input_var on the kernel side.
"""
import numpy as np

from .. import sym as cs
from ..sym import dag
from ..codegen.lower import kind_of, KIND_EQ, KIND_SET, KIND_VELEQ, _col
from .qp_solver import ConicSolver


class InitialProblem(object):
    def __init__(self, ctrl):
        spec = ctrl.skill_spec
        self.spec = spec
        nvirt = spec.n_virtual_var if spec.virtual_var is not None else 0
        nslack = spec.n_slack_var
        mu = ctrl.weight_shifter
        self.nvirt, self.nslack = nvirt, nslack
        weights = []
        if nvirt > 0:
            weights.append(mu * ctrl.virtual_var_weights)
        if nslack > 0:
            weights.append((1 + mu) * ctrl.slack_var_weights)
        self.active = False
        if not weights:
            return
        H = cs.diag(cs.vertcat(*weights))
        rows_A, rows_lb, rows_ub = [], [], []
        slack_ind = 0
        found_any = False
        for c in spec.constraints:
            e = c.expression
            rows = e.size()[0]
            kind = kind_of(c)
            found_virt = found_slack = False
            if nvirt > 0:
                Jv = cs.jacobian(e, spec.virtual_var)
                if Jv.nnz() > 0:
                    found_virt = True
                    expr = Jv
                else:
                    expr = cs.DM.zeros(rows, nvirt)
            Jt = cs.jacobian(e, spec.time_var)
            rob_der = c.jtimes(spec.robot_var, spec.robot_vel_var)
            lb = -Jt - rob_der
            ub = -Jt - rob_der
            if kind == KIND_EQ:
                ke = c.gain_times(e)
                lb, ub = lb + (-ke), ub + (-ke)
            elif kind == KIND_SET:
                smin = cs.MX(cs.vertcat(*_col(c.set_min, rows, "set_min", c.label)))
                smax = cs.MX(cs.vertcat(*_col(c.set_max, rows, "set_max", c.label)))
                lb, ub = lb + c.gain_times(smin - e), ub + c.gain_times(smax - e)
            elif kind == KIND_VELEQ:
                tg = cs.MX(cs.vertcat(*_col(c.target, rows, "target", c.label)))
                lb, ub = lb + tg, ub + tg
            else:
                lb = lb + cs.MX(cs.vertcat(*_col(c.set_min, rows, "set_min", c.label)))
                ub = ub + cs.MX(cs.vertcat(*_col(c.set_max, rows, "set_max", c.label)))
            if nslack > 0:
                smat = cs.DM.zeros(rows, nslack)
                if c.constraint_type == "soft":
                    smat[:, slack_ind:slack_ind + rows] = -cs.DM.eye(rows)
                    slack_ind += rows
                    found_slack = True
                expr = cs.horzcat(expr, smat) if nvirt > 0 else smat
            if found_virt or found_slack:
                found_any = True
                rows_A.append(expr)
                rows_lb.append(lb)
                rows_ub.append(ub)
        if not found_any:
            return
        ins = [spec.time_var, spec.robot_var, spec.robot_vel_var]
        names = ["time_var", "robot_var", "robot_vel_var"]
        if spec._has_virtual:
            ins.append(spec.virtual_var)
            names.append("virtual_var")
        if spec._has_input:
            ins.append(spec.input_var)
            names.append("input_var")
        self.funcs = {
            "H": cs.Function("H_initial", ins, [H], names, ["H"]),
            "A": cs.Function("A_initial", ins, [cs.vertcat(*rows_A)], names, ["A"]),
            "Blb": cs.Function("Blb_initial", ins, [cs.vertcat(*rows_lb)], names, ["Blb"]),
            "Bub": cs.Function("Bub_initial", ins, [cs.vertcat(*rows_ub)], names, ["Bub"]),
        }
        self.solver = ConicSolver("solver", ctrl.options["solver_name"], {},
                                  ctrl.options["initial_solver_opts"])
        self.active = True
        self._exprs = (H, cs.vertcat(*rows_A), cs.vertcat(*rows_lb), cs.vertcat(*rows_ub))
        self._batch = None

    # ---- N instances ---------------------------------------------------------------------------------
    def _batch_setup(self):
        """Emit + compile the fused kernel of the initial QP (cached like every skill cubin)."""
        from .. import build, runtime
        from ..codegen import emit_skill
        prog = InitialQpProgram(self.spec, *self._exprs)
        source, meta = emit_skill(qp=prog, label=self.spec.label + "_initial")
        cubin, path = build.compile_cubin(source, tag="qpinit_" + self.spec.label)
        self._batch = {"prog": prog, "meta": meta, "cubin": cubin, "path": path, "skills": {}}
        return self._batch

    def solve_batch(self, t0, q0, x0=None, dq0=None, y0=None, max_iter=0):
        """reactive_qp.py:426-459 for N instances.  q0 (n_robot, N), x0 (n_virtual, N) | None (zeros),
        dq0 (n_robot, N) | None (zeros), y0 (n_input, N): torch CUDA tensors (or NumPy arrays -> host path).
        Returns (virtual_vel (n_virtual, N) | None, slack (n_slack, N) | None, status (N,) int32)."""
        from .. import runtime
        from .base_controller import Batch, run_step
        b = self._batch or self._batch_setup()
        prog = b["prog"]
        on_dev = runtime._is_torch(q0)
        if on_dev:
            import torch
            N = int(q0.shape[1])
            dq = torch.zeros_like(q0) if dq0 is None else dq0
            y = dq if prog.n_y_user == 0 else torch.cat([y0, dq], dim=0).contiguous()
        else:
            q0 = np.ascontiguousarray(q0, dtype=np.float64)
            N = q0.shape[1]
            dq = np.zeros_like(q0) if dq0 is None else np.ascontiguousarray(dq0, dtype=np.float64)
            y = dq if prog.n_y_user == 0 else np.ascontiguousarray(np.vstack([np.asarray(y0, dtype=np.float64), dq]))
        batch = Batch(prog.n_rob, prog.n_virt, prog.n_in, t0, q0, x0, y)

        def skill(dev):
            if dev not in b["skills"]:
                b["skills"][dev] = runtime.CompiledSkill(b["cubin"], b["meta"], n_slack=self.nslack, device=dev)
            return b["skills"][dev]

        sol, status, active = batch.empty(prog.nx), batch.empty(0, "i32"), batch.empty(2, "i32")
        run_step(skill, "qp", batch, None, None, None, batch.ptr(sol), batch.ptr(status), batch.ptr(active),
                 int(max_iter))
        virt = sol[:self.nvirt] if self.nvirt > 0 else None
        slack = sol[self.nvirt:self.nvirt + self.nslack] if self.nslack > 0 else None
        return virt, slack, status

    def solve(self, t0, q0, x0=None, dq0=None, y0=None):
        spec = self.spec
        if dq0 is None:
            dq0 = [0.0] * spec.n_robot_var
        vals = [t0, q0, dq0]
        if spec._has_virtual:
            vals.append([0.0] * self.nvirt if x0 is None else x0)
        if spec._has_input:
            vals.append([0.0] * spec.n_input_var if y0 is None else y0)
        H, A, lb, ub = (self.funcs[k](*vals) for k in ("H", "A", "Blb", "Bub"))
        res = self.solver(h=H, a=A, lba=lb, uba=ub)
        x = np.asarray(res["x"].toarray()).reshape(-1)
        res_virt = cs.DM(x[:self.nvirt].reshape(-1, 1)) if self.nvirt > 0 else None
        res_slack = (cs.DM(x[self.nvirt:self.nvirt + self.nslack].reshape(-1, 1))
                     if self.nslack > 0 else None)
        return res_virt, res_slack


class InitialQpProgram(object):
    """The initial-value QP in the shape codegen.emit_skill expects of a QP program (see
    codegen.lower.QpProgram): variables [virtual_vel; slack], and the fixed robot velocity as extra
    per-instance inputs y[n_input .. n_input + n_robot)."""
    emit_rollout = False        # the solution holds no robot velocity: nothing to integrate

    def __init__(self, spec, H, A, lb, ub):
        from ..codegen.lower import Symbols
        self.syms = Symbols(spec)
        self.n_y_user = len(self.syms.y)
        for k, n in enumerate(spec.robot_vel_var.nodes()):
            self.syms.names[n.id] = "y[%d]" % (self.n_y_user + k)
        self.syms.y = list(self.syms.y) + list(spec.robot_vel_var.nodes())
        self.n_rob = spec.n_robot_var
        self.n_virt = spec.n_virtual_var if spec.virtual_var is not None else 0
        self.n_in = len(self.syms.y)
        Hm, Am = cs.MX(H), cs.MX(A)
        self.nx = Hm.shape[0]
        self.h = [Hm._a[k, k] for k in range(self.nx)]
        self.m = Am.shape[0]
        self.A = [[Am._a[r, c] for c in range(self.nx)] for r in range(self.m)]
        self.lb, self.ub = cs.MX(lb).nodes(), cs.MX(ub).nodes()
        self.labels = ["initial[%d]" % r for r in range(self.m)]
        nodes = self.h + self.lb + self.ub + [n for r in self.A for n in r]
        self.syms.check_closed(nodes, "initial-value QP")
        self.unit_rows, self.dense_rows = [], []
        for r, row in enumerate(self.A):
            nz = [(j, n) for j, n in enumerate(row) if n is not dag.ZERO]
            if len(nz) == 1 and nz[0][1].is_const and nz[0][1].val != 0.0:
                self.unit_rows.append((r, nz[0][0], nz[0][1].val))
            else:
                self.dense_rows.append(r)
