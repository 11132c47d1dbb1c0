"""ReactiveNLPController — reactive controller with a general smooth cost, evaluated on the GPU for one
or N instances.

Counterpart of the reference's casclik/controllers/reactive_nlp.py (setup :254-277, solve :469-534):
the decision variables and the constraint rows are those of the reactive QP
(x = [robot vel; virtual vel; slack], lb <= A x <= ub, rows as ReactiveQPController builds them), only
the objective is a user expression `cost_expr(t, q, x, y; robot_vel_var, virtual_vel_var)` instead of
the fixed diagonal quadratic.  The reference hands the problem to IPOPT through cs.nlpsol; here setup
emits one CUDA kernel that evaluates the constraint rows once per step and runs an exact-Hessian SQP per
thread over the dense QP core (csrc/clik_nlp.cuh).

The cost convention (get_cost_expr) is a restatement of the reference from memory that could not be
checked against its source; DESIGN.md §4.4 says so.  Like cs.nlpsol, `solve` does not raise when the
solver does not converge: the outcome is in `self.res["status"]`.
"""
import ctypes

import numpy as np

from .. import build, runtime
from .. import sym as cs
from ..codegen import NlpProgram, emit_skill
from ..sym import dag
from .base_controller import (BaseController, Batch, as_vector, dm_column, multipliers_batch, one_instance, run_step,
                              jacobian_batch, jvp_batch, rollout_batch_differentiable, rollout_jacobian, rollout_jvp,
                              rollout_vjp, solve_batch_differentiable, vjp_batch)
from .reactive_qp import _weights

#: per-instance outcome of the NLP step (status array): the QP codes plus a stalled line search
NLP_SOLVED, NLP_MAXITER, NLP_INFEASIBLE, NLP_INVALID, NLP_STALLED = 0, 1, 2, 4, 5


class ReactiveNLPController(BaseController):
    """Reactive NLP controller.

    Args:
        skill_spec (SkillSpecification): skill specification
        cost_expr (cs.MX): scalar cost of time/robot/virtual/input variables and the decision variables
            robot_vel_var / virtual_vel_var (and slack_var) of the skill
        slack_var_weights: weights of the slack penalty; default cnstr.slack_weight per soft row
        options (dict): solver_name (default "ipopt"), solver_opts, function_opts (accepted for
            compatibility, not used), "max_iter" (SQP iteration cap, default 50) and "tol" (default 1e-10).
            A step is solved when the last SQP step p has |p|_inf * max(1, delta) <= tol * (1 + |x|_inf)
            (delta: the shift that made the Hessian positive definite, 0 for a convex cost), or when a step
            with |p|_inf <= 100 * tol * (1 + |x|_inf) left the cost unchanged within its rounding (1e-15
            relative): the subproblem's own accuracy can keep |p| a few tol above tol (DESIGN.md §4.4).
    """
    controller_type = "ReactiveNLPController"
    options_info = """solver_name, solver_opts, function_opts, max_iter, tol"""
    weight_shifter = 0.001  # eTaSL's mu

    def __init__(self, skill_spec, cost_expr, slack_var_weights=None, options=None):
        self.skill_spec = skill_spec
        self.cost_expr = cost_expr
        self.slack_var_weights = slack_var_weights
        self.options = options
        self._cubin = None
        self._compiled = {}
        self._vjp = None
        self._jvp = None
        self._rollout_jvp = None
        self._rollout_vjp = None
        self._has_initial = False
        self.res = None
        self._prog = self._program()     # validates the cost and the problem size now

    # ---- weights / options ------------------------------------------------------------------------
    @property
    def slack_var_weights(self):
        return self._slack_var_weights

    @slack_var_weights.setter
    def slack_var_weights(self, weights):
        if weights is None:
            vals = []
            for c in self.skill_spec.constraints:
                if c.constraint_type == "soft":
                    vals += [c.slack_weight] * c.expression.size()[0]
            weights = vals
        self._slack_var_weights = _weights(weights, self.skill_spec.n_slack_var,
                                           "slack_var_weights", "slack_var")

    @property
    def options(self):
        return self._options

    @options.setter
    def options(self, opt):
        if opt is None or not isinstance(opt, dict):
            opt = {}
        opt.setdefault("solver_name", "ipopt")
        opt.setdefault("solver_opts", {})
        opt.setdefault("function_opts", {})
        opt.setdefault("max_iter", 50)
        opt.setdefault("tol", 1e-10)
        if not (int(opt["max_iter"]) > 0):
            raise ValueError("options['max_iter'] must be a positive integer")
        if not (float(opt["tol"]) > 0.0 and np.isfinite(float(opt["tol"]))):
            raise ValueError("options['tol'] must be a positive number")
        self._options = opt

    # ---- expressions ------------------------------------------------------------------------------
    def get_cost_expr(self):
        """The objective the kernel minimises:

            cost_expr + slack' diag(weight_shifter + slack_var_weights) slack

        (no factor 1/2 on the slack term).  This is the only place that states the convention; it is a
        restatement of the reference's reactive_nlp.py that could not be checked (DESIGN.md §4.4)."""
        spec = self.skill_spec
        cost = self.cost_expr if isinstance(self.cost_expr, cs.GenericMatrixCommon) else cs.MX(cs.DM(self.cost_expr))
        if spec.n_slack_var > 0:
            w = self.weight_shifter + self.slack_var_weights
            cost = cost + cs.dot(spec.slack_var, w * spec.slack_var)
        return cost

    def get_constraints_expr(self):
        prog = self._prog
        A = cs.MX(cs.vertcat(*[cs.horzcat(*row) for row in prog.A]))
        return A, cs.MX(cs.vertcat(*prog.lb)), cs.MX(cs.vertcat(*prog.ub))

    def _program(self):
        return NlpProgram(self.skill_spec, self.get_cost_expr())

    # ---- setup ------------------------------------------------------------------------------------
    def setup_problem_functions(self, load=True):
        """Emit + compile (+ load) the NLP kernels of the skill."""
        prog = self._prog = self._program()
        source, meta = emit_skill(nlp=prog, label=self.skill_spec.label, nlp_tol=float(self.options["tol"]))
        cubin, path = build.compile_cubin(source, tag="nlp_" + self.skill_spec.label)
        self.kernel_source, self.kernel_meta, self.cubin_path = source, meta, path
        self._nxv, self._ny, self._qn, self._qm = prog.n_virt, prog.n_in, prog.nx, prog.m
        self.row_labels = prog.labels
        self._cubin = cubin
        self._compiled = {}
        self._vjp = None
        self._jvp = None
        self._rollout_jvp = None
        self._rollout_vjp = None
        if load:
            self._skill()

    def setup_solver(self):
        """Compiles and loads the kernels if setup_problem_functions has not (either order works)."""
        if self._cubin is None:
            self.setup_problem_functions()

    def _max_iter(self, max_iter):
        return int(max_iter if max_iter is not None else self.options["max_iter"])

    # ---- initial problem ----------------------------------------------------------------------------
    def setup_initial_problem_solver(self):
        spec = self.skill_spec
        self._has_initial = (spec.virtual_var is not None and spec._has_virtual) or spec.n_slack_var > 0
        return None

    def solve_initial_problem(self, time_var0, robot_var0, virtual_var0=None, robot_vel_var0=None,
                              input_var0=None):
        spec = self.skill_spec
        if not ((spec.virtual_var is not None and spec._has_virtual) or spec.n_slack_var > 0):
            return None, None
        raise NotImplementedError("the initial-value problem of the NLP controller (virtual velocities and slack "
                                  "with the robot velocity fixed) is not implemented yet; it is the follow-up "
                                  "to this controller (DESIGN.md §8)")

    # ---- step --------------------------------------------------------------------------------------
    def solve_batch(self, time_var, robot_var, virtual_var=None, input_var=None, warmstart=None, out=None,
                    max_iter=None, devices=None):
        """NLP controller step for N instances (layout of ReactiveQPController.solve_batch): torch CUDA
        tensors run on their device (asynchronously on the current stream), NumPy arrays go through the
        host entry point.  warmstart: optional (nx, N) start point of the SQP iteration (the first
        subproblem restores feasibility from it).
        devices: as in PseudoInverseController.solve_batch (host arrays sharded over several GPUs,
        bit-identical to one GPU).
        Returns (sol (nx, N), status (N,) int32, active (2, N) int32 bit masks [upper; lower] of the last
        subproblem's working set, iterations (N,) int32)."""
        spec = self.skill_spec
        b = Batch(spec.n_robot_var, self._nxv, self._ny, time_var, robot_var, virtual_var,
                  input_var if self._ny else None)
        if out is None:
            sol, status, active, iters = b.empty(self._qn), b.empty(0, "i32"), b.empty(2, "i32"), b.empty(0, "i32")
        else:
            sol, status, active, iters = out
            if sol is None:
                raise runtime.ClikError("out=(sol, status, active, iterations): the solution buffer is required")
        solp = b.out_ptr(sol, self._qn, "f64", "out[0] (sol)")
        stp = b.out_ptr(status, 0, "i32", "out[1] (status)")
        acp = b.out_ptr(active, 2, "i32", "out[2] (active)")
        itp = b.out_ptr(iters, 0, "i32", "out[3] (iterations)")
        x0p = None
        if warmstart is not None:
            if b.on_device:
                x0p = runtime.dev_ptr(warmstart, "f64", self._qn * b.N, "warmstart")
            else:
                x0p, warmstart = runtime.host_ptr(warmstart, np.float64, self._qn * b.N, "warmstart")
        run_step(self._skill, "nlp", b, devices, x0p, solp, stp, itp, acp, self._max_iter(max_iter))
        return sol, status, active, iters

    def multipliers_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, out=None):
        """Constraint multipliers (the reference's lam_g) of a solve_batch result, as
        ReactiveQPController.multipliers_batch: lam (m, N) float64 with grad F + A' lam = 0 on the last
        subproblem's working set; NaN for an instance whose status is not 0 (include/clik.h clik_nlp_duals)."""
        return multipliers_batch(self, "nlp", time_var, robot_var, virtual_var, input_var, sol, status, active, out)

    def _vjp_source(self):
        """Source of the VJP image: the default image plus the VJP kernel."""
        return emit_skill(nlp=self._prog, label=self.skill_spec.label, nlp_tol=float(self.options["tol"]), vjp=True)

    def vjp_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, sol_bar, out=None):
        """Reverse-mode derivative of a solve_batch result, as ReactiveQPController.vjp_batch; the adjoint solve
        uses the Hessian of the cost at sol, factored without a shift: an instance whose Hessian is not positive
        definite there gets NaN (include/clik.h clik_nlp_vjp)."""
        return vjp_batch(self, "nlp", time_var, robot_var, virtual_var, input_var, sol, status, active, sol_bar, out)

    def _jvp_source(self):
        """Source of the JVP image: the default image plus the JVP and Jacobian kernels."""
        return emit_skill(nlp=self._prog, label=self.skill_spec.label, nlp_tol=float(self.options["tol"]), jvp=True)

    def jvp_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, t_dot=None, q_dot=None,
                  x_dot=None, y_dot=None, out=None):
        """Forward-mode derivative of a solve_batch result, as ReactiveQPController.jvp_batch; the solve uses the
        Hessian of the cost at sol, factored without a shift (include/clik.h clik_nlp_jvp)."""
        return jvp_batch(self, "nlp", time_var, robot_var, virtual_var, input_var, sol, status, active, t_dot, q_dot,
                         x_dot, y_dot, out)

    def jacobian_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, out=None):
        """The full step Jacobian (nx, n_theta, N) of a solve_batch result, as ReactiveQPController.jacobian_batch."""
        return jacobian_batch(self, "nlp", time_var, robot_var, virtual_var, input_var, sol, status, active, out)

    def solve_batch_differentiable(self, time_var, robot_var, virtual_var=None, input_var=None, warmstart=None,
                                   max_iter=None):
        """solve_batch on torch CUDA tensors as a torch.autograd.Function (see
        ReactiveQPController.solve_batch_differentiable): (sol, status, active, iterations), sol differentiable."""
        return solve_batch_differentiable(self, time_var, robot_var, virtual_var, input_var, warmstart, max_iter)

    def rollout_batch(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None,
                      max_speed=None, max_virtual_speed=None, max_iter=None):
        """Closed-loop simulation on the device (see ReactiveQPController.rollout_batch): robot_var /
        virtual_var (torch CUDA, (n, N)) are UPDATED IN PLACE; every step starts its SQP iteration from the
        previous step's solution.  Returns a dict with the last solution `sol` (nx, N) and `n_failed`
        (steps that were not solved: zero velocity)."""
        spec = self.skill_spec
        b = Batch(spec.n_robot_var, self._nxv, self._ny, time_var0, robot_var, virtual_var,
                  input_var if self._ny else None)
        if not b.on_device:
            raise ValueError("rollout_batch needs CUDA tensors (state is updated in place on the device)")
        skill = self._skill(b.device_index)
        if self._nxv and virtual_var is None:
            raise ValueError("the skill has a virtual_var: pass its initial value")
        sol, failed = b.empty(self._qn), b.empty(0, "i32")
        inf = float("inf")
        runtime.check(runtime.load_library().clik_nlp_rollout(
            skill.handle, b.N, int(steps), ctypes.c_double(float(dt)), b.tp, b.t_stride, b.qp, b.xp, b.yp,
            ctypes.c_double(inf if max_speed is None else float(max_speed)),
            ctypes.c_double(inf if max_virtual_speed is None else float(max_virtual_speed)),
            b.ptr(sol), b.ptr(failed), self._max_iter(max_iter), b.stream()))
        return {"sol": sol, "n_failed": failed}

    def _rollout_jvp_source(self):
        """Source of the rollout-JVP image: the JVP image plus the tangent and Jacobian rollout kernels."""
        return emit_skill(nlp=self._prog, label=self.skill_spec.label, nlp_tol=float(self.options["tol"]), jvp=True,
                          rollout_jvp=True)

    def rollout_jvp(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None, max_speed=None,
                    max_virtual_speed=None, max_iter=None, t_dot=None, q_dot=None, x_dot=None, y_dot=None):
        """rollout_batch with the tangent of the closed loop, as ReactiveQPController.rollout_jvp; each step's
        tangent is the jvp_batch tangent of its solution (Hessian at sol, no shift: NaN where it is not positive
        definite).  The dependence of a step on its warm start (below tol) is not differentiated."""
        return rollout_jvp(self, "nlp", time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                           max_virtual_speed, self._max_iter(max_iter), t_dot, q_dot, x_dot, y_dot)

    def rollout_jacobian(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None, max_speed=None,
                         max_virtual_speed=None, max_iter=None):
        """rollout_batch with d(q_K, x_K)/d(t0, q0, x0, y), as ReactiveQPController.rollout_jacobian."""
        return rollout_jacobian(self, "nlp", time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                                max_virtual_speed, self._max_iter(max_iter))

    def _rollout_vjp_source(self):
        """Source of the rollout-VJP image: the VJP image plus the taped rollout and reverse sweep kernels."""
        return emit_skill(nlp=self._prog, label=self.skill_spec.label, nlp_tol=float(self.options["tol"]), vjp=True,
                          rollout_vjp=True)

    def rollout_vjp(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None, max_speed=None,
                    max_virtual_speed=None, max_iter=None, q_bar=None, x_bar=None, sol_bar=None):
        """rollout_batch followed by the reverse sweep of the closed loop, as ReactiveQPController.rollout_vjp; each
        step's cotangent is pulled back with the vjp_batch of its solution (Hessian at sol, no shift: NaN where it
        is not positive definite).  The dependence of a step on its warm start (below tol) is not differentiated."""
        return rollout_vjp(self, "nlp", time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                           max_virtual_speed, self._max_iter(max_iter), q_bar, x_bar, sol_bar)

    def rollout_batch_differentiable(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None,
                                     max_speed=None, max_virtual_speed=None, max_iter=None):
        """rollout_batch as a torch.autograd.Function, as ReactiveQPController.rollout_batch_differentiable."""
        return rollout_batch_differentiable(self, "nlp", time_var0, robot_var, steps, dt, virtual_var, input_var,
                                            max_speed, max_virtual_speed, self._max_iter(max_iter))

    def solve(self, time_var, robot_var, virtual_var=None, input_var=None,
              warmstart_robot_vel_var=None, warmstart_virtual_vel_var=None, warmstart_slack_var=None):
        """One controller step -> (robot_vel, virtual_vel | None, slack | None).  Sets
        self.res = {"x", "f", "status", "iterations", "lam_g", "lam_x"}; a step that did not converge does not
        raise.  lam_g (m x 1): the constraint multipliers (multipliers_batch; NaN when not solved, None for skills
        with more than 32 rows); lam_x (n x 1): zeros (no simple bounds)."""
        spec = self.skill_spec
        q, x, y = one_instance(self, robot_var, virtual_var, input_var)
        nrob, nvirt, nslack = spec.n_robot_var, spec.n_virtual_var, spec.n_slack_var
        has_virtual = spec._has_virtual
        warm = None
        if warmstart_robot_vel_var is not None or warmstart_virtual_vel_var is not None or \
                warmstart_slack_var is not None:
            parts = [as_vector(warmstart_robot_vel_var, nrob, "warmstart_robot_vel_var")
                     if warmstart_robot_vel_var is not None else np.zeros(nrob)]
            if self._nxv:
                parts.append(as_vector(warmstart_virtual_vel_var, self._nxv, "warmstart_virtual_vel_var")
                             if warmstart_virtual_vel_var is not None else np.zeros(self._nxv))
            if nslack:
                parts.append(as_vector(warmstart_slack_var, nslack, "warmstart_slack_var")
                             if warmstart_slack_var is not None else np.zeros(nslack))
            warm = np.ascontiguousarray(np.concatenate(parts))
        sol = np.empty(self._qn)
        status, iters = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
        active = np.zeros(2, dtype=np.uint32)
        lam = np.empty(self._qm) if self.kernel_meta.get("duals") else None
        vp = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)  # noqa: E731
        skill = self._skill()
        runtime.check(skill._lib.clik_nlp_solve_one_lam(
            skill.handle, ctypes.c_double(float(time_var)), vp(q), vp(x), vp(y), vp(warm), vp(sol), vp(status),
            vp(iters), vp(active), self._max_iter(None), vp(lam)))
        self.res = {"x": dm_column(sol), "f": self._objective(time_var, q, x, y, sol),
                    "status": int(status[0]), "iterations": int(iters[0]),
                    "lam_g": None if lam is None else dm_column(lam), "lam_x": cs.DM.zeros(self._qn, 1)}
        res_robot_vel = dm_column(sol[:nrob])
        res_virtual_vel = dm_column(sol[nrob:nrob + nvirt]) if (nvirt > 0 and has_virtual) else None
        off = nrob + self._nxv
        res_slack = dm_column(sol[off:off + nslack]) if nslack > 0 else None
        return res_robot_vel, res_virtual_vel, res_slack

    def _objective(self, t, q, x, y, sol):
        """F at the returned point, evaluated on the host (the `f` entry of cs.nlpsol's result)."""
        prog = self._prog
        vals = {prog.syms.t[0].id: float(t)}
        for arr, nodes in ((q, prog.syms.q), (x, prog.syms.x), (y, prog.syms.y)):
            if arr is not None:
                vals.update({n.id: float(arr[i]) for i, n in enumerate(nodes)})
        vals.update({n.id: float(sol[j]) for j, n in enumerate(prog.dec)})
        return float(dag.evaluate([prog.F], vals)[0])
