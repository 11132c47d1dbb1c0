"""ReactiveQPController — eTaSL-style reactive QP controller, evaluated on the GPU for one or N
instances.

Drop-in for reference casclik/controllers/reactive_qp.py: same constructor and weight handling
(:46-133; None / list / ndarray weights, list -> column), option keys (:141-173),
`weight_shifter` class attribute (:44), `setup_problem_functions`, `setup_solver`,
`setup_initial_problem_solver`, `solve_initial_problem`, `solve` (:248-528) and the 3-tuple
result `(robot_vel, virtual_vel | None, slack | None)`.

Problem per instance (x = [robot vel; virtual vel; slack]):
    min 1/2 x' H x,  H = diag([mu*w_rob ; mu*w_virt ; mu + w_slack])          (:175-189)
    s.t. lb <= A x <= ub,  rows per constraint [de/dq | de/dx | -I on own slack]  (:191-246)
Instead of four JIT-compiled CasADi functions + qpOASES, setup emits one fused CUDA kernel that
evaluates H, A, lb, ub and solves the QP per thread (csrc/clik_qp.cuh).  Infeasible problems do
not raise out of `solve_batch`; they are reported per instance in `status` (the single-instance
`solve` raises RuntimeError like the reference's conic call does).
"""
import os

import numpy as np

from .. import build, runtime
from .. import sym as cs
from ..codegen import QpProgram, emit_skill
from .base_controller import (BaseController, Batch, as_vector, dm_column, multipliers_batch, one_instance, run_step,
                              jacobian_batch, jvp_batch, rollout_batch_differentiable, rollout_jacobian, rollout_jvp,
                              rollout_vjp, set_overlap, solve_batch_differentiable, vjp_batch)
from .qp_solver import ConicSolver


def _weights(weights, n, what, of):
    """None -> ones; list / ndarray -> column (length checked); symbolic columns are accepted too
    (the reference's own check for CasADi-typed weights can never pass, Appendix A17)."""
    if weights is None:
        return cs.vertcat([1.0] * n) if n else cs.DM.zeros(0, 1)
    if isinstance(weights, cs.GenericMatrixCommon):
        if weights.size2() != 1:
            raise ValueError(what + " must be a vector.")
        if weights.size1() != n:
            raise ValueError(what + " and " + of + " dimensions do not match.")
        return weights
    if isinstance(weights, (list, np.ndarray)):
        if len(weights) != n:
            raise ValueError(what + " and " + of + " dimensions do not match")
        return cs.vertcat(list(weights))
    raise TypeError(what + " must be None, a list, a numpy array or a column matrix")


class ReactiveQPController(BaseController):
    """Reactive QP controller.

    Args:
        skill_spec (SkillSpecification): skill specification
        robot_var_weights, virtual_var_weights, slack_var_weights: QP weights (floats or
            expressions of time/robot/virtual/input variables); default 1.0 / cnstr.slack_weight
        options (dict): solver_name, solver_opts, initial_solver_opts, function_opts (accepted
            for compatibility), plus "max_iter" (cap of active-set iterations, default
            10*(nx+m))
    """
    controller_type = "ReactiveQPController"
    options_info = """solver_name, solver_opts, initial_solver_opts, function_opts, max_iter"""
    weight_shifter = 0.001  # eTaSL's mu

    def __init__(self, skill_spec, robot_var_weights=None, virtual_var_weights=None,
                 slack_var_weights=None, options=None):
        self.skill_spec = skill_spec
        self.robot_var_weights = robot_var_weights
        self.virtual_var_weights = virtual_var_weights
        self.slack_var_weights = slack_var_weights
        self.options = options
        self._compiled = {}
        self._cubin = None
        self._vjp = None
        self._jvp = None
        self._rollout_jvp = None
        self._rollout_vjp = None
        self._has_initial = False
        self.res = None

    # ---- weights ----------------------------------------------------------------------------------
    @property
    def robot_var_weights(self):
        return self._robot_var_weights

    @robot_var_weights.setter
    def robot_var_weights(self, weights):
        self._robot_var_weights = _weights(weights, self.skill_spec.n_robot_var,
                                           "robot_var_weights", "robot_var")

    @property
    def virtual_var_weights(self):
        return self._virtual_var_weights

    @virtual_var_weights.setter
    def virtual_var_weights(self, weights):
        self._virtual_var_weights = _weights(weights, self.skill_spec.n_virtual_var,
                                             "virtual_var_weights", "virtual_var")

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

    # ---- options ----------------------------------------------------------------------------------
    @property
    def options(self):
        return self._options

    @options.setter
    def options(self, opt):
        if opt is None or not isinstance(opt, dict):
            opt = {}
        opt.setdefault("solver_name", "qpoases")
        sopts = opt.setdefault("solver_opts", {})
        sopts.setdefault("print_time", False)
        if opt["solver_name"] == "qpoases":
            sopts.setdefault("printLevel", "none")
        elif opt["solver_name"] == "ooqp":
            sopts.setdefault("print_level", 0)
        sopts.setdefault("jit", True)
        sopts.setdefault("jit_options", {"flags": "-O2"})
        opt.setdefault("initial_solver_opts", sopts)
        fopts = opt.setdefault("function_opts", {})
        fopts.setdefault("jit", True)
        fopts.setdefault("print_time", False)
        fopts.setdefault("jit_options", {"flags": "-O2"})
        self._options = opt

    # ---- expressions (kept for API parity / inspection) -------------------------------------------
    def _program(self):
        return QpProgram(self.skill_spec, self.robot_var_weights, self.virtual_var_weights,
                         self.slack_var_weights, self.weight_shifter)

    def get_cost_expr(self):
        prog = self._program()
        return cs.diag(cs.MX(cs.vertcat(*prog.h)))

    def get_constraints_expr(self):
        prog = self._program()
        A = cs.MX(cs.vertcat(*[cs.horzcat(*row) for row in prog.A]))
        return A, cs.MX(cs.vertcat(*prog.lb)), cs.MX(cs.vertcat(*prog.ub))

    def _input_list(self):
        spec = self.skill_spec
        ins, names = [spec.time_var, spec.robot_var], ["time_var", "robot_var"]
        if spec.virtual_var is not None and spec._has_virtual:
            ins.append(spec.virtual_var)
            names.append("virtual_var")
        if spec.input_var is not None and spec._has_input:
            ins.append(spec.input_var)
            names.append("input_var")
        return ins, names

    # ---- setup ------------------------------------------------------------------------------------
    def setup_problem_functions(self, load=True):
        """Emit + compile + load the fused QP kernel; also exposes H_func / A_func / Blb_func /
        Bub_func (host-evaluated `cs.Function`s, for inspection as in the reference :283-298)."""
        prog = self._program()
        bad = [k for k, n in enumerate(prog.h) if n.is_const and not (n.val > 0.0 and np.isfinite(n.val))]
        if bad:
            # (the reference hands a semidefinite H to qpOASES, which copes when the constraints pin x
            # down; the GPU solver works in sqrt(H)-scaled variables and needs a strictly convex cost)
            raise ValueError("QP cost weights must be positive and finite: entries %s of the diagonal of H "
                             "(mu*robot weights; mu*virtual weights; mu + slack weights) are not" % bad)
        source, meta = emit_skill(qp=prog, label=self.skill_spec.label)
        cubin, path = build.compile_cubin(source, tag="qp_" + self.skill_spec.label)
        regs = build.kernel_registers(path, "clik_qp_fast_kernel") if meta.get("qp_split") else None
        if regs is not None and regs > 168 and "CLIK_QP_FAST_MINBLOCKS" not in os.environ:
            # The fast kernel holds two phases: the prediction passes every instance runs, and the rarely
            # executed continuation for slow instances (more passes + the one-row rule), whose register
            # needs must not cost the first phase an occupancy step: cap at 3 CTAs/SM (168 registers) when
            # the spills that causes stay small (UR5 9x15: 208 -> 168 registers; same rule as the pinv kernels).
            src3, meta3 = emit_skill(qp=prog, label=self.skill_spec.label, qp_fast_min_blocks=3)
            cubin3, path3 = build.compile_cubin(src3, tag="qp_" + self.skill_spec.label)
            local3 = build.kernel_stack_bytes(path3, "clik_qp_fast_kernel")
            natural_local = build.kernel_stack_bytes(path, "clik_qp_fast_kernel") or 0
            if local3 is not None and local3 <= natural_local + 400:
                source, meta, cubin, path = src3, meta3, cubin3, path3
                meta["register_cap"] = ("fast kernel launch_bounds(128, 3): natural allocation was %d registers, "
                                        "%d B local under the cap" % (regs, local3))
                # one more step (4 CTAs/SM, 128 registers) when even that leaves a small frame: UR5 9x15 232 B,
                # +2-5 %; Moe-2016 496 B, -4 % (profiles/r2_ab14.txt)
                src4, meta4 = emit_skill(qp=prog, label=self.skill_spec.label, qp_fast_min_blocks=4)
                cubin4, path4 = build.compile_cubin(src4, tag="qp_" + self.skill_spec.label)
                local4 = build.kernel_stack_bytes(path4, "clik_qp_fast_kernel")
                if local4 is not None and local4 <= 256:
                    source, meta, cubin, path = src4, meta4, cubin4, path4
                    meta["register_cap"] = ("fast kernel launch_bounds(128, 4): natural allocation was %d registers, "
                                            "%d B local under the cap" % (regs, local4))
        self.kernel_source, self.kernel_meta, self.cubin_path = source, meta, path
        self._nxv, self._ny, self._qn, self._qm = prog.n_virt, prog.n_in, prog.nx, prog.m
        self.row_labels = prog.labels
        # constant cost weights (the usual case): keep the numbers, so `solve` does not have to
        # evaluate H_func through the expression interpreter at every call
        self._h_const = (np.array([n.val for n in prog.h]) if all(n.is_const for n in prog.h) else None)
        self._cubin = cubin
        self._compiled = {}
        self._vjp = None
        self._jvp = None
        self._rollout_jvp = None
        self._rollout_vjp = None
        ins, names = self._input_list()
        H = cs.diag(cs.MX(cs.vertcat(*prog.h)))
        A = cs.MX(cs.vertcat(*[cs.horzcat(*row) for row in prog.A]))
        self.H_func = cs.Function("H_func", ins, [H], names, ["H"])
        self.A_func = cs.Function("A_func", ins, [A], names, ["A"])
        self.Blb_func = cs.Function("Blb_expr", ins, [cs.MX(cs.vertcat(*prog.lb))], names, ["Blb"])
        self.Bub_func = cs.Function("Bub_expr", ins, [cs.MX(cs.vertcat(*prog.ub))], names, ["Bub"])
        if load:
            self._skill()

    def setup_solver(self):
        """`self.solver`: the conic-call object (reference :248-260).  Either order of
        setup_solver / setup_problem_functions works (Appendix A9)."""
        self.solver = ConicSolver("solver", self.options["solver_name"], {},
                                  self.options["solver_opts"])
        if self._cubin is None:
            self.setup_problem_functions()

    set_overlap = set_overlap

    # ---- initial problem (virtual + slack with robot velocity fixed), reference :300-459 ---------------
    def setup_initial_problem_solver(self):
        from .initial_problem import InitialProblem
        self._initial = InitialProblem(self)
        self._has_initial = self._initial.active
        return None

    def solve_initial_problem(self, time_var0, robot_var0, virtual_var0=None, robot_vel_var0=None,
                              input_var0=None):
        if not self._has_initial:
            return None, None
        return self._initial.solve(time_var0, robot_var0, virtual_var0, robot_vel_var0, input_var0)

    def solve_initial_problem_batch(self, time_var0, robot_var0, virtual_var0=None, robot_vel_var0=None,
                                    input_var0=None, max_iter=None):
        """solve_initial_problem (reference reactive_qp.py:426-459) for N instances at once: the initial
        virtual velocities and slack of every scenario of a batch, e.g. to seed the warm start of its first
        steps.  Arrays are coordinate-major like solve_batch's; robot_vel_var0 / virtual_var0 default to
        zeros.  Returns (virtual_vel (n_virtual, N) | None, slack (n_slack, N) | None, status (N,))."""
        if not getattr(self, "_has_initial", None):
            if getattr(self, "_initial", None) is None:
                self.setup_initial_problem_solver()
            if not self._has_initial:
                return None, None, None
        return self._initial.solve_batch(time_var0, robot_var0, virtual_var0, robot_vel_var0, input_var0,
                                         int(max_iter or self.options.get("max_iter", 0) or 0))

    # ---- step --------------------------------------------------------------------------------------
    def solve_batch(self, time_var, robot_var, virtual_var=None, input_var=None, warmstart=None,
                    out=None, max_iter=None, warm_active=None, devices=None):
        """QP controller step for N instances (same layout rules as
        PseudoInverseController.solve_batch).  warmstart: optional (nx, N) primal guess;
        warm_active: optional (2, N) int32 working-set guess in the format of the returned `active`
        (e.g. the previous step's).  Either only shortens the active-set iteration.
        devices: as in PseudoInverseController.solve_batch (host arrays sharded over several GPUs).
        Returns (sol (nx, N), status (N,) int32, active (2, N) int32 bit masks [upper; lower]);
        rows of `sol` are [robot vel; virtual vel; slack]."""
        spec = self.skill_spec
        b = Batch(spec.n_robot_var, self._nxv, self._ny, time_var, robot_var, virtual_var,
                  input_var if self._ny else None)
        if out is None:
            sol = b.empty(self._qn)
            status = b.empty(0, "i32")
            active = b.empty(2, "i32")
        else:
            sol, status, active = out
            if sol is None:
                raise runtime.ClikError("out=(sol, status, active): the solution buffer is required")
        solp = b.out_ptr(sol, self._qn, "f64", "out[0] (sol)")
        stp = b.out_ptr(status, 0, "i32", "out[1] (status)")
        acp = b.out_ptr(active, 2, "i32", "out[2] (active)")
        x0p = None
        if warmstart is not None:
            if b.on_device:
                x0p = runtime.dev_ptr(warmstart, "f64", self._qn * b.N, "warmstart")
            else:
                x0p, warmstart = runtime.host_ptr(warmstart, np.float64, self._qn * b.N, "warmstart")
        a0p = None
        if warm_active is not None:
            if b.on_device:
                a0p = runtime.dev_ptr(warm_active, "u32", 2 * b.N, "warm_active")
            else:
                a0p, warm_active = runtime.host_ptr(warm_active, np.int32, 2 * b.N, "warm_active")
        mi = int(max_iter if max_iter is not None else self.options.get("max_iter", 0) or 0)
        run_step(self._skill, "qp", b, devices, x0p, a0p, solp, stp, acp, mi)
        return sol, status, active

    def multipliers_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, out=None):
        """Constraint multipliers (the reference's lam_a) of a solve_batch result: the step's inputs and its
        (sol, status, active), same layout rules as solve_batch (torch CUDA tensors on their device and the
        current stream, NumPy arrays through the host entry point; out= a (m, N) float64 buffer).
        Returns lam (m, N) float64: > 0 at an upper bound, < 0 at a lower bound, 0 off the working set; NaN for
        an instance that is not solved or whose working set is rank-deficient (include/clik.h clik_qp_duals).
        Skills with more than 32 constraint rows raise ValueError."""
        return multipliers_batch(self, "qp", time_var, robot_var, virtual_var, input_var, sol, status, active, out)

    def _vjp_source(self):
        """Source of the VJP image: the default image's emission (same fast-kernel register cap) plus the VJP kernel."""
        return emit_skill(qp=self._program(), label=self.skill_spec.label, vjp=True,
                          qp_fast_min_blocks=self.kernel_meta.get("qp_fast_min_blocks"))

    def vjp_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, sol_bar, out=None):
        """Reverse-mode derivative (vector-Jacobian product) of a solve_batch result: the step's inputs and its
        (sol, status, active) as torch CUDA tensors, and the cotangent sol_bar (nx, N) float64 of sol.  Runs on the
        current stream.  Returns (t_bar (N,), q_bar (n_robot, N), x_bar (n_virtual, N) | None, y_bar (n_input, N) |
        None): (d sol / d theta)' sol_bar for the face problem of the returned working set, the one-sided derivative
        that keeps the working set where a held row has a zero multiplier (DESIGN.md §4.6).  t_bar is per instance
        also for a shared t.  An all-zero cotangent column gives exactly 0; otherwise an unsolved instance or a
        rank-deficient working set gives NaN (include/clik.h clik_qp_vjp).  out= (t_bar, q_bar, x_bar, y_bar)
        buffers of those shapes.  The VJP image is compiled and loaded on the first call (one per device).
        NumPy inputs and skills with more than 32 constraint rows raise ValueError."""
        return vjp_batch(self, "qp", time_var, robot_var, virtual_var, input_var, sol, status, active, sol_bar, out)

    def _jvp_source(self):
        """Source of the JVP image: the default image's emission (same fast-kernel register cap) plus the JVP and
        Jacobian kernels."""
        return emit_skill(qp=self._program(), label=self.skill_spec.label, jvp=True,
                          qp_fast_min_blocks=self.kernel_meta.get("qp_fast_min_blocks"))

    def jvp_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, t_dot=None, q_dot=None,
                  x_dot=None, y_dot=None, out=None):
        """Forward-mode derivative (Jacobian-vector product) of a solve_batch result: the step's inputs and its
        (sol, status, active) as torch CUDA tensors, and the tangent (t_dot (N,) or one entry for every instance,
        q_dot (n_robot, N), x_dot (n_virtual, N), y_dot (n_input, N); None is a zero tangent), float64.  Runs on the
        current stream and returns sol_dot (nx, N) = (d sol / d theta) theta_dot for the face problem of the
        returned working set, the exact adjoint of vjp_batch (DESIGN.md §4.7).  An all-zero tangent gives exactly 0;
        otherwise an unsolved instance or a rank-deficient working set gives NaN (include/clik.h clik_qp_jvp).
        out= a (nx, N) buffer.  The JVP image is compiled and loaded on the first call (one per device).  NumPy
        inputs and skills with more than 32 constraint rows raise ValueError."""
        return jvp_batch(self, "qp", time_var, robot_var, virtual_var, input_var, sol, status, active, t_dot, q_dot,
                         x_dot, y_dot, out)

    def jacobian_batch(self, time_var, robot_var, virtual_var, input_var, sol, status, active, out=None):
        """The full step Jacobian of a solve_batch result: (nx, n_theta, N) float64 on the inputs' device, column c
        the derivative along entry c of theta = (t, q, x, y) (n_theta = 1 + n_robot + n_virtual + n_input), one
        factorisation per instance.  The rules of jvp_batch per column: an unsolved or rejected instance gets NaN
        everywhere (include/clik.h clik_qp_jacobian).  out= a buffer of that shape."""
        return jacobian_batch(self, "qp", time_var, robot_var, virtual_var, input_var, sol, status, active, out)

    def solve_batch_differentiable(self, time_var, robot_var, virtual_var=None, input_var=None, warmstart=None,
                                   max_iter=None):
        """solve_batch on torch CUDA tensors as a torch.autograd.Function: (sol, status, active) with sol attached
        to the graph of time_var, robot_var, virtual_var and input_var (backward: vjp_batch); status and active are
        not differentiable.  A 0-d / one-element tensor t gets the summed t_bar; a Python float t gets none."""
        return solve_batch_differentiable(self, time_var, robot_var, virtual_var, input_var, warmstart, max_iter)

    def rollout_batch(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None,
                      max_speed=None, max_virtual_speed=None, max_iter=None):
        """Closed-loop simulation on the device (see PseudoInverseController.rollout_batch):
        robot_var / virtual_var (torch CUDA, (n, N)) are UPDATED IN PLACE.  Returns a dict with the
        last QP solution `sol` (nx, N) and `n_failed` (steps whose QP was not solved: zero velocity)."""
        import ctypes
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
        mi = int(max_iter if max_iter is not None else self.options.get("max_iter", 0) or 0)
        runtime.check(runtime.load_library().clik_qp_rollout(
            skill.handle, b.N, int(steps), ctypes.c_double(float(dt)), b.tp, b.t_stride, b.qp, b.xp, b.yp,
            ctypes.c_double(inf if max_speed is None else float(max_speed)),
            ctypes.c_double(inf if max_virtual_speed is None else float(max_virtual_speed)),
            b.ptr(sol), b.ptr(failed), mi, b.stream()))
        return {"sol": sol, "n_failed": failed}

    def _rollout_jvp_source(self):
        """Source of the rollout-JVP image: the JVP image plus the tangent and Jacobian rollout kernels."""
        return emit_skill(qp=self._program(), label=self.skill_spec.label, jvp=True, rollout_jvp=True,
                          qp_fast_min_blocks=self.kernel_meta.get("qp_fast_min_blocks"))

    def rollout_jvp(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None, max_speed=None,
                    max_virtual_speed=None, max_iter=None, t_dot=None, q_dot=None, x_dot=None, y_dot=None):
        """rollout_batch (robot_var / virtual_var UPDATED IN PLACE, bit for bit the same states, `sol` and `n_failed`)
        with the tangent of the closed loop carried along in one kernel: the inputs p = (t0, q0, x0, y) move along
        (t_dot (N,) or one entry for every instance, q_dot (n_robot, N), x_dot (n_virtual, N), y_dot (n_input, N);
        None is a zero tangent; none is modified).  Every step takes the jvp_batch tangent of its solution on its
        own working set, keeps the entries the clip max_speed / max_virtual_speed does not hold (|sol_j| < max) and
        integrates them like the state (DESIGN.md §4.8).  Returns {"sol", "n_failed", "q_dot" (n_robot, N), "x_dot"
        (n_virtual, N) | None, "sol_dot" (nx, N)}: the tangents of the final state and of `sol`.  An instance whose
        tangent hits a step with status != 0, a rank-deficient working set gets NaN from that step on; an all-zero
        tangent stays exactly 0.  The image is compiled and loaded on the first call (one per device).  NumPy
        inputs and skills with more than 32 constraint rows raise ValueError."""
        mi = int(max_iter if max_iter is not None else self.options.get("max_iter", 0) or 0)
        return rollout_jvp(self, "qp", time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                           max_virtual_speed, mi, t_dot, q_dot, x_dot, y_dot)

    def rollout_jacobian(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None, max_speed=None,
                         max_virtual_speed=None, max_iter=None):
        """rollout_batch (state UPDATED IN PLACE, the same bits) with the Jacobian of the final state carried along:
        {"sol", "n_failed", "jac"}, jac (n_robot + n_virtual, n_theta, N) = d(q_K, x_K)/d(t0, q0, x0, y), column c
        the rollout_jvp tangent along the unit tangent e_c, computed with one factorisation per step; the rules of
        rollout_jvp per instance (a NaN block)."""
        mi = int(max_iter if max_iter is not None else self.options.get("max_iter", 0) or 0)
        return rollout_jacobian(self, "qp", time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                                max_virtual_speed, mi)

    def _rollout_vjp_source(self):
        """Source of the rollout-VJP image: the VJP image plus the taped rollout and reverse sweep kernels."""
        return emit_skill(qp=self._program(), label=self.skill_spec.label, vjp=True, rollout_vjp=True,
                          qp_fast_min_blocks=self.kernel_meta.get("qp_fast_min_blocks"))

    def rollout_vjp(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None, max_speed=None,
                    max_virtual_speed=None, max_iter=None, q_bar=None, x_bar=None, sol_bar=None):
        """rollout_batch (robot_var / virtual_var UPDATED IN PLACE, bit for bit the same states, `sol` and `n_failed`)
        followed by the reverse sweep of the closed loop: the cotangents q_bar (n_robot, N), x_bar (n_virtual, N) of
        the final state and sol_bar (nx, N) of `sol` (None is zero) are pulled back to p = (t0, q0, x0, y), one
        step VJP per step on the step's own solution and working set, masked where the clip max_speed /
        max_virtual_speed holds (DESIGN.md §4.9).  Returns {"sol", "n_failed", "t_bar" (N,), "q_bar" (n_robot, N),
        "x_bar" (n_virtual, N) | None, "y_bar" (n_input, N) | None}, the exact adjoint of rollout_jvp; t_bar is per
        instance also for a shared t0.  A zero cotangent gives exactly 0; an instance whose nonzero cotangent
        reaches a step with status != 0 or a rank-deficient working set gets NaN everywhere.  The image is compiled
        and loaded on the first call (one per device); the tape between the two launches takes
        steps * N * (8 (n_robot + n_virtual + nx) + 12) bytes of device memory.  NumPy inputs and skills with more
        than 32 constraint rows raise ValueError."""
        mi = int(max_iter if max_iter is not None else self.options.get("max_iter", 0) or 0)
        return rollout_vjp(self, "qp", time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                           max_virtual_speed, mi, q_bar, x_bar, sol_bar)

    def rollout_batch_differentiable(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None,
                                     max_speed=None, max_virtual_speed=None, max_iter=None):
        """rollout_batch as a torch.autograd.Function on torch CUDA tensors: returns new tensors (q_K, x_K | None,
        sol, n_failed) and modifies no input.  backward() runs the reverse sweep of rollout_vjp over the tape the
        forward kept (once differentiable), forward-mode AD the tangent of rollout_jvp; n_failed is not
        differentiable.  A 0-d / one-element tensor t0 gets the summed t_bar; a Python float t0 gets none."""
        mi = int(max_iter if max_iter is not None else self.options.get("max_iter", 0) or 0)
        return rollout_batch_differentiable(self, "qp", time_var0, robot_var, steps, dt, virtual_var, input_var,
                                            max_speed, max_virtual_speed, mi)

    def solve(self, time_var, robot_var, virtual_var=None, input_var=None,
              warmstart_robot_vel_var=None, warmstart_virtual_vel_var=None,
              warmstart_slack_var=None):
        """One controller step -> (robot_vel, virtual_vel | None, slack | None).  Sets self.res = {"x", "status",
        "active_upper", "active_lower", "cost", "lam_a", "lam_x"}: lam_a (m x 1) are the constraint multipliers
        (multipliers_batch; None for skills with more than 32 rows), lam_x (n x 1) zeros (no simple bounds)."""
        spec = self.skill_spec
        q, x, y = (None if a is None else a.reshape(-1, 1)
                   for a in one_instance(self, robot_var, virtual_var, input_var))
        nrob, nvirt, nslack = spec.n_robot_var, spec.n_virtual_var, spec.n_slack_var
        has_virtual = spec._has_virtual
        ws_rob = warmstart_robot_vel_var is not None
        ws_virt = warmstart_virtual_vel_var is not None and has_virtual
        ws_slack = warmstart_slack_var is not None and nslack > 0
        warm = None
        if ws_rob or ws_virt or ws_slack:
            parts = [as_vector(warmstart_robot_vel_var, nrob, "warmstart_robot_vel_var")
                     if ws_rob else np.zeros(nrob)]
            if self._nxv:
                parts.append(as_vector(warmstart_virtual_vel_var, self._nxv, "warmstart_virtual_vel_var")
                             if ws_virt else np.zeros(self._nxv))
            if nslack:
                parts.append(as_vector(warmstart_slack_var, nslack, "warmstart_slack_var")
                             if ws_slack else np.zeros(nslack))
            warm = np.ascontiguousarray(np.concatenate(parts).reshape(-1, 1))
        # one instance: the single-instance ABI entry (page-locked mapped slot inside the library)
        import ctypes
        one = getattr(self, "_one", None)
        if one is None or one["qn"] != self._qn or one["lam"].size != self._qm:
            buf = {"qn": self._qn, "sol": np.empty(self._qn), "status": np.zeros(1, dtype=np.int32),
                   "active": np.zeros(2, dtype=np.uint32), "lam": np.empty(self._qm)}
            for k in ("sol", "status", "active", "lam"):
                buf[k + "_p"] = ctypes.c_void_p(buf[k].ctypes.data)
            one = self._one = buf
        skill = self._skill()
        mi = int(self.options.get("max_iter", 0) or 0)
        duals = bool(self.kernel_meta.get("duals"))
        runtime.check(skill._lib.clik_qp_solve_one_lam(
            skill.handle, ctypes.c_double(float(time_var)), ctypes.c_void_p(q.ctypes.data),
            ctypes.c_void_p(x.ctypes.data) if x is not None else None,
            ctypes.c_void_p(y.ctypes.data) if y is not None else None,
            ctypes.c_void_p(warm.ctypes.data) if warm is not None else None,
            one["sol_p"], one["status_p"], one["active_p"], mi, one["lam_p"] if duals else None))
        sol, status, active = one["sol"].reshape(-1, 1).copy(), one["status"], one["active"].reshape(2, 1)
        if int(status[0]) != runtime.QP_SOLVED:
            raise RuntimeError("QP %s" % {runtime.QP_INFEASIBLE: "is infeasible",
                                          runtime.QP_INVALID: "has non-finite data or a non-finite solution "
                                                              "(NaN input?)"}.get(int(status[0]), "hit the iteration cap"))
        xs = sol[:, 0]
        hdiag = self._h_const if self._h_const is not None else np.asarray(
            self.H_func(*self._numeric_args(time_var, q, x, y)).toarray()).diagonal()
        self.res = {"x": dm_column(xs), "status": int(status[0]),
                    "active_upper": int(active[0, 0]), "active_lower": int(active[1, 0]),
                    "cost": 0.5 * float(np.sum(hdiag * xs * xs)),
                    "lam_a": dm_column(one["lam"]) if duals else None, "lam_x": cs.DM.zeros(self._qn, 1)}
        res_robot_vel = dm_column(xs[:nrob])
        res_virtual_vel = dm_column(xs[nrob:nrob + nvirt]) if (nvirt > 0 and has_virtual) else None
        off = nrob + self._nxv
        res_slack = dm_column(xs[off:off + nslack]) if nslack > 0 else None
        return res_robot_vel, res_virtual_vel, res_slack

    def _numeric_args(self, t, q, x, y):
        spec = self.skill_spec
        args = [float(t), q[:, 0]]
        if spec.virtual_var is not None and spec._has_virtual:
            args.append(x[:, 0])
        if spec.input_var is not None and spec._has_input:
            args.append(y[:, 0])
        return args
