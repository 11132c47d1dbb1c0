"""PseudoInverseController — set-based singularity-robust multiple-task-priority controller,
evaluated on the GPU for one or N instances.

Drop-in for reference casclik/controllers/pseudo_inverse.py: same constructor, option keys and
defaults (:42-66), `setup_problem_functions` / `setup_solver` / `setup_initial_problem_solver` /
`solve_initial_problem` / `solve` signatures and return conventions (:453-556), and the same
public attributes (`current_mode`, `modes`, `activation_map`, `n_modes`, `n_set_constraints`,
`state_var`, `n_state_var`).  Instead of one JIT-compiled CasADi function per mode, setup emits
one CUDA translation unit for the skill (casclik_b200/codegen) and loads it through the C ABI
(include/clik.h); `solve` runs a batch of one, `solve_batch` runs N.

Options are read when `setup_*` runs, not at construction, because the reference stores the dict
by reference and the notebooks mutate it in between (SURVEY.md Appendix A19).
"""
import os

import numpy as np

from .. import build, runtime
from .. import sym as cs
from ..codegen import PinvProgram, emit_skill
from ..constraints import SetConstraint
from ._modes import activation_map
from .base_controller import BaseController, Batch, dm_column, one_instance, run_step, set_overlap


class PseudoInverseController(BaseController):
    """Pseudo inverse controller.

    Args:
        skill_spec (SkillSpecification): skill specification
        options (dict): feedforward (True), multidim_sets (False),
            converge_final_set_to_max (False), pinv_method ("damped" | "standard"),
            damping_factor (1e-7), function_opts (kept for compatibility; the CUDA build ignores it)
    """
    controller_type = "PseudoInverseController"
    options_info = """feedforward, multidim_sets, converge_final_set_to_max, pinv_method,
    damping_factor, function_opts"""

    def __init__(self, skill_spec, options=None):
        self.current_mode = None
        self._compiled = {}
        self.skill_spec = skill_spec
        self.options = options

    # ---- options / skill -----------------------------------------------------------------------
    @property
    def options(self):
        return self._options

    @options.setter
    def options(self, opt):
        if opt is None:
            opt = {}
        opt.setdefault("feedforward", True)
        opt.setdefault("multidim_sets", False)
        opt.setdefault("converge_final_set_to_max", False)
        opt.setdefault("pinv_method", "damped")   # "standard" | "damped"
        opt.setdefault("damping_factor", 1e-7)
        fopts = opt.setdefault("function_opts", {})
        fopts.setdefault("jit", True)
        fopts.setdefault("print_time", False)
        fopts.setdefault("jit_options", {"flags": "-O2"})
        self._options = opt

    @property
    def skill_spec(self):
        return self._skill_spec

    @skill_spec.setter
    def skill_spec(self, spec):
        counts = spec.count_constraints()
        self.n_set_constraints = counts["set"]
        self.n_modes = 2 ** counts["set"]
        state = [spec.robot_var]
        cntrl = [spec.robot_vel_var]
        n_state = spec.n_robot_var
        if spec.virtual_var is not None:
            state.append(spec.virtual_var)
            cntrl.append(spec.virtual_vel_var)
            n_state += spec.n_virtual_var
        self.state_var = cs.vertcat(*state)
        self.cntrl_var = cntrl
        self.n_state_var = n_state
        self._skill_spec = spec
        self._compiled = {}
        self.create_activation_map()

    def create_activation_map(self):
        self.activation_map = activation_map(self.n_set_constraints)

    # ---- setup ------------------------------------------------------------------------------------
    def get_problem_expressions(self):
        """Mode table.  The reference stores a CasADi expression per mode here; this engine keeps
        the per-mode algebra inside one kernel, so a mode entry only lists which sets it
        activates."""
        sets = [c for c in self.skill_spec.constraints if isinstance(c, SetConstraint)]
        rows = self.activation_map or [[]]
        self.modes = [{"activation": list(bits),
                       "active_set_names": [c.label for c, b in zip(sets, bits) if b],
                       "inactive_set_names": [c.label for c, b in zip(sets, bits) if not b]}
                      for bits in rows]
        return self.modes

    def setup_problem_functions(self, load=True):
        """Lower the skill, emit CUDA, compile for sm_100a (cached) and load the cubin.
        `load=False` stops after compilation (usable without a GPU)."""
        self.get_problem_expressions()
        prog = PinvProgram(self.skill_spec, self.options)
        source, meta = emit_skill(pinv=prog, label=self.skill_spec.label)
        cubin, path = build.compile_cubin(source, tag="pinv_" + self.skill_spec.label)
        regs = build.kernel_registers(path, "clik_pinv_kernel")
        if regs is not None and "CLIK_MINBLOCKS" not in os.environ:
            # Occupancy step by register cap (`__launch_bounds__(128, k)`).  These kernels are bound by the
            # fp64 pipe and by dependency latency, so one more resident CTA per SM pays as long as the cap
            # does not push live values into local memory.  Measured (profiles/r2_ab*.txt, 2^20 instances):
            #   UR5 tracking   66 regs, 7 CTAs/SM 4.07e10 steps/s -> cap 8 (63 regs, no spill)      4.31e10
            #   Moe-2016       92 regs, 5 CTAs    2.66e10         -> cap 7 (72 regs, +56 B local)    2.83e10
            #   iiwa pose     166 regs, 3 CTAs    1.20e10         -> cap 4 (128 regs, 200 B local)   1.33e10,
            #                                                        cap 5 (96 regs, 360 B)          1.08e10
            #   iiwa stress   255 regs, 2 CTAs    4.6e9           -> cap 3 (168 regs, 832 B)         3.9e9
            # Rule: take the highest occupancy step above the natural one whose local-memory frame stays
            # within 64 B of the natural frame (small kernels) / within 400 B (kernels above 128 registers).
            natural = regs
            natural_local = build.kernel_stack_bytes(path, "clik_pinv_kernel") or 0
            if natural > 128:
                levels, limit = ((4, 128), (3, 168)), 400
            else:
                levels, limit = ((8, 64), (7, 72), (6, 80), (5, 96)), natural_local + 64
            for min_blocks, cap in levels:
                if natural <= cap:
                    continue
                src_c, meta_c = emit_skill(pinv=prog, label=self.skill_spec.label, min_blocks=min_blocks)
                cubin_c, path_c = build.compile_cubin(src_c, tag="pinv_" + self.skill_spec.label)
                local_c = build.kernel_stack_bytes(path_c, "clik_pinv_kernel")
                if local_c is not None and local_c <= limit:
                    source, meta, cubin, path = src_c, meta_c, cubin_c, path_c
                    meta["register_cap"] = ("launch_bounds(128, %d): natural allocation was %d registers / %d B "
                                            "local, %d B local under the cap" % (min_blocks, natural, natural_local, local_c))
                    break
            else:
                meta["register_cap"] = "none: natural allocation %d registers" % natural
        self.kernel_source, self.kernel_meta, self.cubin_path = source, meta, path
        self._nx, self._ny = prog.n_virt, prog.n_in
        self._cubin = cubin
        self._compiled = {}
        if load:
            self._skill()

    def setup_initial_problem_solver(self):
        """Nothing to set up (same as the reference, pseudo_inverse.py:485-488)."""
        pass

    def solve_initial_problem(self, time_var0, robot_var0, virtual_var0=None,
                              robot_vel_var0=None, input_var0=None):
        """Zeros, like the reference (pseudo_inverse.py:490-504)."""
        spec = self.skill_spec
        res_virt = cs.DM.zeros(spec.virtual_var.size()) if virtual_var0 is not None else None
        res_slack = cs.DM.zeros(spec.slack_var.size()) if spec.slack_var is not None else None
        return res_virt, res_slack

    def setup_solver(self):
        self.setup_problem_functions()

    def set_input_staging(self, on):
        """Device-resident batches through the TMA-staged persistent kernel (inputs brought into shared memory
        by bulk async copies two tiles ahead of the arithmetic; include/clik.h clik_skill_set_staging).  Same
        bits; faster for HBM-leaning skills when independent batches alternate over two CUDA streams, slightly
        slower on a single stream.  Raises if the skill was compiled without the staged kernel
        (`kernel_meta["pinv_staged_kernel"]`)."""
        if on and not self.kernel_meta.get("pinv_staged_kernel"):
            raise runtime.ClikError("this skill has no staged kernel (two-launch step or too many rows)")
        self._staging = bool(on)
        for sk in self._compiled.values():
            sk.set_staging(self._staging)

    set_overlap = set_overlap

    # ---- step --------------------------------------------------------------------------------------
    def solve_batch(self, time_var, robot_var, virtual_var=None, input_var=None, out=None, devices=None):
        """Controller step for N instances.

        devices (host arrays only): None = one GPU; "all", a count or a list of CUDA ordinals = the
        batch is cut into contiguous shards, one per device, each solved in place on its device
        (no collective, no repacking), results gathered in the returned host arrays — the sharded
        solve of BASELINE.json configs[4].  Bit-identical to the single-device call.

        robot_var (n_robot, N), virtual_var (n_virtual, N), input_var (n_input, N): float64,
        coordinate-major; torch CUDA tensors (zero-copy, asynchronous on the current stream) or
        NumPy arrays (pipelined host path).  time_var: float or (N,).
        Returns (robot_vel (n_robot, N), virtual_vel (n_virtual, N) | None, mode (N,) int32) with
        mode = index into `activation_map` (0 when the skill has no sets), -1 = no admissible
        mode (velocities are zero)."""
        spec = self.skill_spec
        nq, nx, ny = spec.n_robot_var, self._nx, self._ny
        b = Batch(nq, nx, ny, time_var, robot_var, virtual_var, input_var if ny else None)
        if out is None:
            qdot = b.empty(nq)
            xdot = b.empty(nx) if nx else None
            mode = b.empty(0, "i32")
        else:
            qdot, xdot, mode = out
            if qdot is None or (nx and xdot is None):
                raise runtime.ClikError("out=(robot_vel, virtual_vel, mode): the velocity buffers are required")
        qdp, xdp = b.out_ptr(qdot, nq, "f64", "out[0] (robot_vel)"), \
            (b.out_ptr(xdot, nx, "f64", "out[1] (virtual_vel)") if nx else None)
        mdp = b.out_ptr(mode, 0, "i32", "out[2] (mode)")
        run_step(self._skill, "pinv", b, devices, qdp, xdp, mdp)
        return qdot, xdot, mode

    def rollout_batch(self, time_var0, robot_var, steps, dt, virtual_var=None, input_var=None,
                      max_speed=None, max_virtual_speed=None):
        """Closed-loop simulation on the device: `steps` times
        v = solve(t0 + k*dt, q, x, y); v = clip(v, +-max_speed); q += v_rob*dt; x += v_virt*dt
        (the loop of the reference notebooks around solve()).  robot_var / virtual_var are torch
        CUDA tensors (n, N) and are UPDATED IN PLACE.  Returns a dict with the last command
        (`robot_vel`, `virtual_vel`), its `mode`, and `n_failed` (steps with no admissible mode)."""
        import ctypes
        spec = self.skill_spec
        nq, nx, ny = spec.n_robot_var, self._nx, self._ny
        b = Batch(nq, nx, ny, time_var0, robot_var, virtual_var, input_var if ny else None)
        if not b.on_device:
            raise ValueError("rollout_batch needs CUDA tensors (state is updated in place on the device)")
        skill = self._skill(b.device_index)
        if nx and virtual_var is None:
            raise ValueError("the skill has a virtual_var: pass its initial value")
        qdot, xdot = b.empty(nq), (b.empty(nx) if nx else None)
        mode, failed = b.empty(0, "i32"), b.empty(0, "i32")
        inf = float("inf")
        runtime.check(runtime.load_library().clik_pinv_rollout(
            skill.handle, b.N, int(steps), ctypes.c_double(float(dt)), b.tp, b.t_stride, b.qp, b.xp, b.yp,
            ctypes.c_double(inf if max_speed is None else float(max_speed)),
            ctypes.c_double(inf if max_virtual_speed is None else float(max_virtual_speed)),
            b.ptr(qdot), b.ptr(xdot), b.ptr(mode), b.ptr(failed), b.stream()))
        return {"robot_vel": qdot, "virtual_vel": xdot, "mode": mode, "n_failed": failed}

    def solve(self, time_var, robot_var, virtual_var=None, input_var=None,
              warmstart_robot_vel_var=None, warmstart_virtual_vel_var=None,
              warmstart_slack_var=None):
        """One controller step -> (cntrl_rob, cntrl_virt | None, None); sets `current_mode`."""
        spec = self.skill_spec
        q, x, y = one_instance(self, robot_var, virtual_var, input_var)
        nq = spec.n_robot_var
        use_virt = virtual_var is not None and spec._has_virtual
        # one instance: straight to the single-instance ABI entry (a page-locked mapped slot inside the
        # library; no batch plumbing, no allocation) — the call a notebook makes in its control loop
        one = getattr(self, "_one", None)
        if one is None or one["nq"] != nq:
            import ctypes
            buf = {"nq": nq, "qdot": np.empty(nq), "xdot": np.empty(max(self._nx, 1)),
                   "mode": np.zeros(1, dtype=np.int32)}
            buf["qdot_p"] = ctypes.c_void_p(buf["qdot"].ctypes.data)
            buf["xdot_p"] = ctypes.c_void_p(buf["xdot"].ctypes.data) if self._nx else None
            buf["mode_p"] = ctypes.c_void_p(buf["mode"].ctypes.data)
            one = self._one = buf
        import ctypes
        skill = self._skill()
        runtime.check(skill._lib.clik_pinv_solve_one(
            skill.handle, ctypes.c_double(float(time_var)), ctypes.c_void_p(q.ctypes.data),
            ctypes.c_void_p(x.ctypes.data) if x is not None else None,
            ctypes.c_void_p(y.ctypes.data) if y is not None else None,
            one["qdot_p"], one["xdot_p"], one["mode_p"]))
        self.current_mode = int(one["mode"][0])
        cntrl_virt = dm_column(one["xdot"][:self._nx]) if use_virt else None
        return dm_column(one["qdot"]), cntrl_virt, None
