"""Shared pieces of the controllers (the reference's BaseController only defines __repr__,
casclik/controllers/base_controller.py:1-6; the batch plumbing below is new)."""
import ctypes

import numpy as np

from .. import build, runtime
from .. import sym as cs


class BaseController(object):
    controller_type = "BaseController"

    def __repr__(self):
        return "%s<%s>" % (self.controller_type, self.skill_spec.label)

    def _skill(self, device=None):
        """The cubin loaded on `device` (default: runtime.current_device()); one handle per device, created on first
        use with the controller's overlap and staging switches, so a batch always runs on the device its tensors
        live on."""
        if getattr(self, "_cubin", None) is None:
            raise RuntimeError("call setup_problem_functions() / setup_solver() before solve()")
        dev = runtime.current_device() if device is None else int(device)
        if dev not in self._compiled:
            skill = runtime.CompiledSkill(self._cubin, self.kernel_meta, n_slack=self.skill_spec.n_slack_var,
                                          device=dev)
            if getattr(self, "_overlap", None) is not None:
                skill.set_overlap(self._overlap)
            if getattr(self, "_staging", None):
                skill.set_staging(True)
            self._compiled[dev] = skill
        return self._compiled[dev]


def set_overlap(ctrl, level):
    """How successive solve_batch launches on one CUDA stream may overlap (include/clik.h,
    clik_skill_set_overlap): 0 plain stream order, 1 (default) the two launches of one step overlap,
    2 successive steps overlap as well — only for streams of independent batches (step k+1 must not
    read what step k writes; closed loops belong in rollout_batch).

    The set_overlap method of the controllers whose step has two launches (pinv and QP)."""
    level = int(level)
    if level not in (0, 1, 2):
        raise ValueError("overlap level must be 0, 1 or 2")
    ctrl._overlap = level
    for skill in ctrl._compiled.values():
        skill.set_overlap(level)


def run_step(skill, kind, b, devices, *args):
    """Shared dispatch of a controller step (`kind` "pinv", "qp" or "nlp") for the Batch `b`, `skill(device)` the
    controller's handle on a device: CUDA tensors run clik_<kind>_step on their own device and the current stream;
    host arrays run clik_<kind>_step_host_multi with one handle per device of `devices` (resolve_devices; None:
    the default device).  `args`: the kind's arguments after (t, t_stride, q, x, y)."""
    devs = resolve_devices(devices)
    lib = runtime.load_library()
    if b.on_device:
        if devs is not None:
            raise ValueError("devices= applies to host arrays; CUDA tensors run on the device they live on")
        runtime.check(getattr(lib, "clik_%s_step" % kind)(skill(b.device_index).handle, b.N, b.tp, b.t_stride,
                                                          b.qp, b.xp, b.yp, *args, b.stream()))
        return
    skills = [skill(d) for d in (devs or [b.device_index])]
    runtime.check(getattr(lib, "clik_%s_step_host_multi" % kind)(skill_handle_array(skills), len(skills), b.N, b.tp,
                                                                  b.t_stride, b.qp, b.xp, b.yp, *args))


def one_instance(ctrl, robot_var, virtual_var, input_var):
    """Validated (q, x, y) of a single-instance solve() as contiguous float64 vectors; x and y are None when the
    skill has no such rows, and x defaults to zeros when the skill's expressions do not depend on it."""
    if getattr(ctrl, "_cubin", None) is None:
        raise RuntimeError("call setup_problem_functions() / setup_solver() before solve()")
    spec, n_virtual, n_input = ctrl.skill_spec, ctrl.kernel_meta["n_virtual"], ctrl.kernel_meta["n_input"]
    q = np.ascontiguousarray(as_vector(robot_var, spec.n_robot_var, "robot_var"))
    x = None
    if n_virtual:
        if spec._has_virtual and virtual_var is None:
            raise ValueError("the skill depends on virtual_var: a value is required")
        x = np.ascontiguousarray(as_vector(virtual_var, n_virtual, "virtual_var") if virtual_var is not None
                                 else np.zeros(n_virtual))
    y = None
    if n_input:
        if input_var is None:
            raise ValueError("the skill depends on input_var: a value is required")
        y = np.ascontiguousarray(as_vector(input_var, n_input, "input_var"))
    return q, x, y


def resolve_devices(devices):
    """`devices` argument of solve_batch -> list of CUDA ordinals, or None for "the default device".
    "all": every visible GPU; an int n: devices 0..n-1; a sequence: those ordinals."""
    if devices is None:
        return None
    if isinstance(devices, str):
        if devices != "all":
            raise ValueError('devices must be None, "all", a count or a list of CUDA ordinals')
        n = runtime.device_count()
        if n < 1:
            runtime.require_device()
        return list(range(n))
    if isinstance(devices, int):
        if devices < 1 or devices > runtime.device_count():
            raise ValueError("devices=%d but %d CUDA devices are visible" % (devices, runtime.device_count()))
        return list(range(devices))
    devs = [int(d) for d in devices]
    if not devs or len(set(devs)) != len(devs):
        raise ValueError("devices must be a non-empty list of distinct CUDA ordinals")
    return devs


def multipliers_batch(ctrl, kind, time_var, robot_var, virtual_var, input_var, sol, status, active, out):
    """Shared body of ReactiveQPController / ReactiveNLPController.multipliers_batch (`kind` "qp" or "nlp"):
    validates the step's inputs and outputs like solve_batch and calls clik_<kind>_duals[_host]."""
    if ctrl._cubin is None:
        raise RuntimeError("call setup_problem_functions() / setup_solver() before multipliers_batch()")
    if not ctrl.kernel_meta.get("duals"):
        raise ValueError("multipliers need at most 32 constraint rows and at least one (the skill has %d)" % ctrl._qm)
    spec = ctrl.skill_spec
    b = Batch(spec.n_robot_var, ctrl._nxv, ctrl._ny, time_var, robot_var, virtual_var,
              input_var if ctrl._ny else None)
    lam = b.empty(ctrl._qm) if out is None else out
    lamp = b.out_ptr(lam, ctrl._qm, "f64", "out (lam)")
    if sol is None or status is None or active is None:
        raise ValueError("sol, status and active of the step are required")
    if b.on_device:
        if not all(runtime._is_torch(a) for a in (sol, status, active)):
            raise ValueError("sol, status and active must be CUDA tensors when the inputs are CUDA tensors")
        solp = runtime.dev_ptr(sol, "f64", ctrl._qn * b.N, "sol")
        stp = runtime.dev_ptr(status, "i32", b.N, "status")
        acp = runtime.dev_ptr(active, "u32", 2 * b.N, "active")
        if any(a.device != b.device for a in (sol, status, active)):
            raise ValueError("sol, status and active must live on %s like robot_var" % b.device)
    else:
        solp, sol = runtime.host_ptr(sol, np.float64, ctrl._qn * b.N, "sol")
        stp, status = runtime.host_ptr(status, np.int32, b.N, "status")
        acp, active = runtime.host_ptr(active.view(np.int32) if getattr(active, "dtype", None) == np.uint32 else active,
                                       np.int32, 2 * b.N, "active")
    skill = ctrl._skill(b.device_index)
    lib = runtime.load_library()
    if b.on_device:
        runtime.check(getattr(lib, "clik_%s_duals" % kind)(skill.handle, b.N, b.tp, b.t_stride, b.qp, b.xp, b.yp,
                                                            solp, stp, acp, lamp, b.stream()))
    else:
        runtime.check(getattr(lib, "clik_%s_duals_host" % kind)(skill.handle, b.N, b.tp, b.t_stride, b.qp, b.xp,
                                                                 b.yp, solp, stp, acp, lamp))
    return lam


def vjp_image(ctrl, kind, device, which="vjp"):
    """The skill's derivative image `which` loaded on `device`: "vjp" (emit_skill(..., vjp=True): the default image
    plus clik_<kind>_vjp_kernel, source ctrl._vjp_source()), "jvp" (emit_skill(..., jvp=True): the default image
    plus clik_<kind>_jvp_kernel and clik_<kind>_jacobian_kernel, source ctrl._jvp_source()) or "rollout_jvp"
    (emit_skill(..., jvp=True, rollout_jvp=True): the JVP image plus clik_<kind>_rollout_jvp_kernel and
    clik_<kind>_rollout_jacobian_kernel, source ctrl._rollout_jvp_source()) or "rollout_vjp" (emit_skill(...,
    vjp=True, rollout_vjp=True): the VJP image plus clik_<kind>_rollout_tape_kernel and clik_<kind>_rollout_vjp_kernel,
    source ctrl._rollout_vjp_source()).  Built and loaded on
    the first call, cached like every cubin, one handle per device: a controller that never asks for derivatives
    compiles nothing more."""
    attr = "_" + which
    if getattr(ctrl, attr) is None:
        source, meta = getattr(ctrl, "_%s_source" % which)()
        cubin, path = build.compile_cubin(source, tag="%s_%s_%s" % (kind, which, ctrl.skill_spec.label))
        setattr(ctrl, attr, {"source": source, "meta": meta, "cubin": cubin, "path": path, "skills": {}})
    skills = getattr(ctrl, attr)["skills"]
    if device not in skills:
        skills[device] = runtime.CompiledSkill(getattr(ctrl, attr)["cubin"], getattr(ctrl, attr)["meta"],
                                               n_slack=ctrl.skill_spec.n_slack_var, device=device)
    return skills[device]


def vjp_batch(ctrl, kind, time_var, robot_var, virtual_var, input_var, sol, status, active, sol_bar, out):
    """Shared body of ReactiveQPController / ReactiveNLPController.vjp_batch (`kind` "qp" or "nlp"): validates the
    step's inputs, outputs and the cotangent like multipliers_batch and calls clik_<kind>_vjp on the current
    stream.  -> (t_bar (N,), q_bar (n_robot, N), x_bar (n_virtual, N) | None, y_bar (n_input, N) | None)."""
    if ctrl._cubin is None:
        raise RuntimeError("call setup_problem_functions() / setup_solver() before vjp_batch()")
    if not ctrl.kernel_meta.get("duals"):
        raise ValueError("the VJP needs at most 32 constraint rows and at least one (the skill has %d)" % ctrl._qm)
    if not (runtime._is_torch(robot_var) and robot_var.is_cuda):
        raise ValueError("vjp_batch needs torch CUDA tensors (there is no host-array form)")
    spec = ctrl.skill_spec
    b = Batch(spec.n_robot_var, ctrl._nxv, ctrl._ny, time_var, robot_var, virtual_var,
              input_var if ctrl._ny else None)
    if sol is None or status is None or active is None or sol_bar is None:
        raise ValueError("sol, status and active of the step and the cotangent sol_bar are required")
    if not all(runtime._is_torch(a) for a in (sol, status, active, sol_bar)):
        raise ValueError("sol, status, active and sol_bar must be CUDA tensors")
    solp = runtime.dev_ptr(sol, "f64", ctrl._qn * b.N, "sol")
    stp = runtime.dev_ptr(status, "i32", b.N, "status")
    acp = runtime.dev_ptr(active, "u32", 2 * b.N, "active")
    sbp = runtime.dev_ptr(sol_bar, "f64", ctrl._qn * b.N, "sol_bar")
    if any(a.device != b.device for a in (sol, status, active, sol_bar)):
        raise ValueError("sol, status, active and sol_bar must live on %s like robot_var" % b.device)
    rows = (0, spec.n_robot_var, ctrl._nxv, ctrl._ny)
    names = ("t_bar", "q_bar", "x_bar", "y_bar")
    if out is None:
        out = [b.empty(r) if (r or k == 0) else None for k, r in enumerate(rows)]
    else:
        out = list(out)
        if len(out) != 4:
            raise ValueError("out=(t_bar, q_bar, x_bar, y_bar)")
        for k, r in enumerate(rows):
            if (r or k == 0) and out[k] is None:
                raise runtime.ClikError("out[%d] (%s) is required" % (k, names[k]))
            if not (r or k == 0):
                out[k] = None
    ptrs = [b.out_ptr(a, r, "f64", "out[%d] (%s)" % (k, names[k])) if a is not None else None
            for k, (a, r) in enumerate(zip(out, rows))]
    skill = vjp_image(ctrl, kind, b.device_index)
    lib = runtime.load_library()
    runtime.check(getattr(lib, "clik_%s_vjp" % kind)(skill.handle, b.N, b.tp, b.t_stride, b.qp, b.xp, b.yp, solp, stp,
                                                      acp, sbp, *ptrs, b.stream()))
    return tuple(out)


def _step_outputs(ctrl, what, time_var, robot_var, virtual_var, input_var, sol, status, active):
    """Validated Batch and device pointers of a step's inputs and (sol, status, active), as vjp_batch checks them."""
    if ctrl._cubin is None:
        raise RuntimeError("call setup_problem_functions() / setup_solver() before %s()" % what)
    if not ctrl.kernel_meta.get("duals"):
        raise ValueError("the %s needs at most 32 constraint rows and at least one (the skill has %d)"
                         % ("Jacobian" if what == "jacobian_batch" else "JVP", ctrl._qm))
    if not (runtime._is_torch(robot_var) and robot_var.is_cuda):
        raise ValueError("%s needs torch CUDA tensors (there is no host-array form)" % what)
    b = Batch(ctrl.skill_spec.n_robot_var, ctrl._nxv, ctrl._ny, time_var, robot_var, virtual_var,
              input_var if ctrl._ny else None)
    if sol is None or status is None or active is None:
        raise ValueError("sol, status and active of the step are required")
    if not all(runtime._is_torch(a) for a in (sol, status, active)):
        raise ValueError("sol, status and active must be CUDA tensors")
    ptrs = (runtime.dev_ptr(sol, "f64", ctrl._qn * b.N, "sol"), runtime.dev_ptr(status, "i32", b.N, "status"),
            runtime.dev_ptr(active, "u32", 2 * b.N, "active"))
    if any(a.device != b.device for a in (sol, status, active)):
        raise ValueError("sol, status and active must live on %s like robot_var" % b.device)
    return b, ptrs


def _tangent_ptrs(ctrl, b, t_dot, q_dot, x_dot, y_dot):
    """Validated device pointers of a tangent (t_dot, q_dot, x_dot, y_dot) of the Batch `b`: None is a zero tangent,
    t_dot has N entries or one broadcast to every instance."""
    tangents = []
    for a, rows, name in ((t_dot, 0, "t_dot"), (q_dot, ctrl.skill_spec.n_robot_var, "q_dot"),
                          (x_dot, ctrl._nxv, "x_dot"), (y_dot, ctrl._ny, "y_dot")):
        if a is None or (rows == 0 and name != "t_dot"):
            tangents.append(None)
            continue
        if not runtime._is_torch(a) or a.device != b.device:
            raise ValueError("%s must be a CUDA tensor on %s like robot_var" % (name, b.device))
        if name == "t_dot" and a.numel() == 1:
            a = a.reshape(1).expand(b.N).contiguous()
        elif a.dim() != (1 if rows == 0 else 2) or tuple(a.shape) != ((b.N,) if rows == 0 else (rows, b.N)):
            raise ValueError("%s must have shape %s" % (name, (b.N,) if rows == 0 else (rows, b.N)))
        tangents.append(a)
    b.keep = b.keep + tuple(tangents)      # (a broadcast t_dot lives until the launch)
    return [runtime.dev_ptr(a, "f64", (r or 1) * b.N, n) if a is not None else None
            for a, r, n in zip(tangents, (0, ctrl.skill_spec.n_robot_var, ctrl._nxv, ctrl._ny),
                               ("t_dot", "q_dot", "x_dot", "y_dot"))]


def jvp_batch(ctrl, kind, time_var, robot_var, virtual_var, input_var, sol, status, active, t_dot, q_dot, x_dot,
              y_dot, out):
    """Shared body of ReactiveQPController / ReactiveNLPController.jvp_batch (`kind` "qp" or "nlp"): validates the
    step's inputs and outputs like vjp_batch and the tangent (None: zero; t_dot of N entries, or one broadcast to
    every instance), and calls clik_<kind>_jvp on the current stream.  -> sol_dot (nx, N)."""
    b, (solp, stp, acp) = _step_outputs(ctrl, "jvp_batch", time_var, robot_var, virtual_var, input_var, sol, status,
                                        active)
    tptrs = _tangent_ptrs(ctrl, b, t_dot, q_dot, x_dot, y_dot)
    sd = b.empty(ctrl._qn) if out is None else out
    sdp = b.out_ptr(sd, ctrl._qn, "f64", "out (sol_dot)")
    skill = vjp_image(ctrl, kind, b.device_index, "jvp")
    lib = runtime.load_library()
    runtime.check(getattr(lib, "clik_%s_jvp" % kind)(skill.handle, b.N, b.tp, b.t_stride, b.qp, b.xp, b.yp, solp, stp,
                                                      acp, *tptrs, sdp, b.stream()))
    return sd


def n_theta(ctrl):
    """Entries of theta = (t, q, x, y) of one instance: the columns of jacobian_batch."""
    return 1 + ctrl.skill_spec.n_robot_var + ctrl._nxv + ctrl._ny


def jacobian_batch(ctrl, kind, time_var, robot_var, virtual_var, input_var, sol, status, active, out):
    """Shared body of ReactiveQPController / ReactiveNLPController.jacobian_batch: validates like jvp_batch and
    calls clik_<kind>_jacobian on the current stream.  -> jac (nx, n_theta, N), theta ordered (t, q, x, y)."""
    b, (solp, stp, acp) = _step_outputs(ctrl, "jacobian_batch", time_var, robot_var, virtual_var, input_var, sol,
                                        status, active)
    nt = n_theta(ctrl)
    if out is None:
        jac = b.torch.empty((ctrl._qn, nt, b.N), dtype=b.torch.float64, device=b.device)
    else:
        jac = out
        if not runtime._is_torch(jac) or tuple(jac.shape) != (ctrl._qn, nt, b.N):
            raise runtime.ClikError("out (jac) must be a CUDA tensor of shape %s" % ((ctrl._qn, nt, b.N),))
    jp = b.out_ptr(jac, ctrl._qn * nt, "f64", "out (jac)")
    skill = vjp_image(ctrl, kind, b.device_index, "jvp")
    lib = runtime.load_library()
    runtime.check(getattr(lib, "clik_%s_jacobian" % kind)(skill.handle, b.N, b.tp, b.t_stride, b.qp, b.xp, b.yp,
                                                           solp, stp, acp, jp, b.stream()))
    return jac


def _rollout_batch(ctrl, what, time_var0, robot_var, virtual_var, input_var):
    """Validated Batch of a tangent / Jacobian rollout: the checks of rollout_batch and of jvp_batch, all before any
    image is built."""
    if ctrl._cubin is None:
        raise RuntimeError("call setup_problem_functions() / setup_solver() before %s()" % what)
    if not ctrl.kernel_meta.get("duals"):
        raise ValueError("the %s needs at most 32 constraint rows and at least one (the skill has %d)" % (what, ctrl._qm))
    if not (runtime._is_torch(robot_var) and robot_var.is_cuda):
        raise ValueError("%s needs torch CUDA tensors (state is updated in place on the device)" % what)
    if ctrl._nxv and virtual_var is None:
        raise ValueError("the skill has a virtual_var: pass its initial value")
    return Batch(ctrl.skill_spec.n_robot_var, ctrl._nxv, ctrl._ny, time_var0, robot_var, virtual_var,
                 input_var if ctrl._ny else None)


def _speeds(max_speed, max_virtual_speed):
    inf = float("inf")
    return (ctypes.c_double(inf if max_speed is None else float(max_speed)),
            ctypes.c_double(inf if max_virtual_speed is None else float(max_virtual_speed)))


def rollout_jvp(ctrl, kind, time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed, max_virtual_speed,
                max_iter, t_dot, q_dot, x_dot, y_dot):
    """Shared body of ReactiveQPController / ReactiveNLPController.rollout_jvp: the rollout of rollout_batch (state
    updated in place) with the tangent of its state carried along, clik_<kind>_rollout_jvp on the current stream.
    -> {"sol", "n_failed", "q_dot", "x_dot", "sol_dot"}."""
    b = _rollout_batch(ctrl, "rollout_jvp", time_var0, robot_var, virtual_var, input_var)
    tptrs = _tangent_ptrs(ctrl, b, t_dot, q_dot, x_dot, y_dot)
    sol, failed, sd = b.empty(ctrl._qn), b.empty(0, "i32"), b.empty(ctrl._qn)
    qd = b.empty(ctrl.skill_spec.n_robot_var)
    xd = b.empty(ctrl._nxv) if ctrl._nxv else None
    skill = vjp_image(ctrl, kind, b.device_index, "rollout_jvp")
    runtime.check(getattr(runtime.load_library(), "clik_%s_rollout_jvp" % kind)(
        skill.handle, b.N, int(steps), ctypes.c_double(float(dt)), b.tp, b.t_stride, b.qp, b.xp, b.yp,
        *_speeds(max_speed, max_virtual_speed), b.ptr(sol), b.ptr(failed), max_iter, *tptrs, b.ptr(qd), b.ptr(xd),
        b.ptr(sd), b.stream()))
    return {"sol": sol, "n_failed": failed, "q_dot": qd, "x_dot": xd, "sol_dot": sd}


def rollout_jacobian(ctrl, kind, time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                     max_virtual_speed, max_iter):
    """Shared body of ReactiveQPController / ReactiveNLPController.rollout_jacobian: the rollout of rollout_batch
    with d(q_K, x_K)/d(t0, q0, x0, y) carried along, clik_<kind>_rollout_jacobian on the current stream.
    -> {"sol", "n_failed", "jac" (n_robot + n_virtual, n_theta, N)}."""
    b = _rollout_batch(ctrl, "rollout_jacobian", time_var0, robot_var, virtual_var, input_var)
    sol, failed = b.empty(ctrl._qn), b.empty(0, "i32")
    jac = b.torch.empty((ctrl.skill_spec.n_robot_var + ctrl._nxv, n_theta(ctrl), b.N), dtype=b.torch.float64,
                        device=b.device)
    skill = vjp_image(ctrl, kind, b.device_index, "rollout_jvp")
    runtime.check(getattr(runtime.load_library(), "clik_%s_rollout_jacobian" % kind)(
        skill.handle, b.N, int(steps), ctypes.c_double(float(dt)), b.tp, b.t_stride, b.qp, b.xp, b.yp,
        *_speeds(max_speed, max_virtual_speed), b.ptr(sol), b.ptr(failed), max_iter, b.ptr(jac), b.stream()))
    return {"sol": sol, "n_failed": failed, "jac": jac}


def _rollout_tape(ctrl, kind, b, steps, dt, max_speed, max_virtual_speed, max_iter):
    """clik_<kind>_rollout_tape for the Batch `b` (state updated in place, the rollout_batch bits) on the current
    stream -> (sol, n_failed, tape).  The tape is a private buffer of the reverse sweep: step-major (steps, rows, N)
    blocks in the step kernels' layout, allocated through torch, so that a request that does not fit fails there,
    before any launch."""
    steps = int(steps)
    if steps < 0:
        raise ValueError("steps must be >= 0")
    torch, N = b.torch, b.N
    f64 = lambda rows: torch.empty((steps, rows, N), dtype=torch.float64, device=b.device)  # noqa: E731
    tape = {"q": f64(ctrl.skill_spec.n_robot_var), "x": f64(ctrl._nxv) if ctrl._nxv else None, "sol": f64(ctrl._qn),
            "status": torch.empty((steps, N), dtype=torch.int32, device=b.device),
            "active": torch.empty((steps, 2, N), dtype=torch.int32, device=b.device)}
    sol, failed = b.empty(ctrl._qn), b.empty(0, "i32")
    skill = vjp_image(ctrl, kind, b.device_index, "rollout_vjp")
    runtime.check(getattr(runtime.load_library(), "clik_%s_rollout_tape" % kind)(
        skill.handle, N, steps, ctypes.c_double(float(dt)), b.tp, b.t_stride, b.qp, b.xp, b.yp,
        *_speeds(max_speed, max_virtual_speed), b.ptr(sol), b.ptr(failed), max_iter,
        *[b.ptr(tape[k]) for k in ("q", "x", "sol", "status", "active")], b.stream()))
    return sol, failed, tape


def _cotangent(ctrl, b, a, rows, name):
    """Validated cotangent (rows, N) of a rollout output: None (zero) or a CUDA float64 tensor on b's device."""
    if a is None or rows == 0:
        return None
    if not runtime._is_torch(a) or a.device != b.device:
        raise ValueError("%s must be a CUDA tensor on %s like robot_var" % (name, b.device))
    if tuple(a.shape) != (rows, b.N):
        raise ValueError("%s must have shape %s" % (name, (rows, b.N)))
    a = a.contiguous()
    runtime.dev_ptr(a, "f64", rows * b.N, name)
    return a


def _rollout_sweep(ctrl, kind, b, steps, dt, max_speed, max_virtual_speed, tape, q_bar, x_bar, sol_bar):
    """clik_<kind>_rollout_vjp over `tape` on the current stream -> (t_bar (N,), q_bar0, x_bar0 | None,
    y_bar | None)."""
    nq = ctrl.skill_spec.n_robot_var
    cot = [_cotangent(ctrl, b, a, r, n) for a, r, n in ((q_bar, nq, "q_bar"), (x_bar, ctrl._nxv, "x_bar"),
                                                        (sol_bar, ctrl._qn, "sol_bar"))]
    out = (b.empty(0), b.empty(nq), b.empty(ctrl._nxv) if ctrl._nxv else None, b.empty(ctrl._ny) if ctrl._ny else None)
    skill = vjp_image(ctrl, kind, b.device_index, "rollout_vjp")
    runtime.check(getattr(runtime.load_library(), "clik_%s_rollout_vjp" % kind)(
        skill.handle, b.N, int(steps), ctypes.c_double(float(dt)), b.tp, b.t_stride, b.yp,
        *_speeds(max_speed, max_virtual_speed), *[b.ptr(tape[k]) for k in ("q", "x", "sol", "status", "active")],
        *[b.ptr(a) for a in cot], *[b.ptr(a) for a in out], b.stream()))
    return out


def rollout_vjp(ctrl, kind, time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed, max_virtual_speed,
                max_iter, q_bar, x_bar, sol_bar):
    """Shared body of ReactiveQPController / ReactiveNLPController.rollout_vjp: the taped rollout (state updated in
    place, the rollout_batch bits), then the reverse sweep along (q_bar, x_bar, sol_bar), both on the current stream.
    -> {"sol", "n_failed", "t_bar", "q_bar", "x_bar", "y_bar"}."""
    b = _rollout_batch(ctrl, "rollout_vjp", time_var0, robot_var, virtual_var, input_var)
    sol, failed, tape = _rollout_tape(ctrl, kind, b, steps, dt, max_speed, max_virtual_speed, max_iter)
    tb, qb, xb, yb = _rollout_sweep(ctrl, kind, b, steps, dt, max_speed, max_virtual_speed, tape, q_bar, x_bar,
                                    sol_bar)
    return {"sol": sol, "n_failed": failed, "t_bar": tb, "q_bar": qb, "x_bar": xb, "y_bar": yb}


_ROLLOUT_FUNCTION = []


def _rollout_function():
    """torch.autograd.Function of a closed-loop rollout: forward the taped rollout, backward the reverse sweep, jvp
    rollout_jvp."""
    if _ROLLOUT_FUNCTION:
        return _ROLLOUT_FUNCTION[0]
    import torch
    from torch.autograd.function import once_differentiable

    class ControllerRollout(torch.autograd.Function):
        @staticmethod
        def forward(ctx, ctrl, kind, t0, q, x, y, steps, dt, max_speed, max_virtual_speed, max_iter):
            qK = q.detach().clone()
            xK = x.detach().clone() if x is not None else None
            b = _rollout_batch(ctrl, "rollout_batch_differentiable", t0, qK, xK, y)
            sol, failed, tape = _rollout_tape(ctrl, kind, b, steps, dt, max_speed, max_virtual_speed, max_iter)
            ctx.ctrl, ctx.kind, ctx.t0 = ctrl, kind, t0
            ctx.args = (steps, dt, max_speed, max_virtual_speed, max_iter)
            ctx.tape = tape
            ctx.save_for_backward(q, x, y)
            ctx.save_for_forward(q, x, y)
            ctx.mark_non_differentiable(failed)
            return qK, xK, sol, failed

        @staticmethod
        def jvp(ctx, _ctrl, _kind, t_dot, q_dot, x_dot, y_dot, *unused):
            q, x, y = ctx.saved_tensors
            ctrl, t0 = ctx.ctrl, ctx.t0
            steps, dt, vq, vx, mi = ctx.args
            c = lambda a: None if a is None else a.contiguous()  # noqa: E731
            if not torch.is_tensor(t0):
                t_dot = None
            qs = q.detach().clone()
            xs = x.detach().clone() if x is not None else None
            r = rollout_jvp(ctrl, ctx.kind, t0, qs, steps, dt, xs, y, vq, vx, mi, c(t_dot), c(q_dot),
                            c(x_dot) if x is not None else None, c(y_dot) if y is not None else None)
            return r["q_dot"], r["x_dot"], r["sol_dot"], None

        @staticmethod
        @once_differentiable
        def backward(ctx, q_bar, x_bar, sol_bar, _unused):
            q, x, y = ctx.saved_tensors
            ctrl, t0 = ctx.ctrl, ctx.t0
            steps, dt, vq, vx, _ = ctx.args
            b = _rollout_batch(ctrl, "rollout_batch_differentiable", t0, q, x, y)
            tb, qb, xb, yb = _rollout_sweep(ctrl, ctx.kind, b, steps, dt, vq, vx, ctx.tape, q_bar, x_bar, sol_bar)
            ctx.tape = None
            t_grad = None
            if torch.is_tensor(t0):
                t_grad = (tb.sum() if t0.numel() == 1 else tb).reshape(t0.shape).to(t0.dtype)
            return (None, None, t_grad, qb, xb if x is not None else None, yb if y is not None else None,
                    None, None, None, None, None)

    _ROLLOUT_FUNCTION.append(ControllerRollout)
    return ControllerRollout


def rollout_batch_differentiable(ctrl, kind, time_var0, robot_var, steps, dt, virtual_var, input_var, max_speed,
                                 max_virtual_speed, max_iter):
    """Shared body of the controllers' rollout_batch_differentiable: validated like rollout_vjp before anything is
    built, then the autograd Function."""
    _rollout_batch(ctrl, "rollout_batch_differentiable", time_var0, robot_var, virtual_var, input_var)
    return _rollout_function().apply(ctrl, kind, time_var0, robot_var, virtual_var, input_var if ctrl._ny else None,
                                     steps, dt, max_speed, max_virtual_speed, max_iter)


_STEP_FUNCTION = []


def _step_function():
    """torch.autograd.Function of a controller step: forward solve_batch, backward vjp_batch, jvp jvp_batch."""
    if _STEP_FUNCTION:
        return _STEP_FUNCTION[0]
    import torch
    from torch.autograd.function import once_differentiable

    class ControllerStep(torch.autograd.Function):
        @staticmethod
        def forward(ctx, ctrl, t, q, x, y, warmstart, max_iter):
            outs = ctrl.solve_batch(t, q, x, y, warmstart=warmstart, max_iter=max_iter)
            ctx.ctrl, ctx.t, ctx.n_outs = ctrl, t, len(outs)
            ctx.save_for_backward(q, x, y, *outs[:3])
            ctx.save_for_forward(q, x, y, *outs[:3])
            ctx.mark_non_differentiable(*outs[1:])
            return outs

        @staticmethod
        def jvp(ctx, _ctrl, t_dot, q_dot, x_dot, y_dot, *unused):
            # the warm start and max_iter carry no tangent; status / active / iterations get none
            q, x, y, sol, status, active = ctx.saved_tensors
            ctrl, t = ctx.ctrl, ctx.t
            c = lambda a: None if a is None else a.contiguous()  # noqa: E731
            if not torch.is_tensor(t):
                t_dot = None
            sol_dot = ctrl.jvp_batch(t, q, x, y, sol, status, active, t_dot=c(t_dot), q_dot=c(q_dot),
                                     x_dot=c(x_dot) if x is not None else None,
                                     y_dot=c(y_dot) if y is not None else None)
            return (sol_dot,) + (None,) * (ctx.n_outs - 1)

        @staticmethod
        @once_differentiable
        def backward(ctx, sol_bar, *unused):
            q, x, y, sol, status, active = ctx.saved_tensors
            ctrl, t = ctx.ctrl, ctx.t
            t_bar, q_bar, x_bar, y_bar = ctrl.vjp_batch(t, q, x, y, sol, status, active, sol_bar.contiguous())
            t_grad = None
            if torch.is_tensor(t):
                t_grad = (t_bar.sum() if t.numel() == 1 else t_bar).reshape(t.shape).to(t.dtype)
            return (None, t_grad, q_bar, x_bar if x is not None else None, y_bar if y is not None else None,
                    None, None)

    _STEP_FUNCTION.append(ControllerStep)
    return ControllerStep


def solve_batch_differentiable(ctrl, time_var, robot_var, virtual_var, input_var, warmstart, max_iter):
    """Shared body of the controllers' solve_batch_differentiable."""
    if not (runtime._is_torch(robot_var) and robot_var.is_cuda):
        raise ValueError("solve_batch_differentiable needs torch CUDA tensors")
    return _step_function().apply(ctrl, time_var, robot_var, virtual_var, input_var, warmstart, max_iter)


def skill_handle_array(skills):
    arr = (ctypes.c_void_p * len(skills))(*[s.handle for s in skills])
    return arr


def as_vector(value, n, what):
    """float / list / ndarray / DM -> float64 array of length n."""
    if isinstance(value, cs.GenericMatrixCommon):
        value = value.toarray()
    a = np.asarray(value, dtype=np.float64).reshape(-1)
    if a.size != n:
        raise ValueError("%s has %d entries, the skill expects %d" % (what, a.size, n))
    return a


def dm_column(a):
    return cs.DM(np.asarray(a, dtype=np.float64).reshape(-1, 1))


class Batch(object):
    """Validated structure-of-arrays view of (t, q, x, y) for N instances.

    Device path: torch CUDA float64 tensors, q of shape (n_robot, N) (coordinate-major, so
    instance i of coordinate j sits at q[j, i]); t a tensor of shape (N,) or a Python float.
    Host path: the same shapes as NumPy arrays (copied through the pipelined *_host ABI).
    """

    def __init__(self, n_rob, n_virt, n_in, t, q, x, y):
        self.on_device = runtime._is_torch(q)
        if self.on_device:
            import torch
            self.torch = torch
            if q.dim() != 2 or q.shape[0] != n_rob:
                raise ValueError("robot_var batch must have shape (%d, N), got %s" % (n_rob, tuple(q.shape)))
            self.N = int(q.shape[1])
            self.device = q.device
            if not torch.is_tensor(t):
                t = torch.full((1,), float(t), dtype=torch.float64, device=q.device)
            self.t_stride = 0 if t.numel() == 1 else 1
            if self.t_stride and t.numel() != self.N:
                raise ValueError("time_var batch must have N entries")
            if t.device != q.device:
                raise ValueError("time_var lives on %s, robot_var on %s" % (t.device, q.device))
            self.t = t
            self.tp = runtime.dev_ptr(t, "f64", t.numel(), "time_var")
            self.qp = runtime.dev_ptr(q, "f64", n_rob * self.N, "robot_var")
            self.xp = self._dev(x, n_virt, "virtual_var")
            self.yp = self._dev(y, n_in, "input_var")
            self.keep = (t, q, x, y)
        else:
            q = np.ascontiguousarray(q, dtype=np.float64)
            if q.ndim != 2 or q.shape[0] != n_rob:
                raise ValueError("robot_var batch must have shape (%d, N), got %s" % (n_rob, q.shape))
            self.N = q.shape[1]
            t = np.ascontiguousarray(np.asarray(t, dtype=np.float64).reshape(-1))
            self.t_stride = 0 if t.size == 1 else 1
            if self.t_stride and t.size != self.N:
                raise ValueError("time_var batch must have N entries")
            self.tp = ctypes.c_void_p(t.ctypes.data)
            self.qp = ctypes.c_void_p(q.ctypes.data)
            self.xp, x = self._host(x, n_virt, "virtual_var")
            self.yp, y = self._host(y, n_in, "input_var")
            self.keep = (t, q, x, y)

    def _dev(self, a, rows, what):
        if rows == 0:
            return None
        if a is not None and (not runtime._is_torch(a) or a.device != self.device):
            raise ValueError("%s must be a CUDA tensor on %s like robot_var" % (what, self.device))
        if a is None:
            a = self.torch.zeros((rows, self.N), dtype=self.torch.float64, device=self.device)
            self._zeros = getattr(self, "_zeros", []) + [a]
        if a.dim() != 2 or a.shape[0] != rows:
            raise ValueError("%s batch must have shape (%d, N)" % (what, rows))
        return runtime.dev_ptr(a, "f64", rows * self.N, what)

    def _host(self, a, rows, what):
        if rows == 0:
            return None, None
        if a is None:
            a = np.zeros((rows, self.N))
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.shape != (rows, self.N):
            raise ValueError("%s batch must have shape (%d, N), got %s" % (what, rows, a.shape))
        return ctypes.c_void_p(a.ctypes.data), a

    def empty(self, rows, dtype="f64"):
        """Output array (rows, N) on the same side as the inputs."""
        if self.on_device:
            dt = {"f64": self.torch.float64, "i32": self.torch.int32}[dtype]
            shape = (rows, self.N) if rows > 0 else (self.N,)
            return self.torch.empty(shape, dtype=dt, device=self.device)
        dt = {"f64": np.float64, "i32": np.int32}[dtype]
        return np.empty((rows, self.N) if rows > 0 else (self.N,), dtype=dt)

    def ptr(self, arr):
        if arr is None:
            return None
        if self.on_device:
            return ctypes.c_void_p(arr.data_ptr())
        return ctypes.c_void_p(arr.ctypes.data)

    def out_ptr(self, arr, rows, dtype, what):
        """Validated pointer of an output buffer (rows, N) — (N,) when rows == 0 — that the kernel
        writes in place: dtype, element count, contiguity and (device path) the device must match,
        because a wrong buffer would be an out-of-bounds write, not an exception."""
        if arr is None:
            return None
        numel = (rows if rows > 0 else 1) * self.N
        if self.on_device:
            if not runtime._is_torch(arr):
                raise runtime.ClikError("%s must be a CUDA tensor when the inputs are CUDA tensors" % what)
            if arr.device != self.device:
                raise runtime.ClikError("%s lives on %s, the inputs on %s" % (what, arr.device, self.device))
            return runtime.dev_ptr(arr, {"f64": "f64", "i32": "i32"}[dtype], numel, what)
        return runtime.host_out_ptr(arr, {"f64": np.float64, "i32": np.int32}[dtype], numel, what)

    @property
    def device_index(self):
        """CUDA ordinal the batch runs on: the tensors' device, or the default for host arrays."""
        if self.on_device:
            return self.device.index if self.device.index is not None else self.torch.cuda.current_device()
        return runtime.current_device()

    def stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)
