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


def vjp_image(ctrl, kind, device):
    """The skill's VJP image (emit_skill(..., vjp=True): the default image plus clik_<kind>_vjp_kernel) loaded on
    `device`.  Built and loaded on the first call, cached like every cubin, one handle per device: a controller
    that never asks for derivatives compiles nothing more."""
    if ctrl._vjp is None:
        source, meta = ctrl._vjp_source()
        cubin, path = build.compile_cubin(source, tag="%s_vjp_%s" % (kind, ctrl.skill_spec.label))
        ctrl._vjp = {"source": source, "meta": meta, "cubin": cubin, "path": path, "skills": {}}
    skills = ctrl._vjp["skills"]
    if device not in skills:
        skills[device] = runtime.CompiledSkill(ctrl._vjp["cubin"], ctrl._vjp["meta"],
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


_STEP_FUNCTION = []


def _step_function():
    """torch.autograd.Function of a controller step: forward solve_batch, backward vjp_batch."""
    if _STEP_FUNCTION:
        return _STEP_FUNCTION[0]
    import torch
    from torch.autograd.function import once_differentiable

    class ControllerStep(torch.autograd.Function):
        @staticmethod
        def forward(ctx, ctrl, t, q, x, y, warmstart, max_iter):
            outs = ctrl.solve_batch(t, q, x, y, warmstart=warmstart, max_iter=max_iter)
            ctx.ctrl, ctx.t = ctrl, t
            ctx.save_for_backward(q, x, y, *outs[:3])
            ctx.mark_non_differentiable(*outs[1:])
            return outs

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
