"""ctypes loader for oracle/clik_oracle.c (TEST / BASELINE INFRASTRUCTURE ONLY; see the header of
clik_oracle.c).  Importable from tests/ and bench.py only."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "libclik_oracle.so")


class Joint(ctypes.Structure):
    _fields_ = [("type", ctypes.c_int), ("xyz", ctypes.c_double * 3), ("R", ctypes.c_double * 9),
                ("axis", ctypes.c_double * 3)]


_lib = None


def load(build_if_missing=True):
    global _lib
    if _lib is None:
        src = os.path.join(HERE, "clik_oracle.c")
        if (not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src)) and build_if_missing:
            subprocess.run(["make", "-s", "-C", HERE], check=True)
        _lib = ctypes.CDLL(LIB)
        _lib.clik_ref_pinv_track.restype = ctypes.c_int
        _lib.clik_ref_pinv_track.argtypes = [ctypes.POINTER(Joint), ctypes.c_int, ctypes.c_int,
                                             ctypes.c_long, ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.c_double, ctypes.c_double, ctypes.c_void_p,
                                             ctypes.c_int]
        _lib.clik_ref_max_threads.restype = ctypes.c_int
    return _lib


def chain_table(chain):
    """clik_oracle.load_chain(...) output -> C array of joints."""
    arr = (Joint * len(chain))()
    for k, (jt, xyz, Ro, axis, _, _) in enumerate(chain):
        arr[k].type = 1 if jt in ("revolute", "continuous") else 0
        arr[k].xyz[:] = list(map(float, xyz))
        arr[k].R[:] = list(map(float, np.asarray(Ro).reshape(-1)))
        a = np.asarray(axis, dtype=float)
        arr[k].axis[:] = list(a / np.linalg.norm(a))
    return arr


def max_threads():
    """All host cores this process may use.  Deliberately not omp_get_max_threads(): torchrun
    exports OMP_NUM_THREADS=1, which would silently turn the CPU baseline into a 1-core run."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def pinv_track(chain, q, y, gain=1.0, lam=1e-7, threads=0):
    """q (n, N), y (3, N) float64 coordinate-major -> qdot (n, N), threads used."""
    lib = load()
    q = np.ascontiguousarray(q, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    n, N = q.shape
    out = np.empty_like(q)
    tab = chain_table(chain)
    used = lib.clik_ref_pinv_track(tab, len(chain), n, N, q.ctypes.data, y.ctypes.data,
                                   float(gain), float(lam), out.ctypes.data, int(threads))
    return out, used


# ---- generic skills: generated expression code + the hand-written controller logic -------------------

class RefCons(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int), ("row0", ctypes.c_int), ("rows", ctypes.c_int),
                ("set_index", ctypes.c_int)]


class RefSkill(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int), ("m", ctypes.c_int), ("nc", ctypes.c_int),
                ("cons", ctypes.POINTER(RefCons)), ("n_modes", ctypes.c_int),
                ("mode_masks", ctypes.POINTER(ctypes.c_uint)), ("damped", ctypes.c_int),
                ("lam", ctypes.c_double)]


EVAL_DECL = "double t, const double* q, const double* x, const double* y"

_evals = {}


def _compile_eval(nodes, names, tag):
    """Expression graph -> plain C (the emitter's C flavour: what CasADi's code generator + `jit` do in
    the reference) -> gcc -O2 -> function pointer `void ev(t, q, x, y, out)`.  Compiled in a temporary
    directory that is gone once the library is loaded (bench.py runs from trees it may not write to);
    cached per process on the source."""
    import hashlib
    import tempfile
    from casclik_b200.codegen import emit_c_function
    src = emit_c_function("ev", names, nodes, EVAL_DECL)
    key = hashlib.sha256(src.encode()).hexdigest()
    if key not in _evals:
        with tempfile.TemporaryDirectory(prefix="clik_oracle_eval_") as tmp:
            c, so = os.path.join(tmp, "eval_%s.c" % tag), os.path.join(tmp, "eval_%s.so" % tag)
            with open(c, "w") as f:
                f.write(src)
            subprocess.run(["gcc", "-O2", "-shared", "-fPIC", "-o", so, c, "-lm"], check=True)
            _evals[key] = ctypes.CDLL(so)
    lib = _evals[key]
    return lib, ctypes.cast(lib.ev, ctypes.c_void_p)


def _bind_generic(lib):
    if getattr(lib, "_generic_bound", False):
        return
    vp, ci, cl = ctypes.c_void_p, ctypes.c_int, ctypes.c_long
    lib.clik_ref_pinv_batch.restype = ci
    lib.clik_ref_pinv_batch.argtypes = [ctypes.POINTER(RefSkill), vp, cl, vp, ci, vp, ci, vp, ci, vp, ci, vp, vp, ci]
    lib.clik_ref_qp_batch.restype = ci
    lib.clik_ref_qp_batch.argtypes = [ci, ci, vp, cl, vp, ci, vp, ci, vp, ci, vp, ci, vp, vp, vp, ci, ci]
    lib._generic_bound = True


def _arr(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


class PinvPort(object):
    """C restatement of PseudoInverseController.solve for one skill (see clik_oracle.c, generic part)."""

    def __init__(self, spec, options=None):
        from casclik_b200.codegen import PinvProgram
        from casclik_b200.controllers import PseudoInverseController
        from casclik_b200.controllers._modes import activation_map
        from casclik_b200.sym import dag
        opts = PseudoInverseController(spec, options=dict(options or {})).options
        if opts["multidim_sets"] or opts["converge_final_set_to_max"]:
            raise NotImplementedError("the C port restates the default pinv path only")
        prog = PinvProgram(spec, opts)
        self.prog = prog
        m, ns = prog.m, prog.ns
        zero = dag.ZERO
        J, des, e, jt, smin, smax = [], [zero] * m, [zero] * m, [zero] * m, [zero] * m, [zero] * m
        cons = []
        for b in prog.blocks:
            for r in range(b["rows"]):
                g = b["row0"] + r
                J += list(b["J"][r])
                if b["kind"] in (0, 2):
                    des[g] = b["des"][r]
                else:
                    e[g], jt[g], smin[g], smax[g] = b["e"][r], b["jt"][r], b["smin"][r], b["smax"][r]
            cons.append((b["kind"], b["row0"], b["rows"], max(b["set_index"], 0)))
        self._evlib, self._ev = _compile_eval(J + des + e + jt + smin + smax, dict(prog.syms.names),
                                              "pinv_" + "".join(ch if ch.isalnum() else "_" for ch in spec.label))
        self._cons = (RefCons * len(cons))(*[RefCons(*c) for c in cons])
        amap = activation_map(prog.n_sets)
        masks = [sum(b << k for k, b in enumerate(row)) for row in amap] or [0]
        self._masks = (ctypes.c_uint * len(masks))(*masks)
        self.skill = RefSkill(ns, m, len(cons), self._cons, len(masks), self._masks,
                              1 if prog.damped else 0, float(prog.damping))
        self.nq, self.nx, self.ny = prog.n_rob, prog.n_virt, prog.n_in

    def solve(self, inp, threads=0):
        """inp: dict(t (N,), q (nq, N), x, y) coordinate-major -> (v (ns, N), mode (N,), threads used)."""
        lib = load()
        _bind_generic(lib)
        q = _arr(inp["q"])
        N = q.shape[1]
        t = _arr(np.broadcast_to(np.asarray(inp["t"], dtype=np.float64).reshape(-1), (N,)))
        x = _arr(inp.get("x")) if self.nx else None
        if self.nx and x is None:
            x = np.zeros((self.nx, N))
        y = _arr(inp.get("y")) if self.ny else None
        v = np.empty((self.skill.n, N))
        mode = np.empty(N, dtype=np.int32)
        p = lambda a: None if a is None else a.ctypes.data  # noqa: E731
        used = lib.clik_ref_pinv_batch(ctypes.byref(self.skill), self._ev, N, p(t), 1, p(q), self.nq, p(x), self.nx,
                                       p(y), self.ny, p(v), p(mode), int(threads))
        return v, mode, used


class QpPort(object):
    """C restatement of ReactiveQPController.solve for one skill."""

    def __init__(self, spec, **weights):
        from casclik_b200.codegen import QpProgram
        from casclik_b200.controllers import ReactiveQPController
        ctrl = ReactiveQPController(spec, **weights)
        prog = QpProgram(spec, ctrl.robot_var_weights, ctrl.virtual_var_weights, ctrl.slack_var_weights,
                         ctrl.weight_shifter)
        self.prog = prog
        nodes = [n for row in prog.A for n in row] + list(prog.lb) + list(prog.ub) + list(prog.h)
        self._evlib, self._ev = _compile_eval(nodes, dict(prog.syms.names),
                                              "qp_" + "".join(ch if ch.isalnum() else "_" for ch in spec.label))
        self.n, self.m = prog.nx, prog.m
        self.nq, self.nx, self.ny = prog.n_rob, prog.n_virt, prog.n_in

    def solve(self, inp, threads=0, max_iter=0):
        lib = load()
        _bind_generic(lib)
        q = _arr(inp["q"])
        N = q.shape[1]
        t = _arr(np.broadcast_to(np.asarray(inp["t"], dtype=np.float64).reshape(-1), (N,)))
        x = _arr(inp.get("x")) if self.nx else None
        if self.nx and x is None:
            x = np.zeros((self.nx, N))
        y = _arr(inp.get("y")) if self.ny else None
        sol = np.empty((self.n, N))
        status = np.empty(N, dtype=np.int32)
        active = np.empty((2, N), dtype=np.uint32)
        p = lambda a: None if a is None else a.ctypes.data  # noqa: E731
        used = lib.clik_ref_qp_batch(self.n, self.m, self._ev, N, p(t), 1, p(q), self.nq, p(x), self.nx, p(y), self.ny,
                                     p(sol), p(status), p(active), int(max_iter) or 10 * (self.n + self.m),
                                     int(threads))
        return sol, status, active, used
