"""ctypes binding of include/clik.h (csrc/libclik_b200.so) + the compiled-skill handle.

There is no CPU fallback: every entry point that computes needs a CUDA device and raises
`ClikError` if the library, the driver or the device is missing.
"""
import ctypes
import os

import numpy as np

from . import build

_c_double_p = ctypes.POINTER(ctypes.c_double)
_c_int32_p = ctypes.POINTER(ctypes.c_int32)
_c_uint32_p = ctypes.POINTER(ctypes.c_uint32)

ABI_VERSION = 2
QP_SOLVED, QP_MAXITER, QP_INFEASIBLE, QP_INVALID = 0, 1, 2, 4
NLP_STALLED = 5   # NLP step: the line search found no decrease (other codes as the QP's)


class ClikError(RuntimeError):
    pass


class SkillDesc(ctypes.Structure):
    _fields_ = [(name, ctypes.c_int32) for name in (
        "abi_version", "device", "n_robot", "n_virtual", "n_input", "n_slack", "n_modes",
        "has_pinv", "has_qp", "qp_n", "qp_m", "block_threads")]


#: every symbol include/clik.h declares (tests check that the library exports all of them)
EXPORTS = (
    "clik_skill_load", "clik_skill_free", "clik_pinv_step", "clik_pinv_rollout", "clik_qp_step",
    "clik_qp_rollout", "clik_qp_dense",
    "clik_pinv_step_host", "clik_qp_step_host", "clik_skill_launch_info",
    "clik_pinv_step_ld", "clik_qp_step_ld", "clik_pinv_step_host_multi", "clik_qp_step_host_multi",
    "clik_pinv_solve_one", "clik_qp_solve_one", "clik_skill_set_overlap", "clik_skill_get_overlap",
    "clik_nlp_step", "clik_nlp_step_host", "clik_nlp_solve_one", "clik_nlp_rollout",
    "clik_skill_set_staging", "clik_skill_get_staging",
    "clik_measure_fp64_peak", "clik_flush_l2", "clik_device_count", "clik_abi_version",
    "clik_last_error",
)

_lib = None


def library_path():
    return build.LIB_PATH


def load_library():
    """dlopen the in-tree C-ABI library (building it first if the .so is missing or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = build.LIB_PATH
    if not os.path.exists(path) or not build._newer(path, build.library_sources()):
        try:
            build.build_library()
        except build.BuildError as exc:
            if not os.path.exists(path):
                raise ClikError("libclik_b200.so is missing and cannot be built: %s" % exc)
    lib = ctypes.CDLL(path)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    lib.clik_last_error.restype = ctypes.c_char_p
    lib.clik_last_error.argtypes = []
    lib.clik_abi_version.restype = i32
    lib.clik_device_count.restype = i32
    lib.clik_skill_load.restype = i32
    lib.clik_skill_load.argtypes = [vp, ctypes.c_size_t, ctypes.POINTER(SkillDesc),
                                    ctypes.POINTER(vp)]
    lib.clik_skill_free.restype = None
    lib.clik_skill_free.argtypes = [vp]
    lib.clik_pinv_step.restype = i32
    lib.clik_pinv_step.argtypes = [vp, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.clik_pinv_step_host.restype = i32
    lib.clik_pinv_step_host.argtypes = [vp, i64, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.clik_pinv_step_ld.restype = i32
    lib.clik_pinv_step_ld.argtypes = [vp, i64, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.clik_qp_step_ld.restype = i32
    lib.clik_qp_step_ld.argtypes = [vp, i64, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.clik_pinv_step_host_multi.restype = i32
    lib.clik_pinv_step_host_multi.argtypes = [ctypes.POINTER(vp), i32, i64, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.clik_qp_step_host_multi.restype = i32
    lib.clik_qp_step_host_multi.argtypes = [ctypes.POINTER(vp), i32, i64, vp, i32, vp, vp, vp, vp, vp, vp,
                                            vp, vp, i32]
    lib.clik_pinv_solve_one.restype = i32
    lib.clik_pinv_solve_one.argtypes = [vp, ctypes.c_double, vp, vp, vp, vp, vp, vp]
    lib.clik_qp_solve_one.restype = i32
    lib.clik_qp_solve_one.argtypes = [vp, ctypes.c_double, vp, vp, vp, vp, vp, vp, vp, i32]
    lib.clik_pinv_rollout.restype = i32
    lib.clik_pinv_rollout.argtypes = [vp, i64, i32, ctypes.c_double, vp, i32, vp, vp, vp,
                                      ctypes.c_double, ctypes.c_double, vp, vp, vp, vp, vp]
    lib.clik_qp_rollout.restype = i32
    lib.clik_qp_rollout.argtypes = [vp, i64, i32, ctypes.c_double, vp, i32, vp, vp, vp,
                                    ctypes.c_double, ctypes.c_double, vp, vp, i32, vp]
    lib.clik_qp_step.restype = i32
    lib.clik_qp_step.argtypes = [vp, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.clik_qp_step_host.restype = i32
    lib.clik_qp_step_host.argtypes = [vp, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32]
    lib.clik_qp_dense.restype = i32
    lib.clik_qp_dense.argtypes = [i32, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.clik_nlp_step.restype = i32
    lib.clik_nlp_step.argtypes = [vp, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.clik_nlp_step_host.restype = i32
    lib.clik_nlp_step_host.argtypes = [vp, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32]
    lib.clik_nlp_solve_one.restype = i32
    lib.clik_nlp_solve_one.argtypes = [vp, ctypes.c_double, vp, vp, vp, vp, vp, vp, vp, vp, i32]
    lib.clik_nlp_rollout.restype = i32
    lib.clik_nlp_rollout.argtypes = [vp, i64, i32, ctypes.c_double, vp, i32, vp, vp, vp,
                                     ctypes.c_double, ctypes.c_double, vp, vp, i32, vp]
    lib.clik_skill_launch_info.restype = i32
    lib.clik_skill_launch_info.argtypes = [vp, i32, _c_int32_p, _c_int32_p, _c_int32_p, _c_int32_p]
    lib.clik_skill_set_overlap.restype = i32
    lib.clik_skill_set_overlap.argtypes = [vp, i32]
    lib.clik_skill_get_overlap.restype = i32
    lib.clik_skill_get_overlap.argtypes = [vp]
    lib.clik_skill_set_staging.restype = i32
    lib.clik_skill_set_staging.argtypes = [vp, i32]
    lib.clik_skill_get_staging.restype = i32
    lib.clik_skill_get_staging.argtypes = [vp]
    lib.clik_measure_fp64_peak.restype = i32
    lib.clik_measure_fp64_peak.argtypes = [i32, i32, _c_double_p]
    lib.clik_flush_l2.restype = i32
    lib.clik_flush_l2.argtypes = [i32, vp]
    if lib.clik_abi_version() != ABI_VERSION:
        raise ClikError("libclik_b200.so ABI %d != binding %d" % (lib.clik_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(status):
    if status != 0:
        raise ClikError("clik error %d: %s" % (status, load_library().clik_last_error().decode()))


def device_count():
    return int(load_library().clik_device_count())


def require_device():
    if device_count() < 1:
        raise ClikError("no CUDA device: the CLIK controller step runs on the GPU only "
                        "(there is no CPU fallback)")


def current_device():
    """Device ordinal used when the caller gives no device (host-array batches): LOCAL_RANK under
    torchrun, else torch's current device if torch has been imported, else 0.  Batches of CUDA
    tensors never come here: they run on the device the tensors live on."""
    import sys
    if "LOCAL_RANK" in os.environ:
        return int(os.environ["LOCAL_RANK"])
    if "torch" in sys.modules:
        torch = sys.modules["torch"]
        try:
            if torch.cuda.is_available():
                return int(torch.cuda.current_device())
        except Exception:
            pass
    return int(os.environ.get("LOCAL_RANK", "0"))


# ---- pointer helpers -------------------------------------------------------------------------------

def _is_torch(x):
    return type(x).__module__.startswith("torch")


def dev_ptr(tensor, dtype_name, numel, what):
    """Raw pointer of a contiguous CUDA tensor (validated)."""
    if tensor is None:
        return None
    import torch
    want = {"f64": torch.float64, "i32": torch.int32, "u32": torch.int32}[dtype_name]
    if not tensor.is_cuda:
        raise ClikError("%s must be a CUDA tensor" % what)
    if tensor.dtype != want and not (dtype_name == "u32" and tensor.dtype == torch.uint32):
        raise ClikError("%s must have dtype %s, got %s" % (what, want, tensor.dtype))
    if not tensor.is_contiguous():
        raise ClikError("%s must be contiguous (structure-of-arrays: shape (rows, N))" % what)
    if tensor.numel() != numel:
        raise ClikError("%s has %d elements, expected %d" % (what, tensor.numel(), numel))
    return ctypes.c_void_p(tensor.data_ptr())


def host_ptr(arr, dtype, numel, what):
    if arr is None:
        return None, None
    a = np.ascontiguousarray(arr, dtype=dtype)
    if a.size != numel:
        raise ClikError("%s has %d elements, expected %d" % (what, a.size, numel))
    return ctypes.c_void_p(a.ctypes.data), a


def host_out_ptr(arr, dtype, numel, what):
    """Pointer of a caller-supplied OUTPUT array: it is written in place, so it is never copied or
    converted — a buffer of the wrong dtype, size or layout is an error, not something to fix up."""
    if arr is None:
        return None
    if not isinstance(arr, np.ndarray):
        raise ClikError("%s must be a NumPy array when the inputs are host arrays" % what)
    if arr.dtype != np.dtype(dtype) and not (np.dtype(dtype) == np.int32 and arr.dtype == np.uint32):
        raise ClikError("%s must have dtype %s, got %s" % (what, np.dtype(dtype), arr.dtype))
    if not arr.flags["C_CONTIGUOUS"] or not arr.flags["WRITEABLE"]:
        raise ClikError("%s must be a writeable C-contiguous array (structure-of-arrays: shape (rows, N))" % what)
    if arr.size != numel:
        raise ClikError("%s has %d elements, expected %d" % (what, arr.size, numel))
    return ctypes.c_void_p(arr.ctypes.data)


class CompiledSkill(object):
    """A cubin loaded on one device through the C ABI."""

    def __init__(self, cubin_bytes, meta, n_slack=0, device=None):
        require_device()
        lib = load_library()
        self.meta = dict(meta)
        self.device = current_device() if device is None else int(device)
        d = SkillDesc()
        d.abi_version = ABI_VERSION
        d.device = self.device
        d.n_robot = meta["n_robot"]
        d.n_virtual = meta["n_virtual"]
        d.n_input = meta["n_input"]
        d.n_slack = n_slack
        d.n_modes = meta["n_modes"]
        d.has_pinv = int(meta["has_pinv"])
        d.has_qp = int(meta["has_qp"])
        d.qp_n = meta["qp_n"]
        d.qp_m = meta["qp_m"]
        d.block_threads = meta.get("block_threads", 128)
        self.desc = d
        self._image = ctypes.create_string_buffer(cubin_bytes, len(cubin_bytes))
        handle = ctypes.c_void_p()
        check(lib.clik_skill_load(self._image, len(cubin_bytes), ctypes.byref(d),
                                  ctypes.byref(handle)))
        self.handle = handle
        self._lib = lib

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.clik_skill_free(self.handle)
                self.handle = None
        except Exception:
            pass

    def set_overlap(self, level):
        """0: plain stream order; 1 (default): the second launch of a two-launch step is scheduled while
        the first drains; 2: successive step launches on one stream are declared independent (disjoint
        buffers) and may overlap tail and ramp (programmatic dependent launch; include/clik.h)."""
        check(self._lib.clik_skill_set_overlap(self.handle, int(level)))

    def overlap(self):
        return int(self._lib.clik_skill_get_overlap(self.handle))

    def set_staging(self, on):
        """TMA-staged persistent pinv kernel for device-resident batches (include/clik.h clik_skill_set_staging)."""
        check(self._lib.clik_skill_set_staging(self.handle, 1 if on else 0))

    def staging(self):
        return int(self._lib.clik_skill_get_staging(self.handle)) == 1

    def launch_info(self, which=0):
        g, b, r, l = (ctypes.c_int32() for _ in range(4))
        check(self._lib.clik_skill_launch_info(self.handle, which, ctypes.byref(g), ctypes.byref(b),
                                               ctypes.byref(r), ctypes.byref(l)))
        return {"grid": g.value, "block": b.value, "regs": r.value, "local_bytes": l.value}


def measure_fp64_peak(device=0, iters=1 << 16):
    require_device()
    out = ctypes.c_double()
    check(load_library().clik_measure_fp64_peak(device, iters, ctypes.byref(out)))
    return out.value


def flush_l2(device=0, stream=None):
    check(load_library().clik_flush_l2(device, ctypes.c_void_p(stream or 0)))
