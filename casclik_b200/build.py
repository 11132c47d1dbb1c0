"""nvcc drivers: the in-tree C-ABI library and the per-skill cubins.

Both are sm_100a only (`-gencode arch=compute_100a,code=sm_100a`); artefacts stay inside the
package directory (`csrc/libclik_b200.so`, `_cache/<hash>.cubin`) so they travel with the source
tree.  This replaces the reference's per-function shell JIT (`jit: True`, `-O2`; reference
casclik/controllers/pseudo_inverse.py:59-65) with one cached compile per skill.
"""
import contextlib
import fcntl
import hashlib
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
CACHE_DIR = os.path.join(PKG_DIR, "_cache")
LIB_PATH = os.path.join(CSRC_DIR, "libclik_b200.so")
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "--expt-relaxed-constexpr"]


class BuildError(RuntimeError):
    pass


def nvcc_path():
    for cand in (os.environ.get("CLIK_NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise BuildError("nvcc not found (set CLIK_NVCC); skills cannot be compiled")


def _run(cmd, what):
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise BuildError("%s failed (exit %d)\n$ %s\n%s" % (what, proc.returncode, " ".join(cmd),
                                                            proc.stdout[-8000:]))
    return proc.stdout


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


@contextlib.contextmanager
def _build_lock(directory):
    """Serialises builds between processes (torchrun ranks all reach setup at the same moment):
    an exclusive fcntl lock on a file in the artefact directory.  Everything a build writes goes
    to a pid-suffixed temporary first and is renamed into place, so a reader outside the lock
    (another rank's dlopen, a cached-cubin read) never sees a half-written file."""
    os.makedirs(directory, exist_ok=True)
    fd = os.open(os.path.join(directory, ".build.lock"), os.O_CREAT | os.O_RDWR, 0o644)
    try:
        fcntl.flock(fd, fcntl.LOCK_EX)
        yield
    finally:
        try:
            fcntl.flock(fd, fcntl.LOCK_UN)
        finally:
            os.close(fd)


def library_sources():
    return [os.path.join(CSRC_DIR, f) for f in ("clik_abi.cu", "clik_qp.cuh")] + \
           [os.path.join(os.path.dirname(PKG_DIR), "include", "clik.h")]


def build_library(force=False, verbose=False):
    """Compile csrc/clik_abi.cu -> csrc/libclik_b200.so (static cudart: loads without a GPU)."""
    srcs = library_sources()
    if not force and _newer(LIB_PATH, srcs):
        return LIB_PATH
    with _build_lock(CSRC_DIR):
        if not force and _newer(LIB_PATH, srcs):      # another process built it while we waited
            return LIB_PATH
        tmp = LIB_PATH + ".tmp%d" % os.getpid()
        cmd = [nvcc_path()] + ARCH_FLAGS + COMMON_FLAGS + [
            "-shared", "-Xcompiler", "-fPIC", "-cudart", "static",
            "-o", tmp, os.path.join(CSRC_DIR, "clik_abi.cu")]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        try:
            out = _run(cmd, "building libclik_b200.so")
            os.replace(tmp, LIB_PATH)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
        if verbose:
            print(out)
    return LIB_PATH


def _kernel_headers():
    return [os.path.join(CSRC_DIR, f) for f in ("clik_pinv.cuh", "clik_pinv_group.cuh", "clik_qp.cuh", "clik_nlp.cuh",
                                                   "clik_math.cuh")]


def source_hash(source: str) -> str:
    h = hashlib.sha256()
    h.update(source.encode())
    for p in _kernel_headers():
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(ARCH_FLAGS + COMMON_FLAGS).encode())
    return h.hexdigest()[:20]


def compile_cubin(source: str, tag: str = "skill", keep_source=True, extra_flags=()):
    """Generated CUDA source -> cubin bytes (cached on the hash of source + kernel headers)."""
    os.makedirs(CACHE_DIR, exist_ok=True)
    key = source_hash(source + " ".join(extra_flags))
    safe = "".join(ch if ch.isalnum() else "_" for ch in tag)[:40]
    base = os.path.join(CACHE_DIR, "%s_%s" % (safe, key))
    cubin = base + ".cubin"
    if not os.path.exists(cubin):
        with _build_lock(CACHE_DIR):
            if not os.path.exists(cubin):             # not built by another process meanwhile
                pid = os.getpid()
                cu, cu_tmp = base + ".cu", base + ".tmp%d.cu" % pid
                tmp, log_tmp = cubin + ".tmp%d" % pid, base + ".log.tmp%d" % pid
                try:
                    # the source is renamed into place BEFORE nvcc runs so that -lineinfo records
                    # the path that stays on disk (ncu's source page); only the lock holder writes it
                    with open(cu_tmp, "w") as f:
                        f.write(source)
                    os.replace(cu_tmp, cu)
                    cmd = [nvcc_path()] + ARCH_FLAGS + COMMON_FLAGS + list(extra_flags) + [
                        "-cubin", "-I", CSRC_DIR, "-Xptxas=-v", "-o", tmp, cu]
                    log = _run(cmd, "compiling skill %s" % tag)
                    with open(log_tmp, "w") as f:
                        f.write(log)
                    os.replace(log_tmp, base + ".log")
                    os.replace(tmp, cubin)            # last: its existence marks the entry complete
                    if not keep_source:
                        os.remove(cu)
                finally:
                    for leftover in (cu_tmp, tmp, log_tmp):
                        if os.path.exists(leftover):
                            os.remove(leftover)
    with open(cubin, "rb") as f:
        return f.read(), cubin


def kernel_registers(cubin_path, kernel):
    """Registers per thread ptxas reported for `kernel` (from the compile log next to the cubin)."""
    import re
    log_path = cubin_path[:-len(".cubin")] + ".log"
    if not os.path.exists(log_path):
        return None
    with open(log_path) as f:
        log = f.read()
    key = "Compiling entry function '%s'" % kernel
    if key not in log:
        return None
    m = re.search(r"Used (\d+) registers", log[log.index(key):])
    return int(m.group(1)) if m else None


def kernel_stack_bytes(cubin_path, kernel):
    """Local-memory stack frame (spills + arrays) ptxas reported for `kernel`, in bytes per thread."""
    import re
    log_path = cubin_path[:-len(".cubin")] + ".log"
    if not os.path.exists(log_path):
        return None
    with open(log_path) as f:
        log = f.read()
    key = "Compiling entry function '%s'" % kernel
    if key not in log:
        return None
    m = re.search(r"(\d+) bytes stack frame", log[log.index(key):])
    return int(m.group(1)) if m else None
