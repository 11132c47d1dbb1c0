#!/usr/bin/env python
"""Drop-in audit (build container only — it reads the reference's notebooks from /root/reference):
execute the code cells of examples/notebooks/*.ipynb with `casadi`, `casclik` and `urdf2casadi`
resolved to this package, up to — not including — anything that needs a GPU (controller.solve calls
and what depends on their results), plotting or the out-of-scope MPC controller.  Controllers
are set up with load=False: lowered, emitted and compiled by nvcc, not loaded.  Prints per notebook
which cells ran, which were skipped and why, and every exception.

Usage:  python tools/notebook_audit.py [notebook ...]"""
import glob
import json
import os
import re
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
NB_DIR = "/root/reference/examples/notebooks"

import casclik_b200 as cc  # noqa: E402
from casclik_b200 import build as _build, cs, fk  # noqa: E402
import tempfile  # noqa: E402

# the ~60 controllers the notebooks define would otherwise land in the in-tree cubin cache that
# travels to the GPU box
_build.CACHE_DIR = tempfile.mkdtemp(prefix="clik_notebook_audit_")

# --- module stand-ins ------------------------------------------------------------------------------
sys.modules["casadi"] = cs
sys.modules["casclik"] = cc
u2c = types.ModuleType("urdf2casadi")
u2c.converter = fk.converter
for name in ("numpy_geom", "casadi_geom"):
    setattr(u2c, name, getattr(fk, name, types.ModuleType(name)))
sys.modules["urdf2casadi"] = u2c
for name in ("common_plots", "nice_plotting", "matplotlib", "matplotlib.pyplot", "matplotlib.animation",
             "IPython", "IPython.display", "mpl_toolkits", "mpl_toolkits.axes_grid1",
             "mpl_toolkits.axes_grid1.inset_locator"):
    sys.modules.setdefault(name, types.ModuleType(name))


class _Anything(object):
    def __init__(self, name=""):
        self._name = name

    def __getattr__(self, n):
        return _Anything(n)

    def __call__(self, *a, **k):
        if self._name in ("plot", "step", "semilogy", "loglog"):
            return [_Anything()]                      # `line, = ax.plot(...)`
        return _Anything()

    def __iter__(self):
        return iter((_Anything(), _Anything()))

    def __getitem__(self, k):
        return _Anything()

    def __setitem__(self, k, v):
        pass


for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation", "IPython.display", "common_plots",
             "nice_plotting", "mpl_toolkits.axes_grid1.inset_locator"):
    m = sys.modules[name]
    m.__getattr__ = lambda n, _m=m: _Anything(n)
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
sys.modules["matplotlib"].animation = sys.modules["matplotlib.animation"]

# controllers: build, do not load (no GPU here)
for cls in (cc.PseudoInverseController, cc.ReactiveQPController, cc.ReactiveNLPController):
    orig = cls.setup_problem_functions
    cls.setup_problem_functions = (lambda o: lambda self, load=False: o(self, load=False))(orig)
    cls.setup_solver = (lambda o: lambda self: o(self, load=False))(orig)



def _zeros(n):
    return cs.DM.zeros(n, 1) if n else None


def _fake_solve(self, time_var, robot_var, virtual_var=None, input_var=None, warmstart_robot_vel_var=None,
                warmstart_virtual_vel_var=None, warmstart_slack_var=None):
    """No GPU in the build container: zero commands of the right shapes, so that the Python around
    solve() in the notebooks (simulation loops, logging, warm starts) still executes."""
    spec = self.skill_spec
    self.current_mode = 0
    nv = spec.n_virtual_var if (virtual_var is not None and spec._has_virtual) else 0
    if isinstance(self, cc.PseudoInverseController):
        return _zeros(spec.n_robot_var), _zeros(nv), None
    return _zeros(spec.n_robot_var), _zeros(nv), _zeros(spec.n_slack_var)


def _fake_initial(self, time_var0, robot_var0, virtual_var0=None, robot_vel_var0=None, input_var0=None):
    spec = self.skill_spec
    return _zeros(spec.n_virtual_var if spec._has_virtual else 0), _zeros(spec.n_slack_var)


class _OutOfScopeController(object):
    """ModelPredictiveController (an NLP over a horizon; not part of this package)."""

    def __init__(self, skill_spec, *a, **k):
        self.skill_spec = skill_spec
        self.options = k.get("options") or {}

    def __getattr__(self, n):
        if n.startswith("setup"):
            return lambda *a, **k: None
        raise AttributeError(n)

    solve = _fake_solve
    solve_initial_problem = _fake_initial


for cls in (cc.PseudoInverseController, cc.ReactiveQPController, cc.ReactiveNLPController):
    cls.solve = _fake_solve
    cls.solve_initial_problem = _fake_initial
    cls.setup_initial_problem_solver = lambda self: None
cc.ModelPredictiveController = _OutOfScopeController

NEEDS_GPU = re.compile(r"a^")       # (nothing: solve() is faked above)
OUT_OF_SCOPE = re.compile(r"a^")
_UNUSED = re.compile(r"\.solve\(|\.solve_initial_problem\(|timeit|\bres\b|_res\b|controllers\[|cntrllr|ctrl_res")
_UNUSED2 = None
PLOT = re.compile(r"\bplt\.|common_plots|nice_plotting|animation|HTML\(|\bax\d*\.|fig")


def audit(path):
    nb = json.load(open(path))
    ns = {"__name__": "__notebook__", "xrange": range}       # (the notebooks are Python 2)
    os.chdir(NB_DIR)
    ran, skipped, failed = 0, [], []
    for idx, cell in enumerate(nb["cells"]):
        if cell["cell_type"] != "code":
            continue
        src = "".join(cell["source"])
        lines = [l for l in src.splitlines() if not l.lstrip().startswith(("%", "!"))]
        src = "\n".join(lines)
        if not src.strip():
            continue
        src = re.sub(r"(?m)^(\s*)print\s+(?!\()(.*)$", r"\1print(\2)", src)     # the notebooks are Python 2
        imports = "\n".join(l for l in src.splitlines() if re.match(r"(import|from)\s", l))
        if imports:
            exec(compile(imports, "imports", "exec"), ns)
        why = ("out of scope" if OUT_OF_SCOPE.search(src) else "needs GPU" if NEEDS_GPU.search(src) else None)
        if why:
            skipped.append((idx, why))
            continue
        try:
            exec(compile(src, "%s[cell %d]" % (os.path.basename(path), idx), "exec"), ns)
            ran += 1
        except NameError as exc:          # a name from a skipped cell: not a finding
            skipped.append((idx, "depends on a skipped cell (%s)" % exc))
        except Exception as exc:          # noqa: BLE001
            failed.append((idx, "%s: %s" % (type(exc).__name__, str(exc).splitlines()[0][:160] if str(exc) else "")))
    return ran, skipped, failed


if __name__ == "__main__":
    paths = sys.argv[1:] or sorted(glob.glob(os.path.join(NB_DIR, "*.ipynb")))
    total_failed = 0
    for p in paths:
        ran, skipped, failed = audit(p)
        print("%-62s ran %2d  skipped %2d  failed %d" % (os.path.basename(p), ran, len(skipped), len(failed)))
        for idx, msg in failed:
            print("    cell %d: %s" % (idx, msg))
        if os.environ.get("AUDIT_VERBOSE"):
            for idx, why in skipped:
                print("    (cell %d skipped: %s)" % (idx, why[:110]))
        total_failed += len(failed)
    sys.exit(1 if total_failed else 0)
