"""The C-ABI library loads on a machine without a GPU and exports every symbol that
include/clik.h declares; entry points that need a device fail with an error code, not a crash."""
import ctypes
import os
import re

import pytest

from casclik_b200 import runtime, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "clik.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(clik_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = runtime.load_library()
    names = _declared()
    assert len(names) >= 13
    for n in names:
        assert hasattr(lib, n), "libclik_b200.so does not export %s" % n
    assert sorted(runtime.EXPORTS) == names
    assert lib.clik_abi_version() == runtime.ABI_VERSION
    assert os.path.dirname(build.LIB_PATH).endswith(os.path.join("casclik_b200", "csrc"))


def test_descriptor_layout_matches_header():
    text = open(os.path.join(ROOT, "include", "clik.h")).read()
    body = text[text.index("typedef struct {"):text.index("} clik_skill_desc;")]
    fields = re.findall(r"int32_t\s+(\w+);", body)
    assert fields == [f[0] for f in runtime.SkillDesc._fields_]
    assert ctypes.sizeof(runtime.SkillDesc) == 4 * len(fields)


def test_argument_validation_needs_no_device():
    lib = runtime.load_library()
    out = ctypes.c_void_p()
    assert lib.clik_skill_load(None, 0, None, ctypes.byref(out)) == 1          # CLIK_ERR_INVALID
    assert b"NULL" in lib.clik_last_error()
    assert lib.clik_pinv_step(None, 4, None, 0, None, None, None, None, None, None, None) == 1
    assert lib.clik_qp_dense(0, 4, 99, 3, None, None, None, None, None, None, None, None, 0, None) == 1
    assert b"nx <= 32, m <= 64" in lib.clik_last_error()


# Host-array and single-instance entry points with a NULL skill or an empty handle array: (name, arguments after
# the handle(s) with N = 4 and every array NULL, message).  The *_multi forms are called with no array, with a
# count of 0 and with one NULL handle.
_HOST_ENTRY_POINTS = [
    ("clik_pinv_step_host", (4, None, 0) + (None,) * 6, b"no skill handles"),
    ("clik_qp_step_host", (4, None, 0) + (None,) * 8 + (0,), b"no skill handles"),
    ("clik_nlp_step_host", (4, None, 0) + (None,) * 8 + (0,), b"no skill handles"),
    ("clik_pinv_step_host_multi", (4, None, 0) + (None,) * 6, b"no skill handles"),
    ("clik_qp_step_host_multi", (4, None, 0) + (None,) * 8 + (0,), b"no skill handles"),
    ("clik_nlp_step_host_multi", (4, None, 0) + (None,) * 8 + (0,), b"no skill handles"),
    ("clik_qp_duals_host", (4, None, 0) + (None,) * 7, b"skill is NULL"),
    ("clik_nlp_duals_host", (4, None, 0) + (None,) * 7, b"skill is NULL"),
    ("clik_pinv_solve_one", (0.0,) + (None,) * 6, b"NULL argument"),
    ("clik_qp_solve_one", (0.0,) + (None,) * 7 + (0,), b"NULL argument"),
    ("clik_qp_solve_one_lam", (0.0,) + (None,) * 7 + (0, None), b"NULL argument"),
    ("clik_nlp_solve_one", (0.0,) + (None,) * 8 + (0,), b"NULL argument"),
    ("clik_nlp_solve_one_lam", (0.0,) + (None,) * 8 + (0, None), b"NULL argument"),
]


@pytest.mark.parametrize("name,args,message", _HOST_ENTRY_POINTS, ids=[e[0] for e in _HOST_ENTRY_POINTS])
def test_host_entry_points_reject_a_missing_skill_without_a_device(name, args, message):
    lib = runtime.load_library()
    fn = getattr(lib, name)
    if name.endswith("_multi"):
        one_null = (ctypes.c_void_p * 1)(None)
        calls = [(None, 1), (one_null, 0), (one_null, 1)]
    else:
        calls = [(None,)]
    for handles in calls:
        assert fn(*handles, *args) == 1, (name, handles)      # CLIK_ERR_INVALID
        assert message in lib.clik_last_error(), (name, handles, lib.clik_last_error())


def test_no_cpu_fallback_without_a_device():
    if runtime.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from casclik_b200 import scenarios
    ctrl = scenarios.get("ur5_track").make_controller()
    ctrl.setup_problem_functions(load=False)          # compiling needs no GPU ...
    with pytest.raises(runtime.ClikError):            # ... running does, loudly
        ctrl.solve(0.0, [0.1] * 6, input_var=[0.3, 0.3, 0.3])
    with pytest.raises(runtime.ClikError):
        ctrl.setup_solver()


def test_product_tree_never_touches_the_oracle_or_the_reference():
    """oracle/ is test infrastructure and /root/reference does not exist on the GPU box: nothing under
    casclik_b200/ (Python, CUDA, headers) may import, include, link or open either."""
    import re
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "casclik_b200")
    bad = []
    for dirpath, dirnames, filenames in os.walk(root):
        dirnames[:] = [d for d in dirnames if d not in ("_cache", "__pycache__")]
        for fn in filenames:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, fn), encoding="utf-8", errors="replace").read()
                if re.search(r"clik_oracle|oracle[/\\.]|/root/reference", text) or \
                        re.search(r"^\s*(import|from)\s+casadi\b", text, re.M):
                    bad.append(os.path.join(dirpath, fn))
    assert bad == []


def test_overlap_and_staging_switches_validate_without_a_device():
    """clik_skill_set_overlap / clik_skill_set_staging: argument errors need no GPU, and the controller-level
    switches are remembered until a skill handle exists."""
    from casclik_b200 import scenarios
    lib = runtime.load_library()
    assert lib.clik_skill_set_overlap(None, 1) == 1 and b"NULL" in lib.clik_last_error()
    assert lib.clik_skill_set_staging(None, 1) == 1
    assert lib.clik_skill_get_overlap(None) == -1 and lib.clik_skill_get_staging(None) == -1
    ctrl = scenarios.get("ur5_track").make_controller()
    ctrl.setup_problem_functions(load=False)
    assert ctrl.kernel_meta["pinv_staged_kernel"] is True
    ctrl.set_overlap(2)
    ctrl.set_input_staging(True)
    assert ctrl._overlap == 2 and ctrl._staging is True
    with pytest.raises(ValueError):
        ctrl.set_overlap(3)
    big = scenarios.get("iiwa_multitask_stress").make_controller()
    big.setup_problem_functions(load=False)
    assert big.kernel_meta["pinv_staged_kernel"] is False       # 19 input rows, 16 task rows
    with pytest.raises(runtime.ClikError):
        big.set_input_staging(True)
    qp = scenarios.get("ur5_qp").make_controller()
    qp.setup_problem_functions(load=False)
    qp.set_overlap(0)
    assert qp._overlap == 0
    assert qp.kernel_meta["qp_tail_cap"] == 4 and qp.kernel_meta["qp_dense_nnz"] == 17
