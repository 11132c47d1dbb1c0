"""The controller steps at and near kinematic singularities, against the 50-digit referee of
tests/mp_reference.py.  The kernels' own source runs as a host (g++) build through the harness of
test_kernel_code_on_host.py; tests/test_gpu_singular.py runs the sm_100a build on the same families.

Criterion (derived in mp_reference.py): where the 50-digit condition number kappa has kappa u < 1e-2,
results lie within C u kappa s + 1e-12 (s: the size of the terms the step adds up), and mode flags / working-set masks equal the 50-digit ones
wherever the decision margin exceeds its error bound.  Elsewhere no accuracy is claimed, but every output
must be written.  The largest ratios of error to bound and the number of instances inside a decision margin
are printed by the last test of the module."""
import ctypes
import math
import os

import numpy as np
import pytest

import casclik_b200 as cc
from casclik_b200 import scenarios
import mp_reference as mr
from oracle_bridge import oracle_pinv, oracle_qp_problem, orc
from test_kernel_code_on_host import _host_library, _inputs, _p

OBSERVED = {}
SENTINEL = 12345.678


def _note(key, v):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(v))


PINV_SKILLS = ["ur5_track", "ur5_moe2016_pinv", "iiwa_multitask", "iiwa_multitask_stress"]
PINV_OPTIONS = {"lam_1e-7": {}, "lam_1e-12": {"damping_factor": 1e-12}, "lam_1e-26": {"damping_factor": 1e-26},
                "standard": {"pinv_method": "standard"}}
# the undamped 50-digit kappa of the task Jacobian each family must reach somewhere in its delta sweep (its
# smallest value, at delta = 0.1, stays below 1e4 for every family): the straight-arm sets are singular, the
# iiwa's single joints and pairs only ill-conditioned for this 4-row pose task
FAMILY_KAPPA = {"elbow": 1e20, "wrist": 1e20, (1,): 1e2, (3,): 1e3, (5,): 1e3, (1, 3): 1e3, (1, 5): 1e5,
                (3, 5): 1e9, (1, 3, 5): 1e13}


def _families(name):
    return mr.UR5_FAMILIES if name.startswith("ur5") else mr.IIWA_FAMILIES


def family_batch(sc, draws, seed=0):
    """Every family of the skill, reachable and (where the skill has a target input) unreachable targets,
    concatenated -> (inputs, labels)."""
    parts, labels = [], []
    has_y = sc.sample(1)["y"] is not None
    for f in _families(sc.name):
        for reach in ((True, False) if has_y else (True,)):
            parts.append(mr.singular_inputs(sc, f, draws, seed=seed, reachable=reach))
            labels += [(f, reach)] * len(parts[-1]["delta"])
    inp = {k: (None if parts[0][k] is None else np.concatenate([p[k] for p in parts], axis=-1)) for k in parts[0]}
    return inp, labels


def check_family_kappa(sc, blocks, labels):
    """The inputs really sit where they are meant to: each family's undamped 50-digit kappa sweeps from a
    well-conditioned ~1e2 up to its singular end."""
    fk = mr.family_kappa(blocks)
    if blocks[-1].J.shape[1] > blocks[-1].J.shape[2]:
        # the 9-row three-point pose task of iiwa_multitask_stress has rank 6 at every configuration (DESIGN §5)
        assert fk.min() > 1e40, (sc.name, fk.min())
        return
    lab = np.array([str(l[0]) for l in labels])
    for f in set(l[0] for l in labels):
        k = fk[lab == str(f)]
        assert k.min() < 1e4 and k.max() >= FAMILY_KAPPA[f], (sc.name, f, k.min(), k.max())


def run_pinv(lib, inp, nq, kernel="clik_pinv_kernel", extra=()):
    t, q, x, y = _inputs({k: v for k, v in inp.items() if v is not None and k != "delta"})
    N = q.shape[1]
    v, mode = np.full((nq, N), SENTINEL), np.full(N, -9, dtype=np.int32)
    getattr(lib, kernel)(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y),
                         _p(v), None, _p(mode), *extra)
    return v, mode


def check_pinv(v, mode, ref, what, n_modes):
    """The criterion of the module docstring.  -> number of instances inside a decision margin."""
    assert not np.any(v == SENTINEL) and np.all((mode >= -1) & (mode < n_modes)), what + ": outputs not written"
    claim = ref["kappa"] * mr.U < mr.CLAIM
    decided = ref["ratio"] > 1.0
    bad = claim & decided & (mode != ref["mode"])
    assert not bad.any(), "%s: %d mode flags differ outside the decision margin (first %d: %d vs %d)" % (
        what, bad.sum(), np.argmax(bad), mode[np.argmax(bad)], ref["mode"][np.argmax(bad)])
    same = claim & (mode == ref["mode"])
    err = np.linalg.norm(v - ref["v"], axis=0)
    r = err[same] / mr.velocity_bound(ref)[same]
    _note("pinv " + what, r.max(initial=0.0))
    assert r.max(initial=0.0) <= 1.0, "%s: error / bound %.3e at kappa %.2e" % (
        what, r.max(), ref["kappa"][same][np.argmax(r)])
    undecided = int((claim & ~decided).sum())
    _note("pinv undecided " + what, undecided)
    return undecided


_REF = {}


def pinv_case(name, opts_key):
    """(scenario, inputs, 50-digit reference) for one skill and option set, cached for the module.  Four draws
    per delta for the UR5 skills, two for the iiwa, which has seven families."""
    draws = 4 if name.startswith("ur5") else 2
    key = (name, opts_key)
    if key not in _REF:
        sc = scenarios.get(name)
        if name not in _REF:
            inp, labels = family_batch(sc, draws)
            blocks, n = mr.mp_blocks(sc.spec, inp)
            check_family_kappa(sc, blocks, labels)
            _REF[name] = (sc, inp, blocks, n)
        sc, inp, blocks, n = _REF[name]
        opts = dict(sc.options or {}, **PINV_OPTIONS[opts_key])
        _REF[key] = (sc, inp, mr.pinv_reference(blocks, n, opts), opts)
    return _REF[key]


def test_referee_agrees_with_the_fp64_oracle_on_the_benchmark_distributions():
    """On the well-conditioned samplers the 50-digit referee and the fp64 oracle (orc.pinv_step,
    orc.solve_qp_single) agree to rounding: the referee evaluates the same formulas."""
    for name in PINV_SKILLS:
        sc = scenarios.get(name)
        inp = sc.sample(40, seed=11)
        blocks, n = mr.mp_blocks(sc.spec, inp)
        ref = mr.pinv_reference(blocks, n, sc.options)
        v64, m64 = oracle_pinv(sc.spec, inp, sc.options)
        assert np.array_equal(m64, ref["mode"])
        r = np.linalg.norm(v64 - ref["v"], axis=0) / mr.velocity_bound(ref)
        _note("fp64 oracle pinv " + name, r.max())
        assert r.max() <= 1.0, (name, r.max())
    for name in ("ur5_qp", "ur5_moe2016_qp"):
        sc = scenarios.get(name)
        inp = sc.sample(40, seed=11)
        h, A, lb, ub = oracle_qp_problem(sc.spec, inp)
        for i, rf in enumerate(mr.qp_reference(sc.spec, inp)):
            x64, lam64, st = orc.solve_qp_single(h, A[i], lb[i], ub[i])
            assert st == 0 and rf["cert"], (name, i)
            z = np.concatenate([x64 * np.sqrt(h), lam64])
            zr = np.concatenate([rf["x"] * np.sqrt(h), rf["lam"]])
            _note("fp64 oracle qp " + name, np.linalg.norm(z - zr) / rf["bound"])
            assert np.linalg.norm(z - zr) <= rf["bound"], (name, i)


def test_mp_eval_covers_every_op_and_raises_on_an_unknown_one():
    from casclik_b200.sym import dag
    import mpmath as mp
    a, b = dag.symbol("a"), dag.symbol("b")
    outs = [dag.if_else(dag.lt(a, b), dag.fmin(a, b), dag.fmax(a, b)), dag.atan2(a, b), dag.pow_(a, dag.const(3.0)),
            dag.logic_and(dag.le(a, b), dag.ne(a, b)), dag.logic_not(dag.eq(a, b)), dag.sign(dag.neg(a))]
    got = mr.mp_eval(outs, {a.id: 0.5, b.id: 2.0})
    assert got[0] == 0.5 and got[3] == 1 and got[4] == 1 and got[5] == -1 and got[2] == mp.mpf(0.125)
    with mp.workdps(mr.DPS):
        assert abs(got[1] - mp.atan2(0.5, 2.0)) < mp.mpf(10) ** -45
    odd = dag._new("bogus", (a,))
    with pytest.raises(NotImplementedError):
        mr.mp_eval([odd], {a.id: 1.0})


@pytest.mark.parametrize("fuse", ["1", "0"])
@pytest.mark.parametrize("name", PINV_SKILLS)
def test_pinv_near_singularities_against_the_50_digit_referee(name, fuse, tmp_path, monkeypatch):
    """Every damping the controller offers (1e-7, 1e-12, 1e-26, pinv_method="standard") on the singular
    families, with the fused first-equality form and the literal one (CLIK_FUSE_FIRST_EQ)."""
    monkeypatch.setenv("CLIK_FUSE_FIRST_EQ", fuse)
    for opts_key in PINV_OPTIONS:
        sc, inp, ref, opts = pinv_case(name, opts_key)
        ctrl = cc.PseudoInverseController(sc.spec, options=dict(opts))
        lib = _host_library(ctrl, _tmpdir(tmp_path, opts_key))
        v, mode = run_pinv(lib, inp, sc.spec.n_robot_var)
        check_pinv(v, mode, ref, "%s %s fuse=%s" % (name, opts_key, fuse), ctrl.n_modes)
        if opts_key == "standard" and name == "ur5_track":
            # lambda = 0 at the singular end: the Cholesky pivot of J J' is rounding noise.  What the kernel
            # returns there (DESIGN §5): NaN or inf where rounding makes a pivot zero or negative, otherwise a
            # finite vector of rounding-sized directions; never an unwritten output (checked above).
            hopeless = ref["kappa"] * mr.U >= mr.CLAIM
            _note("standard: instances without an accuracy claim", hopeless.sum())
            _note("standard: non-finite there", (~np.isfinite(v[:, hopeless]).all(axis=0)).sum())


def _tmpdir(tmp_path, name):
    p = tmp_path / name
    p.mkdir(exist_ok=True)
    return p


def test_pinv_split_and_group_routes_near_singularities(tmp_path, monkeypatch):
    """The two-launch form (fast pass + sub-warp group pass) and the group kernel from mode 0, on the iiwa
    skill with the run-time mode tail (closed-form unit-set modes off), against the referee."""
    monkeypatch.setenv("CLIK_UNIT_SETS", "0")
    for opts_key in ("lam_1e-7", "lam_1e-12"):
        sc, inp, ref, opts = pinv_case("iiwa_multitask", opts_key)
        ctrl = cc.PseudoInverseController(sc.spec, options=dict(opts))
        lib = _host_library(ctrl, _tmpdir(tmp_path, opts_key))
        meta = ctrl.kernel_meta
        assert meta["pinv_split"] and meta["pinv_group"]
        v, mode = run_pinv(lib, inp, 7)
        check_pinv(v, mode, ref, "iiwa one kernel " + opts_key, ctrl.n_modes)
        n_static = meta["pinv_static_modes"]
        t, q, x, y = _inputs({k: v_ for k, v_ in inp.items() if v_ is not None and k != "delta"})
        N = q.shape[1]
        v2, m2 = np.full((7, N), SENTINEL), np.full(N, -9, dtype=np.int32)
        head = (ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y), _p(v2), None, _p(m2))
        lib.clik_pinv_fast_kernel(*head)
        lib.clik_pinv_group_kernel(*head, ctypes.c_int(n_static), ctypes.c_int(1))
        assert np.array_equal(m2, mode)
        check_pinv(v2, m2, ref, "iiwa split " + opts_key, ctrl.n_modes)
        v3, m3 = run_pinv(lib, inp, 7, "clik_pinv_group_kernel", (ctypes.c_int(0), ctypes.c_int(0)))
        assert np.array_equal(m3, mode)
        check_pinv(v3, m3, ref, "iiwa group " + opts_key, ctrl.n_modes)


# ----------------------------------------------------------------------------------------------
# QP and multipliers
# ----------------------------------------------------------------------------------------------

def run_qp(lib, ctrl, inp, kernels=("clik_qp_kernel",), x0=None, active0=None):
    t, q, x, y = _inputs({k: v for k, v in inp.items() if v is not None and k != "delta"})
    N = q.shape[1]
    sol, status = np.full((ctrl._qn, N), SENTINEL), np.full(N, -9, dtype=np.int32)
    active = np.zeros((2, N), dtype=np.uint32)
    args = (ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x), _p(y if ctrl._ny else None),
            _p(x0), _p(active0), _p(sol), _p(status), _p(active), ctypes.c_int(10 * (ctrl._qn + ctrl._qm)))
    for k in kernels:
        getattr(lib, k)(*args)
    return sol, status, active


def check_qp(sol, status, active, refs, h, what, lam=None):
    """Status 0 on every instance the 50-digit certificate shows feasible; x (and lam) within the kappa-scaled
    bound in the metric of H; masks equal where the margin exceeds the bound; the multipliers' NaN rule."""
    sh = np.sqrt(h)
    undecided = 0
    for i, rf in enumerate(refs):
        if rf["status64"] != 0:
            assert status[i] in (0, 2), (what, i, status[i], rf["status64"])
            if status[i] == 0:   # the kernel found a point: it must be feasible at 50 digits (checked by the face)
                _note(what + " kernel solved an instance the fp64 oracle called infeasible", 1)
            continue
        assert rf["cert"], (what, i, "the fp64 working set fails the 50-digit certificate")
        assert status[i] == 0, (what, i, int(status[i]))
        assert np.all(sol[:, i] != SENTINEL)
        if lam is not None:
            check_rank_rule(lam[:, i], rf["problem"], int(active[0, i]), int(active[1, i]), (what, i))
        if rf["kappa"] * mr.U >= mr.CLAIM:
            continue
        masks_equal = (int(active[0, i]), int(active[1, i])) == (rf["up"], rf["lo"])
        if rf["ratio"] > 1.0:
            assert masks_equal, (what, i, rf["ratio"])
        else:
            undecided += 1
        if not masks_equal:
            continue
        zr = rf["x"] * sh
        r = np.linalg.norm(sol[:, i] * sh - zr) / rf["bound"]
        _note("qp x " + what, r)
        assert r <= 1.0, (what, i, r, rf["kappa"])
        if lam is not None and not np.isnan(lam[:, i]).any():
            li = lam[:, i]
            if True:
                r = np.linalg.norm(li - rf["lam"]) / rf["bound"]
                _note("qp lam " + what, r)
                assert r <= 1.0, (what, i, r, rf["kappa"])
    _note("qp undecided " + what, undecided)
    return undecided


def check_rank_rule(li, problem, up, lo, where):
    """The multipliers of a working set are NaN only where its rows (in the metric of H) have
    sigma_min / sigma_max below the kernel's 1e-12 rank threshold widened by RANK_BAND, and NaN wherever that
    ratio is below the threshold narrowed by RANK_BAND.  -> the 50-digit ratio."""
    h, A = problem[0], problem[1]
    rows = [r for r in range(A.shape[0]) if ((up | lo) >> r) & 1]
    ratio = mr.face_rank_ratio(h, A, rows) if rows else 1.0
    if np.isnan(li).any():
        assert np.isnan(li).all() and ratio < 1e-12 * mr.RANK_BAND, (where, "NaN on a full-rank face", ratio)
    else:
        assert ratio > 1e-12 / mr.RANK_BAND, (where, "finite multipliers on a rank-deficient face", ratio)
    return ratio


_QREF = {}


def qp_case(name, draws=3):
    if name not in _QREF:
        sc = scenarios.get(name)
        inp, labels = family_batch(sc, draws)
        blocks, _ = mr.mp_blocks(sc.spec, inp)
        check_family_kappa(sc, [b for b in blocks if b.kind == orc.EQ], labels)
        h, _, _, _ = oracle_qp_problem(sc.spec, {k: v for k, v in inp.items() if k != "delta"})
        _QREF[name] = (sc, inp, mr.qp_reference(sc.spec, inp, blocks), h, draws)
    return _QREF[name]


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_qp_and_multipliers_near_singularities(name, tmp_path):
    """Cold solves, the fast + tail split, warm starts from the neighbouring delta of the same draw, and the
    multipliers of the cold solution."""
    sc, inp, refs, h, draws = qp_case(name)
    ctrl = sc.make_controller()
    lib = _host_library(ctrl, tmp_path)
    sol, status, active = run_qp(lib, ctrl, inp)
    t, q, x, y = _inputs({k: v for k, v in inp.items() if v is not None and k != "delta"})
    N = q.shape[1]
    lam = np.full((ctrl._qm, N), -7.0)
    lib.clik_qp_duals_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x),
                             _p(y if ctrl._ny else None), _p(sol), _p(status), _p(active), _p(lam))
    assert not np.any(lam == -7.0)
    check_qp(sol, status, active, refs, h, name + " cold", lam)
    if ctrl.kernel_meta.get("qp_split"):
        # what the prediction pass certifies ends on its own face to rounding (mp_reference.qp_residuals),
        # whatever kappa: the check that sees a working set accepted by a loosened row test
        sf, stf, af = run_qp(lib, ctrl, inp, ("clik_qp_fast_kernel",))
        fast = np.nonzero(stf == 0)[0]
        assert len(fast) > len(stf) // 3
        for i in fast:
            r = mr.qp_residuals(*refs[i]["problem"], sf[:, i], int(af[0, i]), int(af[1, i]))
            _note("qp fast-pass residual " + name, r)
            assert r <= 1.0, (name, i, r)
        s2, st2, a2 = run_qp(lib, ctrl, inp, ("clik_qp_fast_kernel", "clik_qp_tail_kernel"))
        assert np.array_equal(s2, sol) and np.array_equal(st2, status) and np.array_equal(a2, active)
    # warm start: instance i takes the solution and working set of the instance one delta step before it
    prev = np.roll(np.arange(N), draws)
    x0 = np.ascontiguousarray(sol[:, prev])
    x0[~np.isfinite(x0)] = 0.0
    a0 = np.ascontiguousarray(active[:, prev])
    sw, stw, aw = run_qp(lib, ctrl, inp, x0=x0, active0=a0)
    check_qp(sw, stw, aw, refs, h, name + " warm")


@pytest.mark.parametrize("name", ["ur5_qp", "ur5_moe2016_qp"])
def test_multipliers_rank_rule_on_dependent_faces(name, tmp_path):
    """Working sets chosen to be rank deficient, handed to the multiplier kernel: on ur5_qp a joint-limit row
    and the speed-limit row of the same joint (identical rows, exactly dependent); on Moe-2016 the three box
    rows on the singular families, whose sigma_min / sigma_max sweeps through the kernel's 1e-12 threshold.
    The NaN rule of check_rank_rule must hold on every instance, and both of its branches must run."""
    sc, inp, refs, h, draws = qp_case(name)
    ctrl = sc.make_controller()
    lib = _host_library(ctrl, tmp_path)
    sol, _, _ = run_qp(lib, ctrl, inp)
    sol = np.ascontiguousarray(np.where(np.isfinite(sol), sol, 0.0))
    t, q, x, y = _inputs({k: v for k, v in inp.items() if v is not None and k != "delta"})
    N = q.shape[1]
    if name == "ur5_qp":         # rows: 3 soft position rows, 6 joint limits, 6 joint speeds
        j = np.arange(N) % 6
        up = ((1 << (3 + j)) | (1 << (9 + j))).astype(np.uint32)
    else:                        # rows 0-2: the three box SetConstraints
        up = np.full(N, 7, dtype=np.uint32)
    active = np.ascontiguousarray(np.stack([up, np.zeros(N, dtype=np.uint32)]))
    status = np.zeros(N, dtype=np.int32)
    lam = np.full((ctrl._qm, N), -7.0)
    lib.clik_qp_duals_kernel(ctypes.c_longlong(N), ctypes.c_longlong(N), _p(t), ctypes.c_int(1), _p(q), _p(x),
                             _p(y if ctrl._ny else None), _p(sol), _p(status), _p(active), _p(lam))
    ratios = np.array([check_rank_rule(lam[:, i], refs[i]["problem"], int(up[i]), 0, (name, i)) for i in range(N)])
    nan = np.isnan(lam).any(axis=0)
    if name == "ur5_qp":
        assert np.all(ratios == 0.0) and nan.all()
    else:
        assert nan.any() and (~nan).any() and (ratios < 1e-15).any() and ((ratios > 1e-15) & (ratios < 1e-9)).any()
    _note("rank rule %s: NaN faces" % name, nan.sum())


def test_report_observed_maxima():
    """Runs last in this module: the largest ratios of error to bound, and the instance counts."""
    print("observed maxima:", {k: "%.2e" % v for k, v in sorted(OBSERVED.items())})
