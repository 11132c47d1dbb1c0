"""bench.py's reference arm runs on host cores only, so its side of the JSON contract can be checked
without a GPU: one JSON line, the required keys, rank != 0 silent under a multi-rank launch.  So can the
host side of --dump-outputs and the argument checks."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, *args):
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env.update(extra_env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "8192",
                        "--steps", "2", "--warmup", "1"] + list(args), env=env, capture_output=True, text=True,
                       timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return [l for l in p.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("controller-steps/sec") and d["unit"] == "controller-steps/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None and d["scaling"] == "weak"
    assert d["value"] > 0 and abs(d["value"] - 8192 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["config"]["workload"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0
    # the other BASELINE configs (iiwa multi-task, UR5 QP, Moe-2016 SRMTP + QP) are timed beside it
    sec = d["secondary"]
    assert set(sec) == {"iiwa_multitask", "ur5_qp", "ur5_moe2016_pinv", "ur5_moe2016_qp"}
    for name, leg in sec.items():
        assert "error" not in leg, (name, leg)
        assert leg["value"] > 0 and leg["cpu_baseline"]["kind"] == "port" and leg["cpu_baseline"]["cores"] >= 1


def test_reference_arm_only_rank_zero_works_under_a_multi_rank_launch():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2", "--no-secondary") == []
    lines = _run({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, "--gpus", "2", "--no-secondary")
    assert len(lines) == 1 and json.loads(lines[0])["n_gpus"] == 2


def test_dump_outputs_writes_float64_and_samples_the_same_instances_when_too_large(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    vel, mode = rng.standard_normal((6, 5000)), rng.integers(0, 4, 5000).astype(np.int32)
    bench.dump_outputs(str(tmp_path / "all"), {"robot_vel": vel, "virtual_vel": None, "mode": mode})
    assert sorted(os.listdir(tmp_path / "all")) == ["mode.npy", "robot_vel.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "robot_vel.npy"), vel)
    got = np.load(tmp_path / "all" / "mode.npy")
    assert got.dtype == np.float64 and np.array_equal(got, mode)

    monkeypatch.setattr(bench, "DUMP_LIMIT", 8 * 8 * 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"robot_vel": vel, "mode": mode})
    total = sum(os.path.getsize(tmp_path / "a" / f) - 128 for f in os.listdir(tmp_path / "a"))
    assert total <= bench.DUMP_LIMIT
    idx = np.load(tmp_path / "a" / "instances.npy").astype(np.int64)
    assert len(idx) == 1000 and np.array_equal(idx, np.unique(idx))
    assert np.array_equal(np.load(tmp_path / "a" / "robot_vel.npy"), vel[:, idx])
    assert np.array_equal(np.load(tmp_path / "a" / "mode.npy"), mode[idx])
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


def test_steps_below_one_is_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 2 and "--steps" in p.stderr
