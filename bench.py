#!/usr/bin/env python
"""bench.py — controller-steps/sec of the batched CLIK controller step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--scenario ur5_track] [--batch 1048576] [--no-secondary] [--dump-outputs DIR]

A "step" is one pass of the hot path (PseudoInverseController.solve for every instance of the
batch — reference casclik/controllers/pseudo_inverse.py:512-556) over one batch of synthetic
inputs (BASELINE.json configs[1]: UR5, one EqualityConstraint, 2^20 random joint states/targets
per GPU, fp64).  One JSON line is printed by rank 0; see the keys at the bottom.

Timing: W warm-up steps, then exactly K steps between (barrier + synchronize), timed with CUDA
events on the launch stream, MAX over ranks.  The step rotates over several resident input AND
output sets whose total size exceeds L2 (126 MB), so no step re-reads a cache-resident batch and
every result has to reach DRAM.  `value` times device-resident inputs; `e2e` times the same step
through the host-buffer C ABI (pinned host inputs, H2D + kernel + D2H inside the timed region).

`secondary` (same JSON line) carries the other BASELINE configs measured the same way in the same
run — configs[2] iiwa multi-task 2^20, configs[3] UR5 QP 2^18, configs[4] Moe-2016 SRMTP and QP with
a global batch of 2^23 sharded over the ranks — each with its own roofline and CPU baseline.

`--impl reference` times the restated reference CPU path (oracle/clik_oracle.c, all host
threads) on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/<name>.npy, so that two
builds run with the same arguments (same seeded inputs) can be compared output for output; see
dump_outputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "controller-steps/sec (fp64, batch N)"
UNIT = "controller-steps/s"

#: BASELINE.json configs measured next to the headline one: (scenario, batch, "weak" = per GPU | "strong" = global)
SECONDARY = (
    ("iiwa_multitask", 1 << 20, "weak", "configs[2]"),
    ("ur5_qp", 1 << 18, "weak", "configs[3]"),
    ("ur5_moe2016_pinv", 1 << 23, "strong", "configs[4] SRMTP"),
    ("ur5_moe2016_qp", 1 << 23, "strong", "configs[4] ReactiveQP"),
)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_counts():
    """Per-scenario figures taken from ncu captures of this bench (profiles/r2_ncu_counts.json, written by
    tools/ncu_counts.py): DRAM bytes per launch and EXECUTED fp64 thread-instructions per instance."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_counts.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def _launch_info(ctrl, is_qp):
    sk = ctrl._skill()
    if is_qp:
        info = sk.launch_info(1)
        if ctrl.kernel_meta.get("qp_split") and os.environ.get("CLIK_QP_SPLIT", "1") != "0":
            info = {"fast": sk.launch_info(3), "tail": sk.launch_info(4), "full (status == NULL)": info,
                    "used": "fast + tail"}
            try:
                info["tail, capped (batches with more tail tiles than resident tail CTAs)"] = sk.launch_info(7)
            except Exception:
                pass
        return info
    info = {"plain": sk.launch_info(0)}
    try:
        info["tma"] = sk.launch_info(2)
        info["used"] = "tma" if sk.staging() else "plain"
    except Exception:
        info["used"] = "plain"
    return info


# ---- reference CPU path --------------------------------------------------------------------------------

class CpuPort(object):
    """The restated reference CPU path of one scenario (oracle/, the one place bench.py may execute it):
    ur5_track -> the hand-written FK + literal pinv of round 1 (cheaper than AD code: errs in the
    reference's favour); every other scenario -> generated expression C + literal per-mode algebra +
    mode search / dual active-set QP (oracle/clik_oracle.c, generic part)."""

    def __init__(self, scenario):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import c_port
        self.c_port, self.scenario = c_port, scenario
        if scenario.name == "ur5_track":
            import clik_oracle as orc
            from casclik_b200 import fk
            self.chain = orc.load_chain(fk.UR5_URDF, "base_link", "tool0")
            self.port = None
            self.what = "oracle/clik_oracle.c:clik_ref_pinv_track (gcc -O2 -fopenmp)"
        elif scenario.controller == "qp":
            self.port = c_port.QpPort(scenario.spec)
            self.what = "oracle/clik_oracle.c:clik_ref_qp_batch + generated expression C (gcc -O2 -fopenmp)"
        else:
            self.port = c_port.PinvPort(scenario.spec, scenario.options)
            self.what = "oracle/clik_oracle.c:clik_ref_pinv_batch + generated expression C (gcc -O2 -fopenmp)"
        self.cores = c_port.max_threads()

    def run(self, inp):
        if self.port is None:
            return self.c_port.pinv_track(self.chain, inp["q"], inp["y"], threads=self.cores)[1]
        return self.port.solve(inp, threads=self.cores)[-1]

    def measure(self, batch, seconds_target):
        """-> (cpu_baseline dict, sample size, wall seconds)"""
        n = 4096
        inp = self.scenario.sample(n, seed=0)
        self.run(inp)                                                     # warm
        t0 = time.perf_counter()
        self.run(inp)
        rate = n / max(time.perf_counter() - t0, 1e-9)
        sample = int(min(batch, max(4096, rate * seconds_target)))
        passes = max(1, int(round(rate * seconds_target / sample)))
        inp = self.scenario.sample(sample, seed=0)
        t0 = time.perf_counter()
        for _ in range(passes):
            used = self.run(inp)
        dt = time.perf_counter() - t0
        return {"value": sample * passes / dt, "unit": UNIT, "cores": int(used), "kind": "port",
                "sample": "%d passes over the first %d instances of the %d-instance batch, %.2f s wall, %s"
                          % (passes, sample, batch, dt, self.what)}, sample, dt


def run_reference(args, scenario, rank, world):
    if rank != 0:
        return
    steps, warm = max(args.steps, 1), max(args.warmup, 0)
    # bounded: every step is a sample of the batch sized so that the whole run (warm-up + K
    # steps) costs about two minutes of host time
    budget = 120.0 / (steps + min(warm, 3))
    port = CpuPort(scenario)
    base, sample, dt = port.measure(args.batch, seconds_target=budget)
    inp = scenario.sample(sample, seed=0)
    for _ in range(min(warm, 3)):
        port.run(inp)
    t0 = time.perf_counter()
    for _ in range(steps):
        port.run(inp)
    dt = time.perf_counter() - t0
    value = sample * steps / dt
    base["value"] = value
    base["sample"] = ("%d-instance sample of the %d-instance batch per step, %d steps, %.2f s wall, %s"
                      % (sample, args.batch, steps, dt, port.what))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": scenario.description, "scenario": scenario.name,
                   "batch_per_gpu": args.batch, "batch_per_step": sample,
                   "note": "reference CPU path restated in C (CasADi/qpOASES are not installable "
                           "here); host threads only, no GPU"},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_secondary:
        from casclik_b200 import scenarios
        sec = {}
        for name, batch, _, cfg in SECONDARY:
            try:
                sc = scenarios.get(name)
                b, _, _ = CpuPort(sc).measure(batch, seconds_target=6.0)
                sec[name] = {"config": cfg, "value": b["value"], "unit": UNIT, "cpu_baseline": b}
            except Exception as exc:      # the headline line must survive a broken secondary leg
                sec[name] = {"config": cfg, "error": "%s: %s" % (type(exc).__name__, exc)}
        line["secondary"] = sec
    print(json.dumps(line))


# ---- our arm ---------------------------------------------------------------------------------------------

def _launches_per_step(meta, is_qp):
    """Kernels of ours per step: QP skills with the working-set prediction run a fast + a tail launch,
    pinv skills with a run-time mode tail a fast + a group launch (both when the status / mode array is given)."""
    if is_qp:
        return 2 if (meta.get("qp_split") and os.environ.get("CLIK_QP_SPLIT", "1") != "0") else 1
    if os.environ.get("CLIK_PINV_GROUP", "0") == "1":
        return 1
    return 2 if (meta.get("pinv_split") and os.environ.get("CLIK_PINV_SPLIT", "1") != "0") else 1


def _use_staging(args, meta, is_qp, counts):
    """The staged persistent kernel pays where HBM is the nearer roof and another stream covers its ragged last
    wave (DESIGN.md §4.2b, profiles/r2_ab12.txt): roofs compared with this pool's measured peaks
    (6.55 TB/s copy bandwidth, 33.8 TFLOP/s DFMA), executed fp64 instructions from ncu when known."""
    if is_qp or not meta.get("pinv_staged_kernel") or args.staged == "off":
        return False
    if args.staged == "on":
        return True
    f64_inst = counts.get("fp64_inst_per_instance") or meta["pinv_flops_mode0"] / 2.0
    return args.streams > 1 and meta["pinv_bytes_per_step"] / 6.55e12 > 2.0 * f64_inst / 33.8e12


def _overlap_note(level, streams=1):
    note = {0: "0: plain stream order on each stream",
            1: "1: plain stream order between the steps of a stream (the two launches of a two-launch step overlap)",
            2: "2: a step kernel may start while the previous one on its stream drains (programmatic "
               "dependent launch; the steps are independent batches on disjoint buffers, completion stays in "
               "stream order)"}[level]
    if streams > 1:
        note += "; the K independent batches alternate over %d CUDA streams (forked from / joined into the " \
                "timed stream), so the drain of one step overlaps the ramp of the next" % streams
    return note + "; `stream_ordered` is the same K steps on one stream, one kernel after the other"


def _kernel_note(staged, is_qp):
    if is_qp:
        return "clik_qp_fast_kernel + clik_qp_tail_kernel (capped variant for batches with more tail tiles than resident CTAs)"
    if staged:
        return ("clik_pinv_tma_kernel: persistent balanced grid, inputs staged into shared memory by bulk async copies "
                "(cp.async.bulk + mbarrier) two tiles ahead; `stream_ordered` is the plain clik_pinv_kernel")
    return "clik_pinv_kernel: one CTA per 128 instances"


def _bytes_per_set(meta, is_qp, B):
    return (meta["qp_bytes_per_step"] if is_qp else meta["pinv_bytes_per_step"]) * B


def time_device_resident(torch, dist, ctrl, scenario, B, steps, warm, rank, world, dev, min_sets=2,
                         seed_base=1000, overlap=2, plain_too=True, n_streams=1):
    """K steps of solve_batch on device-resident inputs -> (ms total max-over-ranks, n_sets, graph?, step,
    ms of the same K steps in plain stream order | None, output buffers of the last timed step).
    Inputs and outputs rotate over enough sets to exceed L2 twice over."""
    meta = ctrl.kernel_meta
    is_qp = scenario.controller == "qp"
    per_set = _bytes_per_set(meta, is_qp, B)
    n_sets = int(max(min_sets, min(16, -(-(300 << 20) // max(per_set, 1)))))
    n_streams = max(1, int(n_streams))
    n_sets = -(-n_sets // n_streams) * n_streams      # buffer set k always travels on stream k % n_streams
    side = [torch.cuda.Stream(device=dev) for _ in range(n_streams - 1)]
    ins, outs = [], []
    for s in range(n_sets):
        inp = scenario.sample(B, seed=seed_base * (rank + 1) + s)
        ins.append(tuple(None if inp[k] is None else torch.from_numpy(np.ascontiguousarray(inp[k])).to(dev)
                         for k in ("t", "q", "x", "y")))
        if is_qp:
            outs.append((torch.empty((meta["qp_n"], B), dtype=torch.float64, device=dev),
                         torch.empty((B,), dtype=torch.int32, device=dev),
                         torch.empty((2, B), dtype=torch.int32, device=dev)))
        else:
            nq, nx = meta["n_robot"], meta["n_virtual"]
            outs.append((torch.empty((nq, B), dtype=torch.float64, device=dev),
                         torch.empty((nx, B), dtype=torch.float64, device=dev) if nx else None,
                         torch.empty((B,), dtype=torch.int32, device=dev)))

    def step(i):
        t, q, x, y = ins[i % n_sets]
        ctrl.solve_batch(t, q, x, y, out=outs[i % n_sets])

    def run_steps(k):
        """k steps; with several streams, independent batches alternate over them (fork from / join into
        the current stream, so events recorded on it bracket all of the work — also under graph capture)."""
        if not side:
            for i in range(k):
                step(i)
            return
        main = torch.cuda.current_stream()
        for st in side:
            st.wait_stream(main)
        for i in range(k):
            j = (i % n_sets) % n_streams
            if j == 0:
                step(i)
            else:
                with torch.cuda.stream(side[j - 1]):
                    step(i)
        for st in side:
            main.wait_stream(st)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(level):
        """K timed steps at overlap level `level` -> (ms max-over-ranks, replayed from a graph?)."""
        ctrl.set_overlap(level)
        run_steps(max(warm, 3))
        barrier()
        # The K timed steps are K launches of the step kernel through the C ABI.  They are captured once
        # into a CUDA graph and replayed, so that host jitter (8 ranks sharing the box's cores with the
        # clock samplers) cannot turn a 27 us kernel into a launch-bound loop; same kernels, same inputs.
        graph = None
        if os.environ.get("CLIK_BENCH_GRAPH", "1") == "1":
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    run_steps(steps)
                g.replay()                       # untimed: uploads the graph
                graph = g
            except Exception as exc:             # capture not possible: time the plain launch loop
                sys.stderr.write("bench: CUDA graph capture failed (%s); timing direct launches\n" % exc)
                graph = None
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            run_steps(steps)
        e1.record()
        barrier()
        tms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        return float(tms.item()), graph is not None

    # The K steps are K independent batches (disjoint rotating buffers).  By default they alternate over two
    # CUDA streams, so the drain of one step kernel (and the latency-bound tail pass of a QP step) overlaps
    # the ramp of the next batch; on one stream the same is available as overlap level 2 (programmatic
    # dependent launch, include/clik.h clik_skill_set_overlap).  The same K steps on one stream in plain
    # stream order are timed as well and reported next to the value (`stream_ordered`).
    ms_plain = None
    if (overlap >= 2 or side) and plain_too:
        keep, side[:] = list(side), []
        staged = bool(getattr(ctrl, "_staging", False))
        if staged:
            ctrl.set_input_staging(False)       # a single-stream caller's default: the plain kernel
        ms_plain, _ = timed(min(overlap, 1))
        if staged:
            ctrl.set_input_staging(True)
        side[:] = keep
    ms, graphed = timed(overlap)
    return ms, n_sets, graphed, step, ms_plain, outs[(steps - 1) % n_sets]


def rooflines(meta, is_qp, B, sec_per_step, hbm_peak, hbm_src, fp64_peak, counts):
    """HBM roofline from the algorithmic bytes; fp64 roofline from the EXECUTED fp64 instruction count
    (ncu, profiles/r2_ncu_counts.json) when there is one, else from the emitter's algorithmic flops
    (pinv mode 0 only).  The bound is the roof the kernel sits closer to."""
    bytes_step = meta["qp_bytes_per_step"] if is_qp else meta["pinv_bytes_per_step"]
    # DRAM bytes per launch from ncu (profiles/r2_ncu_counts.json): measured over a RANGE of launches on
    # distinct buffers when there is such a capture (the outputs of a launch leave L2 after it has ended, so a
    # per-kernel capture misses most of the writes), else the per-kernel figure
    traffic = None
    if counts.get("batch") == B and counts.get("dram_bytes") is not None:
        traffic = counts.get("dram_bytes_range_per_launch", counts["dram_bytes"])
    ach = bytes_step * B / sec_per_step / 1e9
    hbm = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
           "traffic": traffic, "peak_source": hbm_src, "algorithmic_bytes_per_step": bytes_step}
    detail = {"hbm": hbm}
    peak_src = ("measured in this run (DFMA micro-benchmark, clik_measure_fp64_peak; MEASURED_PEAKS.json "
                "has no fp64 entry)")
    if counts.get("fp64_inst_per_instance"):
        # every fp64 instruction (DFMA / DMUL / DADD / DSETP ...) occupies the pipe like one DFMA, so the
        # executed count x 2 flop-equivalents against the measured DFMA peak is the pipe's utilisation
        ach_tf = 2.0 * counts["fp64_inst_per_instance"] * B / sec_per_step / 1e12
        detail["fp64"] = {"bound": "fp64", "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                          "frac": ach_tf / fp64_peak, "traffic": traffic, "peak_source": peak_src,
                          "executed_fp64_inst_per_instance": counts["fp64_inst_per_instance"],
                          "note": "executed fp64 thread-instructions per instance from ncu "
                                  "(profiles/r2_ncu_counts.json), 2 flop-equivalents each"}
    if not is_qp:
        flops = meta["pinv_flops_mode0"]
        ach_tf = flops * B / sec_per_step / 1e12
        detail["fp64_algorithmic"] = {"bound": "fp64", "achieved": ach_tf, "peak": fp64_peak,
                                      "unit": "TFLOP/s", "frac": ach_tf / fp64_peak, "traffic": traffic,
                                      "peak_source": peak_src, "algorithmic_flops_per_step": flops,
                                      "transcendentals_per_step": meta["pinv_eval"]["transcendentals"]}
    cands = [hbm]
    if "fp64" in detail:
        cands.append(detail["fp64"])
    elif "fp64_algorithmic" in detail:
        cands.append(detail["fp64_algorithmic"])
    return max(cands, key=lambda r: r["frac"]), detail


DUMP_LIMIT = 64 * 10 ** 6     # bytes written by --dump-outputs in all


def dump_outputs(directory, arrays):
    """{name: host array (rows, N) or (N,)} -> directory/<name>.npy in float64 (int32 modes, statuses and
    active-set bit masks are exact in it).  When all N instances would exceed DUMP_LIMIT, the same fixed,
    seeded sample of instance columns is written for every array, and its indices as instances.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items() if v is not None}
    N = next(iter(arrays.values())).shape[-1]
    rows = sum(1 if a.ndim == 1 else a.shape[0] for a in arrays.values())
    if 8 * rows * N > DUMP_LIMIT:
        keep = DUMP_LIMIT // (8 * (rows + 1))
        idx = np.sort(np.random.default_rng(0).choice(N, size=keep, replace=False))
        arrays = {k: a[..., idx] for k, a in arrays.items()}
        arrays["instances"] = idx.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenario", default="ur5_track")
    ap.add_argument("--batch", type=int, default=1 << 20, help="instances per GPU per step")
    ap.add_argument("--sets", type=int, default=0, help="resident input/output sets rotated over (0 = enough for 300 MB)")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--streams", type=int, default=int(os.environ.get("CLIK_BENCH_STREAMS", "2")),
                    help="CUDA streams the K independent batches of the device-resident loop alternate over")
    ap.add_argument("--staged", default=os.environ.get("CLIK_BENCH_STAGED", "auto"), choices=["auto", "on", "off"],
                    help="pinv skills: TMA-staged persistent kernel (clik_skill_set_staging); auto = HBM-leaning "
                         "skills when the batches alternate over several streams")
    ap.add_argument("--overlap", type=int, default=int(os.environ.get("CLIK_PDL", "1")), choices=[0, 1, 2],
                    help="clik_skill_set_overlap level of the device-resident loop (2: independent steps overlap)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the other BASELINE configs")
    ap.add_argument("--secondary-only", default="", help="(profiling) run only this secondary scenario's timed loop")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    from casclik_b200 import scenarios
    scenario = scenarios.get(args.scenario)

    if args.impl == "reference":
        run_reference(args, scenario, rank, world)
        return

    import torch
    import torch.distributed as dist
    from casclik_b200 import runtime, sharding
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); "
                         "use --impl reference for the CPU baseline")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        if os.environ.get("CLIK_NUMA_BIND", "1") == "1":
            # one process per GPU: keep each rank (and the pinned host buffers of its e2e leg) on the
            # socket its GPU hangs off.  Not at N = 1, where the cpu_baseline leg wants every host core.
            numa = sharding.bind_to_device_numa_node(local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    hbm_peak, hbm_src = _peaks()
    counts_all = _ncu_counts()

    def secondary_leg(name, batch, mode, cfg, fp64_peak, with_cpu):
        sc = scenarios.get(name)
        c = sc.make_controller()
        c.setup_problem_functions()
        c.setup_solver()
        qp = sc.controller == "qp"
        staged = _use_staging(args, c.kernel_meta, qp, counts_all.get(name, {}))
        if staged:
            c.set_input_staging(True)
        if mode == "strong":
            lo, hi = sharding.shard_range(batch, rank, world)
            Bs = hi - lo
        else:
            Bs = batch
        per = _bytes_per_set(c.kernel_meta, qp, Bs)
        k = int(max(8, min(100, (3 << 30) // max(per, 1))))          # ~3 GB of algorithmic traffic per leg
        ms_tot, n_sets, graphed, _, ms_plain, _ = time_device_resident(torch, dist, c, sc, Bs, k, 3, rank, world, dev,
                                                                       seed_base=2000, overlap=args.overlap,
                                                                       n_streams=args.streams)
        total = batch if mode == "strong" else batch * world
        val = total * k / (ms_tot * 1e-3)
        out = {"config": cfg, "workload": sc.description, "value": val, "unit": UNIT,
               "ms_per_step": ms_tot / k, "steps": k, "batch_per_gpu": Bs, "global_batch": total,
               "scaling": mode, "sets_rotated": n_sets, "overlap": _overlap_note(args.overlap, args.streams), "streams": args.streams,
               "kernel": _kernel_note(staged, qp),
               "gpu_launches": k * _launches_per_step(c.kernel_meta, qp)}
        if ms_plain is not None:
            out["stream_ordered"] = {"value": total * k / (ms_plain * 1e-3), "ms_per_step": ms_plain / k}
        if rank == 0:
            roof, detail = rooflines(c.kernel_meta, qp, Bs, ms_tot * 1e-3 / k, hbm_peak, hbm_src, fp64_peak,
                                     counts_all.get(name, {}))
            out["roofline"], out["roofline_detail"] = roof, detail
            out["launch"] = _launch_info(c, qp)
            if with_cpu:
                out["cpu_baseline"], _, _ = CpuPort(sc).measure(batch, seconds_target=6.0)
        return out

    if args.secondary_only:
        for name, batch, mode, cfg in SECONDARY:
            if name == args.secondary_only:
                print(json.dumps(secondary_leg(name, batch, mode, cfg, 1.0, False)))
        return

    ctrl = scenario.make_controller()
    ctrl.setup_problem_functions()
    ctrl.setup_solver()
    meta = ctrl.kernel_meta
    is_qp = scenario.controller == "qp"
    staged = _use_staging(args, meta, is_qp, counts_all.get(scenario.name, {}))
    if staged:
        ctrl.set_input_staging(True)
    B = args.batch
    # every rank owns an independent shard (weak scaling: B instances per GPU); no collective
    # on the data path — instances are independent (SURVEY.md §8e)
    sampler = ClockSampler(local)
    sampler.start()
    ms, n_sets, graphed, step, ms_plain, last = time_device_resident(
        torch, dist, ctrl, scenario, B, args.steps, args.warmup, rank, world, dev, min_sets=max(args.sets, 2),
        overlap=args.overlap, n_streams=args.streams)
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # now, before the e2e loop and the untimed load steps below reuse the step buffers
        names = ("sol", "status", "active") if is_qp else ("robot_vel", "virtual_vel", "mode")
        dump_outputs(args.dump_outputs, {k: None if a is None else a.cpu().numpy() for k, a in zip(names, last)})

    # ---- end to end through the host-buffer C ABI (pinned host inputs, copies inside) --------------
    inp = scenario.sample(B, seed=1000 * rank + 77)
    pin = {k: (None if inp[k] is None else torch.from_numpy(np.ascontiguousarray(inp[k])).pin_memory())
           for k in ("t", "q", "x", "y")}
    host = {k: (None if v is None else v.numpy()) for k, v in pin.items()}
    if is_qp:
        hout = (torch.empty((meta["qp_n"], B), dtype=torch.float64).pin_memory().numpy(),
                torch.empty((B,), dtype=torch.int32).pin_memory().numpy(),
                torch.empty((2, B), dtype=torch.int32).pin_memory().numpy())
        d2h = B * (8 * meta["qp_n"] + 4 + 8)
    else:
        hout = (torch.empty((meta["n_robot"], B), dtype=torch.float64).pin_memory().numpy(),
                torch.empty((meta["n_virtual"], B), dtype=torch.float64).pin_memory().numpy()
                if meta["n_virtual"] else None,
                torch.empty((B,), dtype=torch.int32).pin_memory().numpy())
        d2h = B * (8 * (meta["n_robot"] + meta["n_virtual"]) + 4)
    # the host ABI copies only the input rows the compiled kernel reads (read masks in the cubin)
    mk = meta["qp_read_masks" if is_qp else "pinv_read_masks"]
    rows_in = (mk[0] if host["t"].size > 1 else 0)
    for mask, key in ((mk[1], "q"), (mk[2], "x"), (mk[3], "y")):
        if host[key] is not None:
            rows_in += bin(mask & ((1 << host[key].shape[0]) - 1)).count("1")
    h2d = 8 * B * rows_in + (8 if (mk[0] and host["t"].size == 1) else 0)

    def e2e_step():
        ctrl.solve_batch(host["t"], host["q"], host["x"], host["y"], out=hout)

    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()          # synchronous: returns when the results are in host memory
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tdt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.e2e_steps / float(tdt.item())
    # keep the GPU under load until the sampler has a few readings (the timed region itself can
    # be only milliseconds long); these extra steps are outside every timed region
    t_load = time.perf_counter()
    while len(sampler.rows) < 4 and time.perf_counter() - t_load < 3.0:
        for i in range(200):
            step(i)
        torch.cuda.synchronize()
    clocks = sampler.summary()
    clocks["note"] = ("sampled every 100 ms from warm-up to the end of the e2e loop (plus up to 3 s "
                      "of extra untimed steps when the run is too short for 4 samples)")

    fp64_peak = runtime.measure_fp64_peak(local) if rank == 0 else 0.0
    line = None
    if rank == 0:
        sec = ms * 1e-3 / args.steps
        roof, detail = rooflines(meta, is_qp, B, sec, hbm_peak, hbm_src, fp64_peak,
                                 counts_all.get(scenario.name, {}))
        bytes_step = meta["qp_bytes_per_step"] if is_qp else meta["pinv_bytes_per_step"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": scenario.description, "scenario": scenario.name,
                       "batch_per_gpu": B, "global_batch": B * world,
                       "parallelism": "independent shards, one per GPU, no collective on the data path",
                       "launch_mode": ("%d step-kernel launches replayed from one CUDA graph" % args.steps
                                       if graphed else "direct launches"),
                       "overlap": _overlap_note(args.overlap, args.streams), "streams": args.streams,
                       "kernel": _kernel_note(staged, is_qp),
                       "host_affinity": ("rank 0 bound to its GPU's NUMA node: %d of %d CPUs" % (len(numa[1]), len(numa[0]))
                                         if numa else "unbound"),
                       "l2": "rotating %d resident input + output sets (%d MB of algorithmic traffic in total) "
                             "> 126 MB L2" % (n_sets, n_sets * bytes_step * B // (1 << 20)),
                       "launch": _launch_info(ctrl, is_qp)},
            "roofline": {k: v for k, v in roof.items()},
            "roofline_detail": detail,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
                    "path": "solve_batch(host arrays) -> clik_*_step_host with pinned host buffers: the "
                            "kernel reads inputs from / writes results to mapped host memory over PCIe "
                            "inside the timed region (pageable buffers would take the chunked H2D / "
                            "kernel / D2H pipeline instead)"},
            "gpu_launches": args.steps * _launches_per_step(meta, is_qp),
            "clocks": clocks,
        }
        if ms_plain is not None:
            # the same K steps with every step kernel waiting for the previous one to finish (overlap level 1)
            line["stream_ordered"] = {"value": world * B * args.steps / (ms_plain * 1e-3), "unit": UNIT,
                                      "ms_per_step": ms_plain / args.steps}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"], _, _ = CpuPort(scenario).measure(B, seconds_target=12.0)
    del step, last
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, same run, same timing rules ---------------------------------------
    if not args.no_secondary:
        secondary = {}
        for name, batch, mode, cfg in SECONDARY:
            if name == scenario.name:
                continue
            try:
                secondary[name] = secondary_leg(name, batch, mode, cfg, fp64_peak,
                                                with_cpu=(world == 1 and not args.no_cpu_baseline))
            except Exception as exc:          # the headline line must survive a broken secondary leg
                secondary[name] = {"config": cfg, "error": "%s: %s" % (type(exc).__name__, exc)}
                if world > 1:
                    raise
            torch.cuda.empty_cache()
        if line is not None:
            line["secondary"] = secondary
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
