"""Throughput of the ReactiveNLPController step (scenarios.NLP_REGISTRY) on one GPU, device-resident.

    python tools/nlp_bench.py [--batch 262144] [--reps 20] [--warmup 3] [--out profiles/nlp_bench.json]

Per scenario: CUDA-event time of solve_batch on torch tensors, with the inputs rotated over several
independent sets whose total exceeds L2 and the L2 flushed before every timed launch (runtime.flush_l2);
mean / max SQP iterations and the status histogram of the timed batches; and, for comparison, the same
kernel source compiled for the host CPU (g++ -O2, OpenMP over all cores, one instance per loop iteration).
The card name and power limit are read in the same run (nvidia-smi --query-gpu=name,power.limit, read-only).
The only published figure of the reference's step is 2.9-3.3 ms per instance (IPOPT, BASELINE.md §1)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

OMP_DRIVER = r'''
#include <omp.h>
extern "C" void run_omp(long long N, const double* t, const double* q, const double* x, const double* y,
                        double* sol, int* status, int* iters, unsigned* active, int max_iter, int chunk) {
  const long long nchunks = (N + chunk - 1) / chunk;
#pragma omp parallel for schedule(dynamic)
  for (long long c = 0; c < nchunks; ++c) {
    const long long lo = c * chunk, cnt = (lo + chunk <= N) ? chunk : N - lo;
    clik_nlp_kernel(cnt, N, t + lo, 1, q + lo, x ? x + lo : nullptr, y ? y + lo : nullptr, nullptr, sol + lo,
                    status + lo, iters + lo, active + lo, max_iter);
  }
}
'''


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout
        return out.strip().splitlines()[0]
    except Exception as exc:  # noqa: BLE001
        return "unavailable (%s)" % exc


def host_figure(ctrl, inp, max_iter):
    from test_kernel_code_on_host import SHIM
    text = ctrl.kernel_source.replace("__device__ const unsigned short", "static const unsigned short")
    with tempfile.TemporaryDirectory() as d:
        src, so = os.path.join(d, "nlp.cpp"), os.path.join(d, "nlp.so")
        with open(src, "w") as f:
            f.write(SHIM + text + OMP_DRIVER)
        subprocess.run(["g++", "-O2", "-fopenmp", "-std=c++17", "-shared", "-fPIC", "-I",
                        os.path.join(ROOT, "casclik_b200", "csrc"), "-o", so, src], check=True)
        lib = ctypes.CDLL(so)
        N = inp["q"].shape[1]
        p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        c = {k: (None if v is None else np.ascontiguousarray(v)) for k, v in inp.items()}
        sol = np.empty((ctrl._qn, N))
        st, it = np.empty(N, dtype=np.int32), np.empty(N, dtype=np.int32)
        act = np.empty((2, N), dtype=np.uint32)
        args = (ctypes.c_longlong(N), p(c["t"]), p(c["q"]), p(c.get("x")), p(c.get("y")), p(sol), p(st), p(it),
                p(act), ctypes.c_int(max_iter), ctypes.c_int(64))
        lib.run_omp(*args)                       # warm-up
        t0 = time.perf_counter()
        lib.run_omp(*args)
        dt = time.perf_counter() - t0
    return {"steps_per_s": N / dt, "batch": N, "threads": os.cpu_count(),
            "status_hist": np.bincount(st, minlength=6).tolist()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sets", type=int, default=4)
    ap.add_argument("--host-batch", type=int, default=1 << 15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "nlp_bench.json"))
    args = ap.parse_args()
    import torch
    from casclik_b200 import runtime, scenarios
    dev = torch.device("cuda", 0)
    rec = {"gpu": gpu_info(), "batch": args.batch, "reps": args.reps, "warmup": args.warmup,
           "reference_published": "2.9-3.3 ms per step, one instance (IPOPT; BASELINE.md §1)", "scenarios": {}}
    for name in sorted(scenarios.NLP_REGISTRY):
        sc = scenarios.get(name)
        ctrl = sc.make_controller()
        ctrl.setup_solver()
        sets = []
        for s in range(args.sets):
            inp = sc.sample(args.batch, seed=s)
            sets.append({k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).to(dev))
                         for k, v in inp.items()})
        out = ctrl.solve_batch(sets[0]["t"], sets[0]["q"], None, sets[0]["y"])
        for k in range(args.warmup):
            s = sets[k % args.sets]
            ctrl.solve_batch(s["t"], s["q"], None, s["y"], out=out)
        torch.cuda.synchronize()
        times, hist, it_sum, it_max = [], np.zeros(6, dtype=np.int64), 0, 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(args.reps):
            s = sets[k % args.sets]
            runtime.flush_l2(0, torch.cuda.current_stream().cuda_stream)
            e0.record()
            ctrl.solve_batch(s["t"], s["q"], None, s["y"], out=out)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) * 1e-3)
            st, it = out[1].cpu().numpy(), out[3].cpu().numpy()
            hist += np.bincount(st, minlength=6)[:6]
            it_sum += int(it.sum())
            it_max = max(it_max, int(it.max()))
        med = float(np.median(times))
        host = host_figure(ctrl, sc.sample(args.host_batch, seed=99), int(ctrl.options["max_iter"]))
        rec["scenarios"][name] = {
            "description": sc.description,
            "steps_per_s": args.batch / med, "median_s": med, "min_s": float(np.min(times)),
            "max_s": float(np.max(times)),
            "sqp_iterations_mean": it_sum / (args.reps * args.batch), "sqp_iterations_max": it_max,
            "status_hist": hist.tolist(),
            "quadratic": ctrl.kernel_meta["nlp_quadratic"], "hoisted_values": ctrl.kernel_meta["nlp_hoisted"],
            "kernel_source_on_the_host_cpu": host,
        }
        print(name, json.dumps(rec["scenarios"][name]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
