#!/usr/bin/env python
"""One process, one host batch of the NLP controller, k GPUs: ReactiveNLPController.solve_batch(host arrays,
devices=k) timed end to end (host arrays in, results in host memory when the call returns) for k = 1, 2, 4, ...
up to the visible GPU count, for both scenarios.NLP_REGISTRY scenarios, with pageable arrays (chunked H2D / kernel
/ D2H pipeline per device) and with page-locked ones (zero-copy kernel per device), each result checked bit for
bit against k = 1.

    python tools/nlp_multi_gpu.py [--per-gpu-log2 18] [--reps 10] [--out profiles/nlp_multi_gpu.json]

The global batch is fixed (strong scaling): 2^per-gpu-log2 instances times the largest k, so every device
gets at least 2^per-gpu-log2 instances.  Times are a host clock around the synchronous call; the figure is the
median over --reps calls after two warm-up calls.  Host bytes per instance are those the kernel reads (the
input rows of its read masks) plus those it writes (sol, status, iterations, two mask words).  The card names
and power limits are read in the same run (nvidia-smi --query-gpu=index,name,power.limit, read-only).  On a box
with one GPU only k = 1 is measured, and the JSON says so."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout
        return out.strip().splitlines()
    except Exception as exc:  # noqa: BLE001
        return ["unavailable (%s)" % exc]


def device_counts(ndev):
    ks, k = [], 1
    while k <= ndev:
        ks.append(k)
        k *= 2
    if ks[-1] != ndev:
        ks.append(ndev)
    return ks


def host_bytes(ctrl):
    masks = ctrl.kernel_meta["nlp_read_masks"]
    rows_in = sum(bin(m).count("1") for m in masks)
    return 8 * rows_in, 8 * ctrl._qn + 4 + 4 + 2 * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-gpu-log2", type=int, default=18)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "nlp_multi_gpu.json"))
    args = ap.parse_args()
    import torch
    from casclik_b200 import scenarios
    ndev = torch.cuda.device_count()
    if ndev < 1:
        sys.exit("nlp_multi_gpu.py needs a CUDA device")
    ks = device_counts(ndev)
    N = (1 << args.per_gpu_log2) * ks[-1]
    pin = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    rec = {"gpu": gpu_info(), "gpus_visible": ndev, "device_counts_measured": ks, "global_batch": N,
           "min_instances_per_gpu": N // ks[-1], "reps": args.reps, "timing": "host clock around the synchronous "
           "call, median of reps after 2 warm-up calls", "rows": []}
    if ndev == 1:
        rec["note"] = "one GPU visible: only k = 1 was measured; multi-GPU scaling was not measured"
    for name in sorted(scenarios.NLP_REGISTRY):
        sc = scenarios.get(name)
        ctrl = sc.make_controller()
        ctrl.setup_solver()
        b_in, b_out = host_bytes(ctrl)
        inp = sc.sample(N, seed=5)
        for memory in ("pageable", "pinned"):
            conv = pin if memory == "pinned" else (lambda a: None if a is None else np.ascontiguousarray(a))
            t, q, y = conv(inp["t"]), conv(inp["q"]), conv(inp["y"])
            out = (conv(np.empty((ctrl._qn, N))), conv(np.empty(N, dtype=np.int32)),
                   conv(np.empty((2, N), dtype=np.int32)), conv(np.empty(N, dtype=np.int32)))
            ref = None
            for k in ks:
                for _ in range(2):
                    ctrl.solve_batch(t, q, None, y, out=out, devices=k)
                times = []
                for _ in range(args.reps):
                    t0 = time.perf_counter()
                    ctrl.solve_batch(t, q, None, y, out=out, devices=k)
                    times.append(time.perf_counter() - t0)
                if ref is None:
                    ref = tuple(a.copy() for a in out)
                same = all(np.array_equal(a, b) for a, b in zip(out, ref))
                med = float(np.median(times))
                row = {"scenario": name, "host_memory": memory, "gpus": k, "global_batch": N,
                       "e2e_steps_per_s": N / med, "median_s": med, "min_s": float(np.min(times)),
                       "max_s": float(np.max(times)), "host_bytes_per_instance": {"in": b_in, "out": b_out},
                       "host_GB_per_s": N / med * (b_in + b_out) / 1e9,
                       "status_hist": np.bincount(out[1], minlength=6).tolist(), "bit_identical_to_1gpu": bool(same)}
                rec["rows"].append(row)
                print("%-18s %-8s %d GPU(s): %.3e steps/s  %.1f GB/s host traffic  (%.2f ms per call)  identical to "
                      "1 GPU: %s" % (name, memory, k, row["e2e_steps_per_s"], row["host_GB_per_s"], 1e3 * med, same),
                      flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
