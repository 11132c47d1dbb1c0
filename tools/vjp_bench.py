"""Cost of the step's reverse-mode derivative next to the step and its multipliers, on one GPU, device-resident.

    python tools/vjp_bench.py [--batch 262144] [--reps 20] [--warmup 3] [--out profiles/vjp_bench.json]

Per scenario (ur5_qp, ur5_moe2016_qp, ur5_nlp_taskspeed, ur5_nlp_quartic): the CUDA-event time of solve_batch,
multipliers_batch and vjp_batch alone (on that step's output, cotangent all ones), and of the forward + backward()
of a summed loss through solve_batch_differentiable; each timed call is preceded by an L2 flush (runtime.flush_l2),
median of `reps` timed calls after `warmup` untimed ones.  Also the cold host compile time of the VJP image
(emit + nvcc into an empty cache directory).  The card name and power limit are read in the same run
(nvidia-smi --query-gpu=name,power.limit, read-only)."""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SCENARIOS = ("ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic")


def cold_compile_seconds(ctrl):
    from casclik_b200 import build
    saved = build.CACHE_DIR
    with tempfile.TemporaryDirectory() as d:
        build.CACHE_DIR = d
        try:
            t0 = time.perf_counter()
            source, _ = ctrl._vjp_source()
            build.compile_cubin(source, tag="vjp_cold")
            return time.perf_counter() - t0
        finally:
            build.CACHE_DIR = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "vjp_bench.json"))
    args = ap.parse_args()
    import torch
    from casclik_b200 import runtime, scenarios
    from nlp_bench import gpu_info
    dev = torch.device("cuda", 0)
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    rec = {"gpu": gpu_info(), "batch": args.batch, "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events around one call, L2 flushed before each timed call, median", "scenarios": {}}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            runtime.flush_l2(0, stream())
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) * 1e-3)
        return float(np.median(times)), float(np.min(times)), float(np.max(times))

    for name in SCENARIOS:
        sc = scenarios.get(name)
        ctrl = sc.make_controller()
        ctrl.setup_solver()
        compile_s = cold_compile_seconds(ctrl)
        inp = {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).to(dev))
               for k, v in sc.sample(args.batch, seed=0).items()}
        t, q, y = inp["t"], inp["q"], inp["y"]
        out = ctrl.solve_batch(t, q, None, y)
        step = timed(lambda: ctrl.solve_batch(t, q, None, y, out=out))
        sol, status, active = out[0], out[1], out[2]
        lam = ctrl.multipliers_batch(t, q, None, y, sol, status, active)
        duals = timed(lambda: ctrl.multipliers_batch(t, q, None, y, sol, status, active, out=lam))
        sb = torch.ones_like(sol)
        vo = ctrl.vjp_batch(t, q, None, y, sol, status, active, sb)
        vjp = timed(lambda: ctrl.vjp_batch(t, q, None, y, sol, status, active, sb, out=vo))
        qg = q.clone().requires_grad_(True)

        def fwd_bwd():
            qg.grad = None
            ctrl.solve_batch_differentiable(t, qg, None, y)[0].sum().backward()
        both = timed(fwd_bwd)
        st = status.cpu().numpy()
        solved = st == 0
        qb = vo[1].cpu().numpy()
        rec["scenarios"][name] = {
            "rows": ctrl._qm, "variables": ctrl._qn,
            "solve_batch_median_s": step[0], "solve_batch_min_max_s": step[1:],
            "multipliers_batch_median_s": duals[0], "multipliers_batch_min_max_s": duals[1:],
            "vjp_batch_median_s": vjp[0], "vjp_batch_min_max_s": vjp[1:],
            "forward_backward_median_s": both[0], "forward_backward_min_max_s": both[1:],
            "vjp_over_step": vjp[0] / step[0],
            "vjp_image_cold_compile_s": compile_s,
            "status_hist": np.bincount(st, minlength=6).tolist(),
            "solved_with_finite_q_bar": int(np.isfinite(qb[:, solved]).all(axis=0).sum()),
        }
        print(name, json.dumps(rec["scenarios"][name]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
