"""Cost of the step's forward-mode derivative and Jacobian next to the step and its VJP, on one GPU, device-resident.

    python tools/jvp_bench.py [--batch 262144] [--reps 20] [--warmup 3] [--out profiles/jvp_bench.json]

Per scenario (ur5_qp, ur5_moe2016_qp, ur5_nlp_taskspeed, ur5_nlp_quartic): the CUDA-event time of solve_batch,
vjp_batch (cotangent all ones), jvp_batch (random tangent), jacobian_batch, n_theta jvp_batch launches with unit
tangents (the Jacobian column by column) and n_x vjp_batch launches with unit cotangents (row by row); each timed call
is preceded by an L2 flush (runtime.flush_l2), median of `reps` timed calls after `warmup` untimed ones, as
tools/vjp_bench.py.  The record says whether the one-factorisation Jacobian kernel beats the n_theta JVP launches on
every scenario.  The card name and power limit are read in the same run (nvidia-smi --query-gpu=name,power.limit,
read-only)."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SCENARIOS = ("ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "jvp_bench.json"))
    args = ap.parse_args()
    import torch
    from casclik_b200 import runtime, scenarios
    from nlp_bench import gpu_info
    dev = torch.device("cuda", 0)
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    rec = {"gpu": gpu_info(), "batch": args.batch, "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events around one call (or loop of calls), L2 flushed before each timed call, median",
           "scenarios": {}}
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
        inp = {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).to(dev))
               for k, v in sc.sample(args.batch, seed=0).items()}
        t, q, y = inp["t"], inp["q"], inp["y"]
        N, nq, ny = args.batch, q.shape[0], ctrl._ny
        nt = 1 + nq + ctrl._nxv + ny
        out = ctrl.solve_batch(t, q, None, y)
        step = timed(lambda: ctrl.solve_batch(t, q, None, y, out=out))
        sol, status, active = out[0], out[1], out[2]
        sb = torch.ones_like(sol)
        vo = ctrl.vjp_batch(t, q, None, y, sol, status, active, sb)
        vjp = timed(lambda: ctrl.vjp_batch(t, q, None, y, sol, status, active, sb, out=vo))
        g = torch.Generator("cuda").manual_seed(1)
        td = torch.randn((N,), dtype=torch.float64, device=dev, generator=g)
        qd = torch.randn(q.shape, dtype=torch.float64, device=dev, generator=g)
        yd = torch.randn(y.shape, dtype=torch.float64, device=dev, generator=g) if ny else None
        jo = ctrl.jvp_batch(t, q, None, y, sol, status, active, td, qd, None, yd)
        jvp = timed(lambda: ctrl.jvp_batch(t, q, None, y, sol, status, active, td, qd, None, yd, out=jo))
        jac = ctrl.jacobian_batch(t, q, None, y, sol, status, active)
        jacobian = timed(lambda: ctrl.jacobian_batch(t, q, None, y, sol, status, active, out=jac))
        # unit tangents, one per theta entry (t, q, y; the ur5 scenarios have no virtual variables)
        units = []
        for c in range(nt):
            tu, qu = torch.zeros(N, dtype=torch.float64, device=dev), torch.zeros_like(q)
            yu = torch.zeros_like(y) if ny else None
            if c == 0:
                tu += 1.0
            elif c <= nq:
                qu[c - 1] = 1.0
            else:
                yu[c - 1 - nq] = 1.0
            units.append((tu, qu, yu))
        cols = [torch.empty_like(sol) for _ in range(nt)]

        def jvp_loop():
            for (tu, qu, yu), o in zip(units, cols):
                ctrl.jvp_batch(t, q, None, y, sol, status, active, tu, qu, None, yu, out=o)
        loop_jvp = timed(jvp_loop)
        cots = []
        for j in range(ctrl._qn):
            e = torch.zeros_like(sol)
            e[j] = 1.0
            cots.append(e)
        vouts = [[a.clone() if a is not None else None for a in vo] for _ in range(ctrl._qn)]

        def vjp_loop():
            for e, o in zip(cots, vouts):
                ctrl.vjp_batch(t, q, None, y, sol, status, active, e, out=o)
        loop_vjp = timed(vjp_loop)
        jvp_loop()
        torch.cuda.synchronize()
        stacked = torch.stack(cols, dim=1)
        fin = torch.isfinite(jac).all(dim=0).all(dim=0)
        dev_rel = float(((jac - stacked).abs().amax(dim=(0, 1)) / (1 + stacked.abs().amax(dim=(0, 1))))[fin].max())
        st = status.cpu().numpy()
        rec["scenarios"][name] = {
            "rows": ctrl._qm, "variables": ctrl._qn, "n_theta": nt,
            "solve_batch_median_s": step[0], "solve_batch_min_max_s": step[1:],
            "vjp_batch_median_s": vjp[0], "vjp_batch_min_max_s": vjp[1:],
            "jvp_batch_median_s": jvp[0], "jvp_batch_min_max_s": jvp[1:],
            "jacobian_batch_median_s": jacobian[0], "jacobian_batch_min_max_s": jacobian[1:],
            "n_theta_jvp_launches_median_s": loop_jvp[0], "n_theta_jvp_launches_min_max_s": loop_jvp[1:],
            "n_x_vjp_launches_median_s": loop_vjp[0], "n_x_vjp_launches_min_max_s": loop_vjp[1:],
            "jacobian_over_jvp_launches": jacobian[0] / loop_jvp[0],
            "jacobian_vs_unit_jvp_max_rel_dev": dev_rel,
            "status_hist": np.bincount(st, minlength=6).tolist(),
            "solved_with_finite_jacobian": int(fin.sum()),
        }
        print(name, json.dumps(rec["scenarios"][name]), flush=True)
    rec["jacobian_kernel_beats_jvp_launches_everywhere"] = all(
        s["jacobian_batch_median_s"] < s["n_theta_jvp_launches_median_s"] for s in rec["scenarios"].values())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
