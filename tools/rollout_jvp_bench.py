"""Cost of the fused tangent and Jacobian rollouts next to rollout_batch and the composed Python loops, on one GPU.

    python tools/rollout_jvp_bench.py [--batch 262144] [--steps 50] [--reps 10] [--warmup 2]
                                      [--out profiles/rollout_jvp_bench.json]

Per scenario (ur5_qp, ur5_moe2016_qp, ur5_nlp_taskspeed, ur5_nlp_quartic), CUDA-event time, median of `reps` timed
calls after `warmup` untimed ones, L2 flushed before each timed call (runtime.flush_l2), of:
  - rollout_batch (K steps);
  - rollout_jvp (random tangent of (t0, q0, y)) and rollout_jacobian;
  - the composed loops: K x (solve_batch(warm_active=...) / solve_batch(warmstart=...) + jvp_batch + clip mask + Euler)
    and K x (solve_batch + jacobian_batch + the chain rule as a batched matrix product + mask + Euler).
Every timed call starts from the same initial state (copied before the timed window).  The record also holds the
largest deviation of the fused tangent / Jacobian from the composed loops, and ptxas registers, stack frame and
spills of the new kernels (read from the compile log).  The card name and power limit are read in the same run
(nvidia-smi --query-gpu=name,power.limit, read-only)."""
import argparse
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SCENARIOS = ("ur5_qp", "ur5_moe2016_qp", "ur5_nlp_taskspeed", "ur5_nlp_quartic")


def ptxas(log_path, kernel):
    """(registers, stack frame bytes, spill stores, spill loads) of `kernel` from an nvcc -Xptxas=-v log."""
    text = open(log_path).read()
    i = text.find("Compiling entry function '%s'" % kernel)
    if i < 0:
        return None
    block = text[i:i + 600]
    regs = re.search(r"Used (\d+) registers", block)
    frame = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
    return {"registers": int(regs.group(1)), "stack_frame_bytes": int(frame.group(1)),
            "spill_store_bytes": int(frame.group(2)), "spill_load_bytes": int(frame.group(3))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 18)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rollout_jvp_bench.json"))
    args = ap.parse_args()
    import torch
    from casclik_b200 import runtime, scenarios
    from nlp_bench import gpu_info
    dev = torch.device("cuda", 0)
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    K, dt, N = args.steps, 0.008, args.batch
    rec = {"gpu": gpu_info(), "batch": N, "steps": K, "dt": dt, "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events around one call (or one composed loop), L2 flushed before each timed call, median",
           "scenarios": {}}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reset):
        for _ in range(args.warmup):
            reset()
            fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            reset()
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
        kind = "qp" if name.endswith("_qp") else "nlp"
        inp = {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).to(dev))
               for k, v in sc.sample(N, seed=0).items()}
        t, q0, y = inp["t"], inp["q"], inp["y"]
        nq, ny, ns = q0.shape[0], ctrl._ny, q0.shape[0] + ctrl._nxv
        nt = 1 + ns + ny
        vq = 0.7 * float(ctrl.solve_batch(t, q0, None, y)[0][:nq].abs().amax())
        q = q0.clone()

        def reset():
            q.copy_(q0)
        g = torch.Generator("cuda").manual_seed(1)
        td = torch.randn((N,), dtype=torch.float64, device=dev, generator=g)
        qd = torch.randn(q0.shape, dtype=torch.float64, device=dev, generator=g)
        yd = torch.randn(y.shape, dtype=torch.float64, device=dev, generator=g) if ny else None
        res = {}
        plain = timed(lambda: res.__setitem__("r", ctrl.rollout_batch(t, q, K, dt, None, y, max_speed=vq)), reset)
        fused_jvp = timed(lambda: res.__setitem__("j", ctrl.rollout_jvp(t, q, K, dt, None, y, max_speed=vq,
                                                                        t_dot=td, q_dot=qd, y_dot=yd)), reset)
        fused_jac = timed(lambda: res.__setitem__("J", ctrl.rollout_jacobian(t, q, K, dt, None, y, max_speed=vq)),
                          reset)
        tangent = [td, qd, None, yd]

        def composed(jacobian):
            warm_a = torch.zeros((2, N), dtype=torch.int32, device=dev)
            warm_x = torch.zeros((ctrl._qn, N), dtype=torch.float64, device=dev)
            tq = qd.clone()
            P = torch.zeros((ns, nt, N), dtype=torch.float64, device=dev)
            for a in range(ns):
                P[a, 1 + a] = 1.0
            T = torch.zeros((nt, nt, N), dtype=torch.float64, device=dev)
            T[0, 0] = 1.0
            for c in range(1 + ns, nt):
                T[c, c] = 1.0
            for k in range(K):
                tk = t + dt * float(k)
                if kind == "qp":
                    sol, status, active = ctrl.solve_batch(tk, q, None, y, warm_active=warm_a)
                else:
                    sol, status, active, _ = ctrl.solve_batch(tk, q, None, y, warmstart=warm_x)
                keep = sol[:ns].abs() < vq
                if jacobian:
                    J = ctrl.jacobian_batch(tk, q, None, y, sol, status, active)[:ns]
                    T[1:1 + ns] = P
                    step = torch.bmm(J.permute(2, 0, 1), T.permute(2, 0, 1)).permute(1, 2, 0)
                    P = P + dt * torch.where(keep[:, None], step, 0.0)
                else:
                    sd = ctrl.jvp_batch(tk, q, None, y, sol, status, active, td, tq, None, yd)
                    tq = tq + torch.where(keep, sd[:ns], 0.0) * dt
                v = torch.where(status == 0, sol, 0.0)
                warm_a, warm_x = active, v
                q.add_(v[:nq].clamp(-vq, vq) * dt)
            res["c"] = P if jacobian else tq
        loop_jvp = timed(lambda: composed(False), reset)
        tq_ref = res["c"]
        loop_jac = timed(lambda: composed(True), reset)
        P_ref = res["c"]
        bad = torch.isnan(res["j"]["q_dot"]).any(dim=0)
        dev_jvp = float(((res["j"]["q_dot"] - tq_ref).abs().amax(dim=0) / (1 + tq_ref.abs().amax(dim=0)))[~bad].max())
        jb = torch.isnan(res["J"]["jac"]).any(dim=0).any(dim=0)
        dev_jac = float(((res["J"]["jac"] - P_ref).abs().amax(dim=(0, 1)) /
                         (1 + P_ref.abs().amax(dim=(0, 1))))[~jb].max())
        log = ctrl._rollout_jvp["path"][:-len(".cubin")] + ".log"
        rec["scenarios"][name] = {
            "rows": ctrl._qm, "variables": ctrl._qn, "n_theta": nt, "max_speed": vq,
            "rollout_batch_median_s": plain[0], "rollout_batch_min_max_s": plain[1:],
            "rollout_jvp_median_s": fused_jvp[0], "rollout_jvp_min_max_s": fused_jvp[1:],
            "rollout_jacobian_median_s": fused_jac[0], "rollout_jacobian_min_max_s": fused_jac[1:],
            "composed_jvp_loop_median_s": loop_jvp[0], "composed_jvp_loop_min_max_s": loop_jvp[1:],
            "composed_jacobian_loop_median_s": loop_jac[0], "composed_jacobian_loop_min_max_s": loop_jac[1:],
            "fused_jvp_speedup_over_composed": loop_jvp[0] / fused_jvp[0],
            "fused_jacobian_speedup_over_composed": loop_jac[0] / fused_jac[0],
            "fused_vs_composed_max_rel_dev": {"q_dot": dev_jvp, "jac": dev_jac},
            "nan_instances": {"rollout_jvp": int(bad.sum()), "rollout_jacobian": int(jb.sum())},
            "n_failed_total": int(res["r"]["n_failed"].sum()),
            "ptxas": {k: ptxas(log, "clik_%s_rollout_%s_kernel" % (kind, k)) for k in ("jvp", "jacobian")},
        }
        print(name, json.dumps(rec["scenarios"][name]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
