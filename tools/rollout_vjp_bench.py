"""Cost of the taped rollout and its reverse sweep next to rollout_batch, autograd, the composed Python loop and the
Jacobian rollout, on one GPU.

    python tools/rollout_vjp_bench.py [--batch 262144] [--steps 50] [--reps 10] [--warmup 2]
                                      [--out profiles/rollout_vjp_bench.json]

Per scenario (ur5_qp, ur5_moe2016_qp, ur5_nlp_taskspeed, ur5_nlp_quartic), CUDA-event time, median of `reps` timed
calls after `warmup` untimed ones, L2 flushed before each timed call (runtime.flush_l2), dt = 0.008 and max_speed at
0.7 times the largest first-step robot speed, of:
  - rollout_batch (K steps);
  - the taped rollout (clik_<kind>_rollout_tape) alone, and the reverse sweep (clik_<kind>_rollout_vjp) alone over
    its tape;
  - rollout_batch_differentiable forward + loss.backward() for the loss <c_q, q_K> + <c_s, sol>;
  - the composed loop: K vjp_batch launches over the tape slices, with the clip mask and the accumulation in torch;
  - rollout_jacobian + the contraction with the same cotangent, which gives the same gradient.
Every timed call starts from the same initial state.  The record also holds the largest deviation of the sweep from
the composed loop and from the Jacobian contraction, the tape size, and ptxas registers, stack frame and spills of
the two new kernels (read from the compile log).  The card name and power limit are read in the same run
(nvidia-smi --query-gpu=name,power.limit, read-only)."""
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
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rollout_vjp_bench.json"))
    args = ap.parse_args()
    import torch
    from casclik_b200 import runtime, scenarios
    from casclik_b200.controllers import base_controller as bc
    from nlp_bench import gpu_info
    from rollout_jvp_bench import ptxas
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

    def rel(a, b):
        bad = torch.isnan(a).any(dim=0) | torch.isnan(b).any(dim=0)
        return float(((a - b).abs().amax(dim=0) / (1 + b.abs().amax(dim=0)))[~bad].max())

    for name in SCENARIOS:
        sc = scenarios.get(name)
        ctrl = sc.make_controller()
        ctrl.setup_solver()
        kind = "qp" if name.endswith("_qp") else "nlp"
        mi = ctrl._max_iter(None) if kind == "nlp" else int(ctrl.options.get("max_iter", 0) or 0)
        inp = {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).to(dev))
               for k, v in sc.sample(N, seed=0).items()}
        t, q0, y = inp["t"], inp["q"], inp["y"]
        nq, ny, ns = q0.shape[0], ctrl._ny, q0.shape[0] + ctrl._nxv
        assert ctrl._nxv == 0
        nt = 1 + ns + ny
        vq = 0.7 * float(ctrl.solve_batch(t, q0, None, y)[0][:nq].abs().amax())
        q = q0.clone()

        def reset():
            q.copy_(q0)
        g = torch.Generator("cuda").manual_seed(1)
        cq = torch.randn(q0.shape, dtype=torch.float64, device=dev, generator=g)
        cs = torch.randn((ctrl._qn, N), dtype=torch.float64, device=dev, generator=g)
        res = {}
        plain = timed(lambda: res.__setitem__("r", ctrl.rollout_batch(t, q, K, dt, None, y, max_speed=vq)), reset)

        def tape_fwd():
            b = bc._rollout_batch(ctrl, "rollout_vjp", t, q, None, y)
            res["tape"] = bc._rollout_tape(ctrl, kind, b, K, dt, vq, None, mi)[2]
        fwd = timed(tape_fwd, reset)
        tape = res["tape"]

        def sweep():
            b = bc._rollout_batch(ctrl, "rollout_vjp", t, q0, None, y)
            res["s"] = bc._rollout_sweep(ctrl, kind, b, K, dt, vq, None, tape, cq, None, cs)
        rev = timed(sweep, lambda: None)
        pb = torch.cat([res["s"][0][None], res["s"][1]] + ([res["s"][3]] if ny else []))

        qg = q0.clone().requires_grad_(True)
        yg = y.clone().requires_grad_(True) if ny else None
        tg = t.clone().requires_grad_(True)

        def autograd():
            for a in (qg, yg, tg):
                if a is not None:
                    a.grad = None
            qK, _, sol, _ = ctrl.rollout_batch_differentiable(tg, qg, K, dt, None, yg, max_speed=vq)
            ((cq * qK).sum() + (cs * sol).sum()).backward()
        ag = timed(autograd, lambda: None)
        pb_ag = torch.cat([tg.grad[None], qg.grad] + ([yg.grad] if ny else []))

        def composed():
            aq, tb = cq.clone(), torch.zeros_like(t)
            yb = torch.zeros_like(y) if ny else None
            for k in range(K - 1, -1, -1):
                sb = torch.zeros((ctrl._qn, N), dtype=torch.float64, device=dev)
                sb[:ns] = dt * aq
                if k == K - 1:
                    sb = sb + cs
                sk = tape["sol"][k]
                sb[:ns] = torch.where(sk[:ns].abs() < vq, sb[:ns], 0.0)
                o = ctrl.vjp_batch(t + dt * float(k), tape["q"][k], None, y, sk, tape["status"][k], tape["active"][k],
                                   sb)
                tb, aq = tb + o[0], aq + o[1]
                if ny:
                    yb = yb + o[3]
            res["c"] = torch.cat([tb[None], aq] + ([yb] if ny else []))
        loop = timed(composed, lambda: None)

        def jac_contract():
            r = ctrl.rollout_jacobian(t, q, K, dt, None, y, max_speed=vq)
            # the sol_bar part of the gradient is not in jac (it holds d(q_K, x_K)/dp only): the contraction gives
            # the q_bar_K part, compared with a sweep along q_bar_K alone below
            res["J"] = torch.einsum("scn,sn->cn", r["jac"], cq)
        jac = timed(jac_contract, reset)
        b = bc._rollout_batch(ctrl, "rollout_vjp", t, q0, None, y)
        sq = bc._rollout_sweep(ctrl, kind, b, K, dt, vq, None, tape, cq, None, None)
        pb_q = torch.cat([sq[0][None], sq[1]] + ([sq[3]] if ny else []))
        log = ctrl._rollout_vjp["path"][:-len(".cubin")] + ".log"
        rec["scenarios"][name] = {
            "rows": ctrl._qm, "variables": ctrl._qn, "n_theta": nt, "max_speed": vq,
            "tape_bytes": sum(a.numel() * a.element_size() for a in tape.values() if a is not None),
            "rollout_batch_median_s": plain[0], "rollout_batch_min_max_s": plain[1:],
            "tape_forward_median_s": fwd[0], "tape_forward_min_max_s": fwd[1:],
            "sweep_median_s": rev[0], "sweep_min_max_s": rev[1:],
            "autograd_forward_backward_median_s": ag[0], "autograd_forward_backward_min_max_s": ag[1:],
            "composed_vjp_loop_median_s": loop[0], "composed_vjp_loop_min_max_s": loop[1:],
            "rollout_jacobian_contraction_median_s": jac[0], "rollout_jacobian_contraction_min_max_s": jac[1:],
            "sweep_speedup_over_composed": loop[0] / rev[0],
            "tape_plus_sweep_speedup_over_jacobian": jac[0] / (fwd[0] + rev[0]),
            "max_rel_dev": {"sweep_vs_composed": rel(pb, res["c"]),
                            "sweep_bit_identical_to_composed": bool(torch.equal(pb.nan_to_num(),
                                                                                res["c"].nan_to_num())),
                            "autograd_vs_sweep": rel(pb_ag, pb),
                            "q_bar_sweep_vs_jacobian_contraction": rel(pb_q, res["J"])},
            "nan_instances": int(torch.isnan(pb).any(dim=0).sum()),
            "n_failed_total": int(res["r"]["n_failed"].sum()),
            "ptxas": {k: ptxas(log, "clik_%s_rollout_%s_kernel" % (kind, k)) for k in ("tape", "vjp")},
        }
        print(name, json.dumps(rec["scenarios"][name]), flush=True)
        del tape, res
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
