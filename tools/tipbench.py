#!/usr/bin/env python3
"""Times the tip-pose terms of the fused rollout cost and of its gradient on the GPU, FR3, device-resident SoA batches.

  (a) rollout_cost            the fused rollout + quadratic cost
  (b) rollout_tip_cost        the same with the tip-pose terms (position and orientation)
  (c) composed                what (b) replaces: rollout (trajectory), fwd_kin over all H*B states, the reduction in
                              torch -- position term only (no batched call returns the tip's orientation)
  (d) rollout_cost_grad       the quadratic cost's gradient (fused adjoint)
  (e) rollout_tip_cost_grad   the same with the tip-pose terms

Sizes: 65 536 x 64 (bench.py's rollout) and 8 192 x 64 (its per-GPU slice on 8 GPUs).  CUDA events around each call,
warm-up first, then the five alternated for --reps rounds; the median is reported.  (c) is checked against (b) run with
the orientation weights and the offset set to zero (the terms (c) can form).  One JSON line per size, after a line
naming the card and its power limit.

    python tools/tipbench.py [--reps 10] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gradbench import card  # noqa: E402


def composed(mb, q0, dq0, tau, dt, w, tip):
    """rollout + fwd_kin of every state reached + the cost in torch: the quadratic terms and the tip-position terms."""
    import torch
    H, n, B = tau.shape
    qt, dqt = mb.rollout(q0, dq0, tau, dt)
    x = mb.fwd_kin(qt.permute(1, 0, 2).reshape(n, H * B).contiguous()).view(3, H, B)
    cw = {k: torch.as_tensor(v, dtype=torch.float64, device=q0.device)[:, None] for k, v in w.items()}
    tw = {k: torch.as_tensor(tip[k], dtype=torch.float64, device=q0.device)[:, None] for k in ("p_ref", "w_p", "w_p_final")}
    e = qt - cw["q_ref"][None]
    cost = dt * ((cw["w_q"][None] * e * e).sum(1) + (cw["w_dq"][None] * dqt * dqt).sum(1) + (cw["w_tau"][None] * tau * tau).sum(1)).sum(0)
    cost = cost + (cw["w_q_final"] * e[-1] * e[-1]).sum(0) + (cw["w_dq_final"] * dqt[-1] * dqt[-1]).sum(0)
    ep = x - tw["p_ref"][:, None]
    cost = cost + dt * (tw["w_p"][:, None] * ep * ep).sum((0, 1)) + (tw["w_p_final"] * ep[:, -1] * ep[:, -1]).sum(0)
    return cost


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--sizes", default="65536,8192")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("tipbench: needs a CUDA device (there is nothing to time on the CPU)")
    import rigidbody_rs_b200 as rb
    mb = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), device=0)
    lines = [dict(card(), kernel_variant=mb.kernel_variant)]
    print(json.dumps(lines[0]), flush=True)
    lim = mb.limits()
    n, H, dt = mb.n, a.horizon, 1e-3
    rng = np.random.default_rng(9)
    w = dict(q_ref=rng.uniform(-1, 1, n), w_q=rng.uniform(0, 2, n), w_dq=rng.uniform(0, 1, n), w_tau=rng.uniform(0, 1e-3, n),
             w_q_final=rng.uniform(0, 50, n), w_dq_final=rng.uniform(0, 5, n))
    tip = dict(offset=[0.0, 0.0, 0.1034], p_ref=[0.4, 0.1, 0.5], w_p=[10.0, 10.0, 10.0], w_p_final=[100.0, 100.0, 100.0],
               R_ref=[[1.0, 0.0, 0.0], [0.0, -1.0, 0.0], [0.0, 0.0, -1.0]], w_R=1.0, w_R_final=10.0)
    tip_pos = dict(p_ref=tip["p_ref"], w_p=tip["w_p"], w_p_final=tip["w_p_final"])      # what the composed path can form
    for B in (int(s) for s in a.sizes.split(",")):
        dev = torch.device("cuda:0")
        q0 = torch.empty((n, B), dtype=torch.float64, device=dev); dq0 = torch.empty_like(q0)
        mb.fill(q0, 0x5EED0001, 0, lim["lower"], lim["upper"])
        mb.fill(dq0, 0x5EED0001, 1, -lim["velocity"], lim["velocity"])
        tau = torch.empty((H, n, B), dtype=torch.float64, device=dev)
        for t in range(H):
            mb.fill(tau[t], 0x5EED0002, 4 + t % 32, -0.3 * lim["effort"], 0.3 * lim["effort"], first_index=t * B)
        runs = {"a_rollout_cost": lambda: mb.rollout_cost(q0, dq0, tau, dt, **w),
                "b_rollout_tip_cost": lambda: mb.rollout_cost(q0, dq0, tau, dt, tip=tip, **w),
                "c_composed": lambda: composed(mb, q0, dq0, tau, dt, w, tip_pos),
                "d_rollout_cost_grad": lambda: mb.rollout_cost_grad(q0, dq0, tau, dt, **w),
                "e_rollout_tip_cost_grad": lambda: mb.rollout_cost_grad(q0, dq0, tau, dt, tip=tip, **w)}
        for f in runs.values():                 # warm-up (module loads, allocator)
            f(); f()
        mb.sync()
        times = {k: [] for k in runs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(a.reps):
            for k, f in runs.items():
                ev0.record(); f(); ev1.record(); ev1.synchronize()
                times[k].append(ev0.elapsed_time(ev1))
        mb.sync()
        b, c = mb.rollout_cost(q0, dq0, tau, dt, tip=tip_pos, **w), runs["c_composed"]()
        agree = float(((b - c).abs() / c.abs().clamp_min(1.0)).amax().item())
        med = {k: float(np.median(v)) for k, v in times.items()}
        res = {"n_traj": B, "horizon": H, "dt": dt, "reps": a.reps,
               **{f"{k}_ms_median": v for k, v in med.items()},
               **{f"{k}_ms_min": float(np.min(v)) for k, v in times.items()},
               "b_over_a": med["b_rollout_tip_cost"] / med["a_rollout_cost"],
               "c_over_b": med["c_composed"] / med["b_rollout_tip_cost"],
               "e_over_d": med["e_rollout_tip_cost_grad"] / med["d_rollout_cost_grad"],
               "composed_vs_fused_max_rel_diff": agree}
        lines.append(res)
        print(json.dumps(res), flush=True)
        del q0, dq0, tau, b, c
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
