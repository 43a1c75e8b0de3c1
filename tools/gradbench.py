#!/usr/bin/env python3
"""Times the gradient of a rollout's quadratic cost on the GPU, FR3, device-resident SoA batches.

  (a) rollout_cost        the fused rollout + cost (what sampling-based MPC runs)
  (b) rollout_cost_grad   the same cost and d cost / d (tau, q0, dq0) through the fused adjoint
  (c) composed            what (b) replaces: rollout (trajectory), fd_derivatives over all H*B pre-step states
                          (3 n^2 doubles each), then the backward recursion as batched mat-vecs in torch

Sizes: 65 536 x 64 (bench.py's rollout) and 8 192 x 64 (its per-GPU slice on 8 GPUs).  CUDA events around each call,
warm-up first, then the three alternated for --reps rounds; the median is reported.  (c) is checked against (b).
One JSON line per size, after a line naming the card and its power limit.

    python tools/gradbench.py [--reps 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:                      # the numbers still stand; say that the limit could not be read
        info["power_limit"] = f"unknown ({e})"
    return info


def composed(mb, q0, dq0, tau, dt, w):
    """rollout + fd_derivatives over every pre-step state + the backward recursion in torch: (cost, grad_tau, grad_q0, grad_dq0)."""
    import torch
    H, n, B = tau.shape
    qt, dqt = mb.rollout(q0, dq0, tau, dt)
    qs = torch.cat([q0[None], qt[:-1]]).permute(1, 0, 2).reshape(n, H * B).contiguous()     # state before step t, [n][H*B]
    dqs = torch.cat([dq0[None], dqt[:-1]]).permute(1, 0, 2).reshape(n, H * B).contiguous()
    us = tau.permute(1, 0, 2).reshape(n, H * B).contiguous()
    D = mb.fd_derivatives(qs, dqs, us).view(3, n, n, H, B)             # [blk][c][r][t][b] = d qdd_r / d x_c
    cw = {k: torch.as_tensor(v, dtype=torch.float64, device=q0.device)[:, None] for k, v in w.items()}
    e = qt - cw["q_ref"][None]
    cost = dt * ((cw["w_q"][None] * e * e).sum(1) + (cw["w_dq"][None] * dqt * dqt).sum(1) + (cw["w_tau"][None] * tau * tau).sum(1)).sum(0)
    cost = cost + (cw["w_q_final"] * e[-1] * e[-1]).sum(0) + (cw["w_dq_final"] * dqt[-1] * dqt[-1]).sum(0)
    a_q = 2 * cw["w_q_final"] * e[-1] + 2 * dt * cw["w_q"] * e[-1]
    a_dq = 2 * cw["w_dq_final"] * dqt[-1] + 2 * dt * cw["w_dq"] * dqt[-1]
    g_tau = torch.empty_like(tau)
    for t in range(H - 1, -1, -1):
        lam = dt * (a_dq + dt * a_q)
        g_tau[t] = torch.einsum("crb,rb->cb", D[2, :, :, t], lam) + 2 * dt * cw["w_tau"] * tau[t]
        a_dq = a_dq + dt * a_q + torch.einsum("crb,rb->cb", D[1, :, :, t], lam)
        a_q = a_q + torch.einsum("crb,rb->cb", D[0, :, :, t], lam)
        if t:
            a_q = a_q + 2 * dt * cw["w_q"] * e[t - 1]
            a_dq = a_dq + 2 * dt * cw["w_dq"] * dqt[t - 1]
    return cost, g_tau, a_q, a_dq


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--sizes", default="65536,8192")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("gradbench: needs a CUDA device (there is nothing to time on the CPU)")
    import rigidbody_rs_b200 as rb
    mb = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), device=0)
    lines = [dict(card(), kernel_variant=mb.kernel_variant)]
    print(json.dumps(lines[0]), flush=True)
    lim = mb.limits()
    n, H, dt = mb.n, a.horizon, 1e-3
    rng = np.random.default_rng(7)
    w = dict(q_ref=rng.uniform(-1, 1, n), w_q=rng.uniform(0, 2, n), w_dq=rng.uniform(0, 1, n), w_tau=rng.uniform(0, 1e-3, n),
             w_q_final=rng.uniform(0, 50, n), w_dq_final=rng.uniform(0, 5, n))
    for B in (int(s) for s in a.sizes.split(",")):
        dev = torch.device("cuda:0")
        q0 = torch.empty((n, B), dtype=torch.float64, device=dev); dq0 = torch.empty_like(q0)
        mb.fill(q0, 0x5EED0001, 0, lim["lower"], lim["upper"])
        mb.fill(dq0, 0x5EED0001, 1, -lim["velocity"], lim["velocity"])
        tau = torch.empty((H, n, B), dtype=torch.float64, device=dev)
        for t in range(H):
            mb.fill(tau[t], 0x5EED0002, 4 + t % 32, -0.3 * lim["effort"], 0.3 * lim["effort"], first_index=t * B)
        runs = {"a_rollout_cost": lambda: mb.rollout_cost(q0, dq0, tau, dt, **w),
                "b_rollout_cost_grad": lambda: mb.rollout_cost_grad(q0, dq0, tau, dt, **w),
                "c_composed": lambda: composed(mb, q0, dq0, tau, dt, w)}
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
        b, c = runs["b_rollout_cost_grad"](), runs["c_composed"]()
        agree = max(float(((x - y).abs().amax() / y.abs().amax().clamp_min(1.0)).item()) for x, y in zip(b, c))
        res = {"n_traj": B, "horizon": H, "dt": dt, "reps": a.reps,
               **{f"{k}_ms_median": float(np.median(v)) for k, v in times.items()},
               **{f"{k}_ms_min": float(np.min(v)) for k, v in times.items()},
               "b_over_a": float(np.median(times["b_rollout_cost_grad"]) / np.median(times["a_rollout_cost"])),
               "c_over_b": float(np.median(times["c_composed"]) / np.median(times["b_rollout_cost_grad"])),
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
