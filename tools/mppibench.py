#!/usr/bin/env python3
"""Times one MPPI iteration (multibody_mppi_step) on the GPU, FR3, device-resident SoA, quadratic and tip-pose terms.

  (a) rollout_cost   the fused rollout cost alone, on samples drawn beforehand (start states broadcast beforehand too)
  (b) mppi_step      the whole iteration: sampler, rollout cost, weights, weighted mean
  (c) composed       what (b) replaces in torch: randn, clamp, broadcast of the start states, rollout_cost, softmin, einsum

Sizes: P = 1 problem of K = 65 536 samples and P = 64 problems of K = 1 024 samples, both H = 64 (the 65 536 x 64
rollouts of bench.py).  CUDA events around each call, warm-up first, then the three alternated for --reps rounds; the
median is reported.  (c) is also run on (b)'s samples and checked against (b).  One JSON line per size, after a line
naming the card, its power limit and its max SM clock.

    python tools/mppibench.py [--reps 10] [--out FILE]
    python tools/mppibench.py --profile [--out FILE]      # per-kernel times of (b) from torch.profiler, in a run of its own
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


def composed(mb, q0, dq0, u_nom, dt, sigma, lo, hi, K, lam, w, tip, tau=None):
    """(u_new [H, n, P], cost [P, K]) in torch around rollout_cost; `tau` [H, n, P K] replaces the drawn samples."""
    import torch
    H, n, P = u_nom.shape
    if tau is None:
        eps = torch.randn((H, n, P, K), dtype=torch.float64, device=u_nom.device)
        eps[..., 0] = 0.0
        tau = torch.minimum(torch.maximum(u_nom[..., None] + sigma[None, :, None, None] * eps, lo[None, :, None, None]), hi[None, :, None, None])
        tau = tau.reshape(H, n, P * K)
    cost = mb.rollout_cost(q0.repeat_interleave(K, 1), dq0.repeat_interleave(K, 1), tau, dt, tip=tip, **w).view(P, K)
    wt = torch.softmax(-cost / lam, dim=1)
    return torch.einsum("hnpk,pk->hnp", tau.view(H, n, P, K), wt), cost


def profile(mb, f, P, K, H, reps=5):
    """Mean CUDA time per call of each kernel f launches, from torch.profiler (warm-up first)."""
    import torch
    from torch.profiler import ProfilerActivity, profile as prof
    f(); f(); torch.cuda.synchronize()
    with prof(activities=[ProfilerActivity.CUDA]) as pr:
        for _ in range(reps):
            f()
        torch.cuda.synchronize()
    us = {}
    for e in pr.key_averages():
        if e.device_type.name == "CUDA" and e.count:
            us[e.key[:80]] = round(e.device_time_total / reps, 2)
    return {"n_problems": P, "n_samples": K, "horizon": H, "profile_reps": reps, "kernel_us_per_call": us}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--sizes", default="1x65536,64x1024")
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("mppibench: needs a CUDA device (there is nothing to time on the CPU)")
    import rigidbody_rs_b200 as rb
    mb = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), device=0)
    lines = [dict(card(), kernel_variant=mb.kernel_variant)]
    print(json.dumps(lines[0]), flush=True)
    lim = mb.limits()
    n, H, dt, lam = mb.n, a.horizon, 1e-3, 10.0
    rng = np.random.default_rng(9)
    w = dict(q_ref=rng.uniform(-1, 1, n), w_q=rng.uniform(0, 2, n), w_dq=rng.uniform(0, 1, n), w_tau=rng.uniform(0, 1e-3, n),
             w_q_final=rng.uniform(0, 50, n), w_dq_final=rng.uniform(0, 5, n))
    tip = dict(offset=[0.0, 0.0, 0.1034], p_ref=[0.4, 0.1, 0.5], w_p=[10.0, 10.0, 10.0], w_p_final=[100.0, 100.0, 100.0],
               R_ref=[[1.0, 0.0, 0.0], [0.0, -1.0, 0.0], [0.0, 0.0, -1.0]], w_R=1.0, w_R_final=10.0)
    dev = torch.device("cuda:0")
    eff = lim["effort"]
    sigma_h = 0.1 * eff
    sigma, lo, hi = (torch.as_tensor(v, device=dev) for v in (sigma_h, -eff, eff))
    for size in a.sizes.split(","):
        P, K = (int(x) for x in size.split("x"))
        q0 = torch.empty((n, P), dtype=torch.float64, device=dev); dq0 = torch.empty_like(q0)
        mb.fill(q0, 0x5EED0001, 0, lim["lower"], lim["upper"])
        mb.fill(dq0, 0x5EED0001, 1, -lim["velocity"], lim["velocity"])
        u_nom = torch.empty((H, n, P), dtype=torch.float64, device=dev)
        for t in range(H):
            mb.fill(u_nom[t], 0x5EED0002, 4 + t % 32, -0.3 * eff, 0.3 * eff, first_index=t * P)
        if a.profile:
            lines.append(profile(mb, lambda: mb.mppi_step(q0, dq0, u_nom, dt, sigma_h, K, lam, 7, tip=tip, **w), P, K, H))
            print(json.dumps(lines[-1]), flush=True)
            continue
        _, _, _, smp = mb.mppi_step(q0, dq0, u_nom, dt, sigma_h, K, lam, 7, samples=True, tip=tip, **w)
        q0s, dq0s = q0.repeat_interleave(K, 1), dq0.repeat_interleave(K, 1)
        runs = {"a_rollout_cost": lambda: mb.rollout_cost(q0s, dq0s, smp, dt, tip=tip, **w),
                "b_mppi_step": lambda: mb.mppi_step(q0, dq0, u_nom, dt, sigma_h, K, lam, 7, tip=tip, **w),
                "c_composed": lambda: composed(mb, q0, dq0, u_nom, dt, sigma, lo, hi, K, lam, w, tip)}
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
        u_b, c_b, _, smp_b = mb.mppi_step(q0, dq0, u_nom, dt, sigma_h, K, lam, 7, samples=True, tip=tip, **w)
        u_c, c_c = composed(mb, q0, dq0, u_nom, dt, sigma, lo, hi, K, lam, w, tip, tau=smp_b)
        rel = lambda x, y: float(((x - y).abs() / y.abs().clamp_min(1.0)).amax().item())
        med = {k: float(np.median(v)) for k, v in times.items()}
        res = {"n_problems": P, "n_samples": K, "horizon": H, "dt": dt, "temperature": lam, "reps": a.reps,
               **{f"{k}_ms_median": v for k, v in med.items()},
               **{f"{k}_ms_min": float(np.min(v)) for k, v in times.items()},
               "b_minus_a_ms": med["b_mppi_step"] - med["a_rollout_cost"],
               "c_over_b": med["c_composed"] / med["b_mppi_step"],
               "samples_bytes": H * n * P * K * 8,
               "same_samples_cost_max_rel_diff": rel(c_b, c_c), "same_samples_u_new_max_rel_diff": rel(u_b, u_c)}
        lines.append(res)
        print(json.dumps(res), flush=True)
        del q0, dq0, u_nom, smp, q0s, dq0s, smp_b, u_b, c_b, u_c, c_c
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
