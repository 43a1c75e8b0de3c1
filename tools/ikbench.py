#!/usr/bin/env python3
"""Times batched inverse kinematics of the tip frame on the GPU, FR3, device-resident SoA batches.

  (a) tip_pose    one batched tip-pose query
  (b) ik          multibody_ik_batch, max_iters = 50, full pose (position and orientation, unit weights)
  (c) composed    what (b) replaces: per iteration tip_pose and jac, a batched torch 6x6 Cholesky solve of the same
                  damped system, clamp, a trial tip_pose and the accept step (the algorithm of include/rigidbody.h,
                  run for all max_iters iterations: stopping early would need a device-to-host sync per iteration)

Problems: targets are the tip poses of random in-limit q*, seeds q* + N(0, 0.3^2) clipped to the limits.  CUDA events
around each call, warm-up first, then the three alternated for --reps rounds; the median is reported.  Also reported:
the converged fraction, the mean and maximum iterations of converged problems, the agreement of (c) with (b), and how
much of each warp's time its lanes spend on their own problem (mean iterations over the mean of each 32-problem
warp's maximum; problems that do not converge count max_iters).  One JSON line per size, after a line naming the card
and its power limit.

    python tools/ikbench.py [--reps 10] [--sizes 65536,1048576] [--out FILE]
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

TOL = 1e-6


def composed(mb, p, R, q0, lo, hi, max_iters, damping=1e-3):
    """The IK loop on batched engine calls and torch: returns (q, pos_err, rot_err, iters)."""
    import torch
    n, B = q0.shape
    sw = torch.tensor([1.0, 1.0, 1.0] + [2.0 ** 0.5] * 3, dtype=torch.float64, device=q0.device)
    eye = torch.eye(6, dtype=torch.float64, device=q0.device)
    Rt = R.T.reshape(B, 3, 3)
    pt = p.T

    def pose(q):
        P = mb.tip_pose(q)
        return P[3:].T.reshape(B, 3, 3), P[:3].T

    def objective(Rq, x):
        e = x - pt
        pos2 = (e * e).sum(1)
        rot2 = ((Rq - Rt) ** 2).sum((1, 2))
        return pos2 + rot2, pos2, rot2

    q = torch.minimum(torch.maximum(q0, lo[:, None]), hi[:, None])
    Rq, x = pose(q)
    F, pos2, rot2 = objective(Rq, x)
    lam = torch.full((B,), damping, dtype=torch.float64, device=q0.device)
    iters = torch.full((B,), -1, dtype=torch.int64, device=q0.device)
    active = torch.ones(B, dtype=torch.bool, device=q0.device)
    angle = lambda r2: 2.0 * torch.asin(torch.clamp(r2.sqrt() / 8.0 ** 0.5, max=1.0))
    for k in range(max_iters + 1):
        conv = active & (pos2.sqrt() <= TOL) & (angle(rot2) <= TOL)
        iters = torch.where(conv, torch.full_like(iters, k), iters)
        active = active & ~conv
        if k == max_iters:
            break
        J = mb.jac(q).view(n, 6, B).permute(2, 1, 0)                    # tip frame [B, 6, n]
        Jb = torch.cat([Rq @ J[:, :3], Rq @ J[:, 3:]], 1)                 # base frame (tracked point = tip origin)
        WJ = sw[None, :, None] * Jb
        A = WJ @ WJ.transpose(1, 2) + lam[:, None, None] * eye
        om = 0.5 * torch.linalg.cross(Rq, Rt, dim=1).sum(2)
        b = sw * torch.cat([pt - x, om], 1)
        L, info = torch.linalg.cholesky_ex(A)
        ok = info == 0
        y = torch.cholesky_solve(b[..., None], L)[..., 0]
        d = torch.einsum("bkn,bk->nb", Jb, sw * y)
        qn = torch.where(ok[None], q + d, q)
        qn = torch.minimum(torch.maximum(qn, lo[:, None]), hi[:, None])
        Rn, xn = pose(qn)
        Fn, pos2n, rot2n = objective(Rn, xn)
        acc = active & ok & (Fn < F)
        rej = active & ~acc
        q = torch.where(acc[None], qn, q)
        Rq = torch.where(acc[:, None, None], Rn, Rq); x = torch.where(acc[:, None], xn, x)
        F, pos2, rot2 = torch.where(acc, Fn, F), torch.where(acc, pos2n, pos2), torch.where(acc, rot2n, rot2)
        lam = torch.where(acc, torch.clamp(lam / 10, min=1e-12), torch.where(rej, torch.clamp(lam * 10, max=1e12), lam))
    return q, pos2.sqrt(), angle(rot2), iters


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--sizes", default="65536,1048576")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("ikbench: needs a CUDA device (there is nothing to time on the CPU)")
    import rigidbody_rs_b200 as rb
    mb = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), device=0)
    lines = [dict(card(), kernel_variant=mb.kernel_variant)]
    print(json.dumps(lines[0]), flush=True)
    lim = mb.limits()
    n = mb.n
    dev = torch.device("cuda:0")
    lo, hi = (torch.as_tensor(lim[k], dtype=torch.float64, device=dev) for k in ("lower", "upper"))
    for B in (int(s) for s in a.sizes.split(",")):
        rng = np.random.default_rng(31)
        qs = torch.as_tensor(rng.uniform(lim["lower"], lim["upper"], (B, n)).T.copy(), device=dev)
        P = mb.tip_pose(qs)
        p, R = P[:3].contiguous(), P[3:].contiguous()
        q0 = torch.minimum(torch.maximum(qs + torch.as_tensor(rng.normal(0, 0.3, (n, B)), device=dev), lo[:, None]), hi[:, None]).contiguous()
        runs = {"a_tip_pose": lambda: mb.tip_pose(q0),
                "b_ik": lambda: mb.ik(p, R, q_init=q0, max_iters=a.iters),
                "c_composed": lambda: composed(mb, p, R, q0, lo, hi, a.iters)}
        for f in runs.values():                 # warm-up (module loads, allocator)
            f(); f()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(a.reps):
            for k, f in runs.items():
                ev0.record(); f(); ev1.record(); ev1.synchronize()
                times[k].append(ev0.elapsed_time(ev1))
        qb, info = runs["b_ik"]()
        qc, pos_c, rot_c, it_c = runs["c_composed"]()
        it = info[2].round().long()
        conv, conv_c = it >= 0, it_c >= 0
        both = conv & conv_c
        itf = torch.where(conv, it, torch.full_like(it, a.iters)).double()
        warp_max = itf[: B // 32 * 32].view(-1, 32).amax(1)
        med = {k: float(np.median(v)) for k, v in times.items()}
        res = {"n_problems": B, "max_iters": a.iters, "reps": a.reps,
               **{f"{k}_ms_median": v for k, v in med.items()},
               **{f"{k}_ms_min": float(np.min(v)) for k, v in times.items()},
               "c_over_b": med["c_composed"] / med["b_ik"],
               "b_over_a": med["b_ik"] / med["a_tip_pose"],
               "converged_fraction": float(conv.double().mean()),
               "iters_mean_converged": float(it[conv].double().mean()),
               "iters_max_converged": int(it[conv].max()),
               "lane_utilisation": float(itf[: B // 32 * 32].mean() / warp_max.mean()),
               "composed_same_converged_flag": float((conv == conv_c).double().mean()),
               "composed_same_iters": float((it == it_c).double().mean()),
               "composed_max_abs_q_diff_both_converged": float((qb - qc).abs().amax(0)[both].max())}
        lines.append(res)
        print(json.dumps(res), flush=True)
        del qs, P, p, R, q0, qb, qc, info
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
