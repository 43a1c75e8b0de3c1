#!/usr/bin/env python3
"""Times the collision-sphere terms of the fused rollout cost and of its gradient on the GPU, FR3, device-resident SoA.

  (a) rollout_tip_cost             the fused rollout + quadratic cost + tip-pose terms
  (b) rollout_collision_cost       the same with the collision-sphere terms
  (c) composed                     what (b) replaces: rollout (trajectory), link_poses over all H*B states, and the tip and
                                   collision terms reduced in torch
  (d) rollout_tip_cost_grad        the gradient of (a) (fused adjoint)
  (e) rollout_collision_cost_grad  the gradient of (b)

The sphere model is synthetic, written out below: four spheres on each of the seven links (28 in all) along the link
frames' axes.  It is NOT a validated FR3 collision model (the repository has no collision geometry).  Obstacles: two
spheres and two half-spaces (a floor and a wall); the share of reached states with an active pair (Phi > 0) is reported.

Sizes: 65 536 x 64 (bench.py's rollout) and 8 192 x 64.  CUDA events around each call, warm-up first, then the five
alternated for --reps rounds; the median is reported.  (c) is checked against (b).  One JSON line per size, after a line
naming the card, its power limit and its max SM clock.

    python tools/collisionbench.py [--reps 10] [--out FILE]
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

# four spheres per link, in the link's (URDF joint) frame: along its z axis and one off-axis; radius 6 cm
SPHERES = [(l, c, 0.06) for l in range(7) for c in ((0.0, 0.0, -0.08), (0.0, 0.0, 0.0), (0.0, 0.0, 0.08), (0.08, 0.0, 0.0))]
COLLISION = dict(link=[s[0] for s in SPHERES], center=[s[1] for s in SPHERES], radius=[s[2] for s in SPHERES],
                 kind=["sphere", "sphere", "halfspace", "halfspace"],
                 obstacle=[[0.45, 0.0, 0.45, 0.12],         # a box-sized sphere in front of the arm
                           [0.25, -0.35, 0.70, 0.10],       # another to its right, higher up
                           [0.0, 0.0, 1.0, 0.10],           # the floor: z >= 0.1
                           [-1.0, 0.0, 0.0, -0.70]],        # a wall: x <= 0.7
                 margin=0.05, w=20.0, w_final=200.0)


def composed(mb, q0, dq0, tau, dt, w, tip, col):
    """rollout + link_poses of every state reached + the cost in torch: the quadratic, tip-pose and collision terms."""
    import torch
    H, n, B = tau.shape
    dev = q0.device
    qt, dqt = mb.rollout(q0, dq0, tau, dt)
    pose = mb.link_poses(qt.permute(1, 0, 2).reshape(n, H * B).contiguous()).view(n, 12, H, B)
    T = lambda v: torch.as_tensor(np.asarray(v, dtype=np.float64), device=dev)
    cw = {k: T(v)[:, None] for k, v in w.items()}
    e = qt - cw["q_ref"][None]
    cost = dt * ((cw["w_q"][None] * e * e).sum(1) + (cw["w_dq"][None] * dqt * dqt).sum(1) + (cw["w_tau"][None] * tau * tau).sum(1)).sum(0)
    cost = cost + (cw["w_q_final"] * e[-1] * e[-1]).sum(0) + (cw["w_dq_final"] * dqt[-1] * dqt[-1]).sum(0)
    P, R = pose[:, 0:3], pose[:, 3:12].reshape(n, 3, 3, H, B)          # [n, 3, H, B], [n, 3(row), 3(col), H, B]
    Rt = R[n - 1]
    x = P[n - 1] + torch.einsum("ijhb,j->ihb", Rt, T(tip["offset"]))
    ep = x - T(tip["p_ref"])[:, None, None]
    dR = ((Rt - T(tip["R_ref"])[:, :, None, None]) ** 2).sum((0, 1))
    run = (T(tip["w_p"])[:, None, None] * ep * ep).sum(0) + tip["w_R"] * dR
    fin = (T(tip["w_p_final"])[:, None] * ep[:, -1] * ep[:, -1]).sum(0) + tip["w_R_final"] * dR[-1]
    cost = cost + dt * run.sum(0) + fin
    link = torch.as_tensor(col["link"], device=dev)
    xs = P[link] + torch.einsum("sijhb,sj->sihb", R[link], T(col["center"]))   # [S, 3, H, B]
    rad, m, ob = T(col["radius"])[:, None, None], col["margin"], T(col["obstacle"])
    phi = torch.zeros((H, B), dtype=torch.float64, device=dev)
    for o, kind in enumerate(col["kind"]):
        if kind == "sphere":
            d = (xs - ob[o, :3][None, :, None, None]).norm(dim=1) - rad - ob[o, 3]
        else:
            nh = ob[o, :3] / ob[o, :3].norm()
            d = torch.einsum("sihb,i->shb", xs, nh) - ob[o, 3] - rad
        phi = phi + (m - d).clamp_min(0.0).pow(2).sum(0)
    return cost + dt * col["w"] * phi.sum(0) + col["w_final"] * phi[-1]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--sizes", default="65536,8192")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("collisionbench: needs a CUDA device (there is nothing to time on the CPU)")
    import rigidbody_rs_b200 as rb
    mb = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), device=0)
    lines = [dict(card(), kernel_variant=mb.kernel_variant, spheres=len(SPHERES), obstacles=len(COLLISION["kind"]))]
    print(json.dumps(lines[0]), flush=True)
    lim = mb.limits()
    n, H, dt = mb.n, a.horizon, 1e-3
    rng = np.random.default_rng(9)
    w = dict(q_ref=rng.uniform(-1, 1, n), w_q=rng.uniform(0, 2, n), w_dq=rng.uniform(0, 1, n), w_tau=rng.uniform(0, 1e-3, n),
             w_q_final=rng.uniform(0, 50, n), w_dq_final=rng.uniform(0, 5, n))
    tip = dict(offset=[0.0, 0.0, 0.1034], p_ref=[0.4, 0.1, 0.5], w_p=[10.0, 10.0, 10.0], w_p_final=[100.0, 100.0, 100.0],
               R_ref=[[1.0, 0.0, 0.0], [0.0, -1.0, 0.0], [0.0, 0.0, -1.0]], w_R=1.0, w_R_final=10.0)
    col = COLLISION
    for B in (int(s) for s in a.sizes.split(",")):
        dev = torch.device("cuda:0")
        q0 = torch.empty((n, B), dtype=torch.float64, device=dev); dq0 = torch.empty_like(q0)
        mb.fill(q0, 0x5EED0001, 0, lim["lower"], lim["upper"])
        mb.fill(dq0, 0x5EED0001, 1, -lim["velocity"], lim["velocity"])
        tau = torch.empty((H, n, B), dtype=torch.float64, device=dev)
        for t in range(H):
            mb.fill(tau[t], 0x5EED0002, 4 + t % 32, -0.3 * lim["effort"], 0.3 * lim["effort"], first_index=t * B)
        runs = {"a_rollout_tip_cost": lambda: mb.rollout_cost(q0, dq0, tau, dt, tip=tip, **w),
                "b_rollout_collision_cost": lambda: mb.rollout_cost(q0, dq0, tau, dt, tip=tip, collision=col, **w),
                "c_composed": lambda: composed(mb, q0, dq0, tau, dt, w, tip, col),
                "d_rollout_tip_cost_grad": lambda: mb.rollout_cost_grad(q0, dq0, tau, dt, tip=tip, **w),
                "e_rollout_collision_cost_grad": lambda: mb.rollout_cost_grad(q0, dq0, tau, dt, tip=tip, collision=col, **w)}
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
        b, c = runs["b_rollout_collision_cost"](), runs["c_composed"]()
        agree = float(((b - c).abs() / c.abs().clamp_min(1.0)).amax().item())
        qt, _ = mb.rollout(q0, dq0, tau, dt)
        phi = mb.sphere_distance(qt.permute(1, 0, 2).reshape(n, H * B).contiguous(), col)[1]
        active = float((phi > 0).double().mean().item())
        med = {k: float(np.median(v)) for k, v in times.items()}
        res = {"n_traj": B, "horizon": H, "dt": dt, "reps": a.reps, "share_of_states_with_an_active_pair": active,
               **{f"{k}_ms_median": v for k, v in med.items()},
               **{f"{k}_ms_min": float(np.min(v)) for k, v in times.items()},
               "b_over_a": med["b_rollout_collision_cost"] / med["a_rollout_tip_cost"],
               "c_over_b": med["c_composed"] / med["b_rollout_collision_cost"],
               "e_over_d": med["e_rollout_collision_cost_grad"] / med["d_rollout_tip_cost_grad"],
               "composed_vs_fused_max_rel_diff": agree}
        lines.append(res)
        print(json.dumps(res), flush=True)
        del q0, dq0, tau, b, c, qt, phi
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
