"""Link poses and collision-sphere terms of the fused rollout cost and its gradient (include/rigidbody.h
multibody_link_poses_batch, multibody_sphere_distance_batch, multibody_rollout_collision_cost,
multibody_rollout_collision_cost_grad).

The checker: per-link poses from the numpy twin's `_R` and parent table (descriptor frames, Rodrigues rotations about
the descriptor axes); Phi and min d from those poses; the rollout cost from the twin's rollout as in
test_rollout_tip_cost.py; the gradient from `rollout_vjp_np` fed with the collision terms' upstream gradient, which comes
from the point Jacobians of the sphere centres -- not from the per-link wrenches the CUDA kernel projects on the joint
screws.  The CPU tests hold the checker against central differences and the wrench projection against the point
Jacobians.  Bar on the GPU: |err| <= 1e-10 * max(1, max|ref|) per trajectory.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import CHAIN32, FR3, TOL
from test_rollout_gradients import (_aos, _chain_inputs, _close, _dev, _fr3_inputs, _np, _per_traj_err, _weights, quad_cost_upstream,
                                    rollout_np, rollout_vjp_np)
from test_rollout_tip_cost import _cost_close, _fr3_chain, _random, _tip, tip_cost_np, tip_grad_np

H_, DT = 16, 2e-3


# ------------------------------------------------------------------------------------------------ the numpy checker
def link_poses_np(ch, q):
    """q [n, B] -> [(R [B, 3, 3], P [B, 3]) of every link in the base frame], descriptor frames."""
    qb = np.asarray(q, dtype=np.float64).T
    out = []
    for i in range(ch.n):
        B = qb.shape[0]
        Rp, Pp = out[ch.parent[i]] if ch.parent[i] >= 0 else (np.tile(np.eye(3), (B, 1, 1)), np.zeros((B, 3)))
        out.append((Rp @ ch._R(i, qb[:, i]), Pp + np.einsum("bij,j->bi", Rp, ch.tp[i])))
    return out


def _col_arrays(col):
    link = np.asarray(col["link"], dtype=int)
    center = np.asarray(col["center"], dtype=np.float64).reshape(-1, 3)
    radius = np.asarray(col["radius"], dtype=np.float64)
    obst = np.asarray(col["obstacle"], dtype=np.float64).reshape(-1, 4)
    kind = list(col["kind"])
    return link, center, radius, kind, obst, float(col.get("margin", 0.0))


def _pairs(ch, q, col):
    """Per pair (k, o): sphere centre x [B, 3], d [B], unit direction u [B, 3] (d's gradient in x)."""
    link, center, radius, kind, obst, m = _col_arrays(col)
    poses = link_poses_np(ch, q)
    for k in range(len(link)):
        R, P = poses[link[k]]
        x = P + R @ center[k]
        for o in range(len(kind)):
            if kind[o] == "sphere":
                v = x - obst[o, :3]
                nrm = np.linalg.norm(v, axis=1)
                u = np.where(nrm[:, None] > 0, v / np.where(nrm > 0, nrm, 1.0)[:, None], 0.0)
                yield k, x, nrm - radius[k] - obst[o, 3], u
            else:
                nh = obst[o, :3] / np.linalg.norm(obst[o, :3])
                yield k, x, x @ nh - obst[o, 3] - radius[k], np.tile(nh, (x.shape[0], 1))


def phi_np(ch, q, col):
    """(min d [B], Phi [B]) of states q [n, B]."""
    m = float(col.get("margin", 0.0))
    dmin, phi = np.inf, 0.0
    for _, _, d, _ in _pairs(ch, q, col):
        dmin = np.minimum(dmin, d)
        phi = phi + np.maximum(0.0, m - d) ** 2
    return dmin, phi


def phi_grad_np(ch, q, col):
    """dPhi/dq [n, B] from the point Jacobians of the sphere centres: dx/dq_j = omega_j x (x - P_j) for the joints j that
    support the sphere's link, omega_j = R_j axis_j the joint's world axis."""
    link, *_ = _col_arrays(col)
    m = float(col.get("margin", 0.0))
    poses = link_poses_np(ch, q)
    qb = np.asarray(q).T
    g = np.zeros((ch.n, qb.shape[0]))
    for k, x, d, u in _pairs(ch, q, col):
        gx = (-2.0 * np.maximum(0.0, m - d))[:, None] * u
        j = link[k]
        while j >= 0:
            R, P = poses[j]
            om = R @ ch.axis[j]
            g[j] += (np.cross(om, x - P) * gx).sum(1)
            j = ch.parent[j]
    return g


def col_cost_np(ch, q0, dq0, tau, dt, q_traj, dq_traj, tip, col, **w):
    """multibody_rollout_collision_cost of a stored trajectory: tip_cost_np plus the collision terms, [B]."""
    H = tau.shape[0]
    qH = q_traj[-1] if H else q0
    run = sum(dt * col["w"] * phi_np(ch, q_traj[t], col)[1] for t in range(H))
    return tip_cost_np(ch, q0, dq0, tau, dt, q_traj, dq_traj, tip, **w) + run + col["w_final"] * phi_np(ch, qH, col)[1]


def col_cost_grad_np(ch, q0, dq0, tau, dt, q_traj, dq_traj, tip, col, **w):
    """(grad_tau, grad_q0, grad_dq0) of col_cost_np: rollout_vjp_np with the quadratic, tip and collision upstream gradients."""
    H = tau.shape[0]
    n = np.shape(q0)[0]
    quad = {k: w.get(k) for k in ("q_ref", "w_q", "w_dq", "w_q_final", "w_dq_final")}
    gq, gdq, gqf, gdqf = quad_cost_upstream(q0, dq0, dt, q_traj, dq_traj, **quad)
    if H:
        gq = gq + np.stack([tip_grad_np(ch, q_traj[t], tip, dt, 0.0) + dt * col["w"] * phi_grad_np(ch, q_traj[t], col) for t in range(H)])
    qH = q_traj[-1] if H else q0
    gqf = gqf + tip_grad_np(ch, qH, tip, 0.0, 1.0) + col["w_final"] * phi_grad_np(ch, qH, col)
    gt, a_q, a_dq = rollout_vjp_np(ch, q0, dq0, tau, dt, q_traj, dq_traj, gq, gdq, gqf, gdqf)
    w_tau = np.zeros(n) if w.get("w_tau") is None else np.asarray(w["w_tau"])
    return gt + 2.0 * dt * w_tau[None, :, None] * tau, a_q, a_dq


def _assert_active(ch, states, col):
    """Some pair is active (Phi > 0) in some of the states [.., n, B]: the collision terms are not a no-op here."""
    assert any((phi_np(ch, q, col)[1] > 0).any() for q in np.asarray(states).reshape(-1, ch.n, np.shape(states)[-1]))


def _collision(ch, q, seed, spheres_per_link=4, w=5.0, w_final=50.0, margin=0.05):
    """A synthetic sphere model (about `spheres_per_link` per link) and two sphere and two half-space obstacles placed
    about the link origins of the states q [n, B] (mean over B), so that a share of the pairs is active."""
    rng = np.random.default_rng(seed)
    link = np.repeat(np.arange(ch.n), spheres_per_link)
    S = len(link)
    center = rng.uniform(-0.08, 0.08, (S, 3))
    radius = rng.uniform(0.02, 0.08, S)
    poses = link_poses_np(ch, q)
    pts = np.array([P.mean(0) for _, P in poses])
    o1, o2 = pts[rng.integers(ch.n)], pts[rng.integers(ch.n)]
    lo = pts[:, 2].min()
    obstacle = [list(o1 + rng.uniform(-0.1, 0.1, 3)) + [0.1], list(o2 + rng.uniform(-0.1, 0.1, 3)) + [0.05],
                [0.0, 0.0, 2.0, lo + 0.02], list(rng.normal(size=3)) + [-0.3]]
    return dict(link=link, center=center, radius=radius, kind=["sphere", "sphere", "halfspace", "halfspace"], obstacle=np.array(obstacle),
                margin=margin, w=w, w_final=w_final)


# ------------------------------------------------------------------------------------------------ the checker, on the CPU
@pytest.mark.parametrize("chain", ["fr3", "random5"])
def test_numpy_collision_gradient_matches_finite_differences(oracle_fr3, chain):
    """col_cost_grad_np against central differences of col_cost_np (quadratic, tip and collision terms), every component
    of tau, q0 and dq0; H = 8, oblique axes for the random chain."""
    from oracle.rb_oracle_np import ChainNP
    H, B, dt = 8, 3, 1e-2
    if chain == "fr3":
        ch = _fr3_chain(oracle_fr3)
        q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H, 0x5EED0081)
        roll = lambda a, b, c: oracle_fr3.rollout_batch(a, b, c, dt)
    else:
        from test_host import _random_chain, AXES
        R, t, m, c, Ic = _random_chain(5, 81)
        ch = ChainNP.from_arrays(R, t, m, c, Ic, axis=AXES[:5])
        q0, dq0, tau = _chain_inputs(5, B, H, 82)
        roll = lambda a, b, c: rollout_np(ch, a, b, c, dt)
    w = _weights(ch.n, 83)
    tip = _tip(84)
    col = _collision(ch, q0, 85, margin=0.3)
    assert (phi_np(ch, q0, col)[1] > 0).all()
    cost = lambda a, b, c: col_cost_np(ch, a, b, c, dt, *roll(a, b, c), tip, col, **w)
    gt, gq, gdq = col_cost_grad_np(ch, q0, dq0, tau, dt, *roll(q0, dq0, tau), tip, col, **w)
    args = [q0, dq0, tau]
    for k, g in enumerate((gq, gdq, gt)):
        x = args[k]
        fd = np.zeros_like(x)
        for idx in np.ndindex(x.shape[:-1]):
            h = 1e-6 * max(1.0, np.abs(x[idx]).max())
            up, dn = [a.copy() for a in args], [a.copy() for a in args]
            up[k][idx] += h; dn[k][idx] -= h
            fd[idx] = (cost(*up) - cost(*dn)) / (2 * h)
        err = np.abs(fd - g).max() / max(1.0, np.abs(g).max())
        assert err < 1e-6, (chain, ("q0", "dq0", "tau")[k], err)


def test_wrench_projection_matches_point_jacobians(oracle_fr3):
    """dPhi/dq_j = s_j . sum_{l supported by j} w_l with s_j = (z_j ; P_j x z_j) and w_l = sum_k (x_k x g_k ; g_k): the form
    the CUDA inward sweep accumulates, against the point-Jacobian form of the checker, on FR3 and a random tree."""
    from oracle.rb_oracle_np import ChainNP
    from test_host import AXES, _random_chain, _random_tree
    R, t, m, c, Ic = _random_chain(9, 86)
    tree = ChainNP.from_arrays(R, t, m, c, Ic, axis=(AXES * 3)[:9], parent=_random_tree(9, 86))
    for ch, q in ((_fr3_chain(oracle_fr3), _fr3_inputs(oracle_fr3, 5, 0, 0x5EED0086)[0]), (tree, np.random.default_rng(86).uniform(-2, 2, (9, 5)))):
        col = _collision(ch, q, 87, margin=0.3)
        link, *_ = _col_arrays(col)
        mg = col["margin"]
        W = np.zeros((ch.n, q.shape[1], 6))
        for k, x, d, u in _pairs(ch, q, col):
            g = (-2.0 * np.maximum(0.0, mg - d))[:, None] * u
            W[link[k], :, :3] += np.cross(x, g)
            W[link[k], :, 3:] += g
        poses = link_poses_np(ch, q)
        proj = np.zeros((ch.n, q.shape[1]))
        for j in range(ch.n):
            Rj, Pj = poses[j]
            z = Rj @ ch.axis[j]
            s = np.concatenate([z, np.cross(Pj, z)], axis=1)
            for l in range(ch.n):                          # links in the subtree of j
                a = l
                while a >= 0 and a != j:
                    a = ch.parent[a]
                if a == j:
                    proj[j] += (s * W[l]).sum(1)
        want = phi_grad_np(ch, q, col)
        assert np.abs(want).max() > 0
        np.testing.assert_allclose(proj, want, rtol=0, atol=1e-12 * max(1.0, np.abs(want).max()))


def test_collision_cost_rejects_unknown_keys_and_shapes():
    from rigidbody_rs_b200 import _collision_cost
    with pytest.raises(ValueError):
        _collision_cost({"spheres": 1})
    with pytest.raises(ValueError):
        _collision_cost({"link": [0, 1], "center": np.zeros((3, 3)), "radius": [0.1, 0.1]})
    with pytest.raises(ValueError):
        _collision_cost({"kind": ["sphere"], "obstacle": np.zeros(3)})


# ------------------------------------------------------------------------------------------------ on the B200
def _poses_close(mb, ch, q):
    got = mb.link_poses(q)
    for l, (R, P) in enumerate(link_poses_np(ch, q)):
        _close(got[12 * l:12 * l + 3], P.T)
        _close(got[12 * l + 3:12 * l + 12], R.reshape(-1, 9).T)
    return got


@pytest.mark.gpu
def test_link_poses(rb, mb_fr3, oracle_fr3, oracle_chain32):
    """FR3, chain32, random chains of 1..40 joints with oblique axes, and trees: every link's pose against the checker;
    the last link's is tip_pose's to rounding; one state gives (P [n, 3], R [n, 3, 3]); the same bits under every family."""
    from oracle.rb_oracle_np import ChainNP
    from test_gpu_parity import _variants
    cases = [(mb_fr3, _fr3_chain(oracle_fr3), _fr3_inputs(oracle_fr3, 77, 0, 0x5EED0090)[0]),
             (rb.Multibody.from_urdf(CHAIN32), ChainNP(oracle_chain32.model), np.random.default_rng(90).uniform(-2, 2, (32, 50)))]
    for n, tree in ((1, False), (2, False), (7, False), (17, False), (40, False), (6, True), (20, True)):
        mb, ch = _random(n, 900 + n, tree)
        cases.append((mb, ch, _chain_inputs(n, 45, 0, 910 + n)[0]))
    for mb, ch, q in cases:
        got = _poses_close(mb, ch, q)
        n = ch.n
        x, Rt = mb.tip_pose(q)[:3], mb.tip_pose(q)[3:]
        _close(got[12 * (n - 1):12 * (n - 1) + 3], x)
        _close(got[12 * (n - 1) + 3:12 * n], Rt)
        P1, R1 = mb.link_poses(q[:, 3].copy())
        np.testing.assert_array_equal(P1, got[:, 3].reshape(n, 12)[:, :3])
        np.testing.assert_array_equal(R1, got[:, 3].reshape(n, 12)[:, 3:].reshape(n, 3, 3))
    q = cases[0][2]
    ref = mb_fr3.link_poses(q)
    for mb in _variants(rb, FR3):
        np.testing.assert_array_equal(mb.link_poses(q), ref, err_msg=mb.kernel_variant)
    aos = mb_fr3.link_poses(_aos(q), layout="aos")
    np.testing.assert_array_equal(aos, _aos(ref))
    np.testing.assert_array_equal(_np(mb_fr3.link_poses(*_dev(q)))[0], ref)


@pytest.mark.gpu
def test_sphere_distance(rb, mb_fr3, oracle_fr3):
    """min d and Phi against the checker on FR3, a random chain and a random tree; host, device and AoS bit for bit."""
    cases = [(mb_fr3, _fr3_chain(oracle_fr3), _fr3_inputs(oracle_fr3, 200, 0, 0x5EED0091)[0])]
    for n, tree in ((9, False), (11, True)):
        mb, ch = _random(n, 920 + n, tree)
        cases.append((mb, ch, _chain_inputs(n, 150, 0, 930 + n)[0]))
    for mb, ch, q in cases:
        col = _collision(ch, q, 91)
        got = mb.sphere_distance(q, col)
        dmin, phi = phi_np(ch, q, col)
        _close(got[0:1], dmin[None])
        _close(got[1:2], phi[None])
        assert (phi > 0).any()
        np.testing.assert_array_equal(_np(mb.sphere_distance(*_dev(q), col))[0], got)
        np.testing.assert_array_equal(mb.sphere_distance(_aos(q), col, layout="aos"), _aos(got))
        one = mb.sphere_distance(q[:, 0].copy(), col)
        assert one == (got[0, 0], got[1, 0])


@pytest.mark.gpu
def test_fr3_every_family(rb, oracle_fr3):
    """FR3 under every kernel family: cost and all three gradients against the checker; the gradient entry's cost is the
    cost entry's, bit for bit."""
    from test_gpu_parity import _variants
    ch = _fr3_chain(oracle_fr3)
    B = 64
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H_, 0x5EED0092)
    w = _weights(7, 92)
    tip = _tip(92, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    col = _collision(ch, q0, 92)
    traj = oracle_fr3.rollout_batch(q0, dq0, tau, DT)
    ref_cost = col_cost_np(ch, q0, dq0, tau, DT, *traj, tip, col, **w)
    ref = col_cost_grad_np(ch, q0, dq0, tau, DT, *traj, tip, col, **w)
    assert np.abs(ref_cost - tip_cost_np(ch, q0, dq0, tau, DT, *traj, tip, **w)).max() > 0
    fams = []
    for mb in _variants(rb, FR3):
        fams.append(mb.kernel_variant)
        cost = mb.rollout_cost(q0, dq0, tau, DT, tip=tip, collision=col, **w)
        _cost_close(cost, ref_cost)
        c2, gt, gq, gdq = mb.rollout_cost_grad(q0, dq0, tau, DT, tip=tip, collision=col, **w)
        np.testing.assert_array_equal(c2, cost, err_msg=mb.kernel_variant)
        for got, want in zip((gt, gq, gdq), ref):
            _close(got, want)
        _same_tip_bits(mb, q0, dq0, tau, DT, tip, col, w)
    assert fams == ["fr3-specialised", "jit-specialised", "generic-7", "generic-n"]


def _same_tip_bits(mb, q0, dq0, tau, dt, tip, col, w, grad=True):
    """collision=None and inactive collision terms give the tip call's bits and launches."""
    ref = mb.rollout_cost(q0, dq0, tau, dt, tip=tip, **w)
    inactive = (None, dict(col, link=[], center=np.zeros((0, 3)), radius=[]), dict(col, kind=[], obstacle=np.zeros((0, 4))),
                dict(col, w=0.0, w_final=0.0))
    for c in inactive:
        n0 = mb.launch_count
        np.testing.assert_array_equal(mb.rollout_cost(q0, dq0, tau, dt, tip=tip, collision=c, **w), ref, err_msg=mb.kernel_variant)
        n1 = mb.launch_count
        mb.rollout_cost(q0, dq0, tau, dt, tip=tip, **w)
        assert mb.launch_count - n1 == n1 - n0
    if grad:
        gref = mb.rollout_cost_grad(q0, dq0, tau, dt, tip=tip, **w)
        for c in inactive:
            for a, b in zip(mb.rollout_cost_grad(q0, dq0, tau, dt, tip=tip, collision=c, **w), gref):
                np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_chain32_every_family(rb, oracle_chain32):
    from test_gpu_parity import _variants
    from oracle.rb_oracle_np import ChainNP
    ch = ChainNP(oracle_chain32.model)
    B, H = 40, 6
    rng = np.random.default_rng(93)
    q0, dq0, tau = rng.uniform(-1, 1, (32, B)), rng.uniform(-0.5, 0.5, (32, B)), rng.uniform(-0.2, 0.2, (H, 32, B))
    w = _weights(32, 93)
    tip = _tip(93, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    col = _collision(ch, q0, 93, spheres_per_link=2)
    traj = rollout_np(ch, q0, dq0, tau, DT)
    _assert_active(ch, traj[0], col)
    ref = col_cost_np(ch, q0, dq0, tau, DT, *traj, tip, col, **w)
    fams = []
    for mb in _variants(rb, CHAIN32):
        fams.append(mb.kernel_variant)
        _cost_close(mb.rollout_cost(q0, dq0, tau, DT, tip=tip, collision=col, **w), ref)
        _same_tip_bits(mb, q0, dq0, tau, DT, tip, col, w, grad=False)
    assert fams == ["chain32-specialised", "generic-n"]


@pytest.mark.gpu
@pytest.mark.parametrize("n,tree", [(1, False), (5, False), (12, False), (20, False), (40, False), (5, True), (20, True)])
def test_random_chains_and_trees_cost(rb, n, tree):
    mb, ch = _random(n, 940 + n, tree)
    B, H = 33, 9
    q0, dq0, tau = _chain_inputs(n, B, H, 950 + n)
    w = _weights(n, 960 + n)
    tip = _tip(970 + n)
    col = _collision(ch, q0, 980 + n, spheres_per_link=3)
    traj = rollout_np(ch, q0, dq0, tau, DT)
    _assert_active(ch, traj[0], col)
    ref = col_cost_np(ch, q0, dq0, tau, DT, *traj, tip, col, **w)
    _cost_close(mb.rollout_cost(q0, dq0, tau, DT, tip=tip, collision=col, **w), ref)
    _same_tip_bits(mb, q0, dq0, tau, DT, tip, col, w, grad=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 5, 7, 12])
def test_random_chains_gradient(rb, n):
    mb, ch = _random(n, 1000 + n)
    B = 48
    q0, dq0, tau = _chain_inputs(n, B, H_, 1010 + n)
    w = _weights(n, 1020 + n)
    tip = _tip(1030 + n)
    col = _collision(ch, q0, 1040 + n, margin=0.2)
    qt, dqt = mb.rollout(q0, dq0, tau, DT)
    assert max(_per_traj_err(a, b).max() for a, b in zip((qt, dqt), rollout_np(ch, q0, dq0, tau, DT))) < TOL
    cost, *got = mb.rollout_cost_grad(q0, dq0, tau, DT, tip=tip, collision=col, **w)
    _assert_active(ch, qt, col)
    _cost_close(cost, col_cost_np(ch, q0, dq0, tau, DT, qt, dqt, tip, col, **w))
    np.testing.assert_array_equal(cost, mb.rollout_cost(q0, dq0, tau, DT, tip=tip, collision=col, **w))
    for a, b in zip(got, col_cost_grad_np(ch, q0, dq0, tau, DT, qt, dqt, tip, col, **w)):
        _close(a, b)


@pytest.mark.gpu
def test_autograd_gradcheck(rb, mb_fr3, oracle_fr3):
    import torch
    q0, dq0, tau = _fr3_inputs(oracle_fr3, 3, 3, 0x5EED0094)
    ch = _fr3_chain(oracle_fr3)
    col = _collision(ch, q0, 94, margin=0.3)
    w = dict(w_q=np.ones(7), w_tau=np.full(7, 1e-3))
    ins = [x.requires_grad_(True) for x in _dev(q0, dq0, tau)]
    f = lambda a, b, c: mb_fr3.rollout_cost_autograd(a, b, c, 1e-2, collision=col, **w)
    assert torch.autograd.gradcheck(f, ins)
    cost = f(*ins)
    np.testing.assert_array_equal(cost.detach().cpu().numpy(), mb_fr3.rollout_cost(q0, dq0, tau, 1e-2, collision=col, **w))
    cost.sum().backward()
    _, gt, gq, gdq = mb_fr3.rollout_cost_grad(q0, dq0, tau, 1e-2, collision=col, **w)
    for x, want in zip(ins, (gq, gdq, gt)):
        np.testing.assert_array_equal(x.grad.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [0, 1, 33])
def test_layouts_memory_and_leading_dimension(rb, mb_fr3, oracle_fr3, H):
    """Host against device and SoA against AoS bit for bit, and a NaN-padded leading dimension through the C ABI."""
    from rigidbody_rs_b200 import _collision_cost, _lib, _tip_cost
    lib = _lib.lib
    mb = mb_fr3
    B = 129
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H, 0x5EED0095)
    ch = _fr3_chain(oracle_fr3)
    w = _weights(7, 95)
    tip = _tip(95)
    col = _collision(ch, q0, 95)
    kw = dict(tip=tip, collision=col, **w)
    host = mb.rollout_cost_grad(q0, dq0, tau, DT, **kw)
    dev = _np(*mb.rollout_cost_grad(*_dev(q0, dq0, tau), DT, **kw))
    aos = mb.rollout_cost_grad(_aos(q0), _aos(dq0), _aos(tau), DT, layout="aos", **kw)
    for k in range(4):
        np.testing.assert_array_equal(dev[k], host[k])
        np.testing.assert_array_equal(aos[k], host[k] if k == 0 else _aos(host[k]))
    for c in (mb.rollout_cost(q0, dq0, tau, DT, **kw), _np(mb.rollout_cost(*_dev(q0, dq0, tau), DT, **kw))[0],
              mb.rollout_cost(_aos(q0), _aos(dq0), _aos(tau), DT, layout="aos", **kw)):
        np.testing.assert_array_equal(c, host[0])
    traj = oracle_fr3.rollout_batch(q0, dq0, tau, DT) if H else (np.zeros((0, 7, B)), np.zeros((0, 7, B)))
    _cost_close(host[0], col_cost_np(ch, q0, dq0, tau, DT, *traj, tip, col, **w))
    if H:
        for got, want in zip(host[1:], col_cost_grad_np(ch, q0, dq0, tau, DT, *traj, tip, col, **w)):
            _close(got, want)
    ld = B + 31
    nan = float("nan")
    p = lambda x: C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data) if x is not None else None
    qc, keep = mb._quad_cost(**w)
    tc, keep_tip = _tip_cost(tip)
    cc, keep_col = _collision_cost(col)
    for mem in (_lib.RB_MEM_DEVICE, _lib.RB_MEM_HOST):
        def wide(x):
            wd = np.full(x.shape[:-1] + (ld,), nan)
            wd[..., :B] = x
            return _dev(wd)[0] if mem == _lib.RB_MEM_DEVICE else wd
        back = lambda x: x.cpu().numpy() if mem == _lib.RB_MEM_DEVICE else x
        wq, wdq, wtau = (wide(x) for x in (q0, dq0, tau))
        cost, gt, gq, gdq = wide(np.full((1, B), nan))[0], wide(np.full((H, 7, B), nan)), wide(np.full((7, B), nan)), wide(np.full((7, B), nan))
        rc = lib.multibody_rollout_collision_cost_grad(mb._h, p(wq), p(wdq), p(wtau), DT, H, C.byref(qc), C.byref(tc), C.byref(cc), p(cost),
                                                       p(gt), p(gq), p(gdq), B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(cost)[:B], host[0])
        for got, want in zip((gt, gq, gdq), host[1:]):
            g = back(got)
            np.testing.assert_array_equal(g[..., :B], want)
            assert np.isnan(g[..., B:]).all()
        cost = wide(np.full((1, B), nan))[0]
        rc = lib.multibody_rollout_collision_cost(mb._h, p(wq), p(wdq), p(wtau), DT, H, C.byref(qc), C.byref(tc), C.byref(cc), p(cost),
                                                  None, None, B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(cost)[:B], host[0])
        pose = wide(np.full((84, B), nan))
        rc = lib.multibody_link_poses_batch(mb._h, p(wq), p(pose), B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(pose)[:, :B], mb.link_poses(q0))
        assert np.isnan(back(pose)[:, B:]).all()


@pytest.mark.gpu
def test_gradient_in_chunks_equals_one_chunk(rb, mb_fr3, oracle_fr3):
    """A batch whose trajectory workspace exceeds one chunk gives, per trajectory, the bits of a one-chunk batch."""
    import torch
    mb = mb_fr3
    B, H, dt = 10_000, 1000, 1e-3
    q0, dq0, _ = _fr3_inputs(oracle_fr3, B, 0, 0x5EED0096)
    gen = torch.Generator(device="cuda:0").manual_seed(96)
    eff = torch.from_numpy(oracle_fr3.model.effort).to("cuda:0")[None, :, None]
    tau = (torch.rand((H, 7, B), dtype=torch.float64, device="cuda:0", generator=gen) * 2 - 1) * 0.2 * eff
    col = _collision(_fr3_chain(oracle_fr3), q0, 96)
    kw = dict(tip=_tip(96), collision=col, **_weights(7, 96))
    tq, tdq = _dev(q0, dq0)
    full = mb.rollout_cost_grad(tq, tdq, tau, dt, **kw)
    for lo, hi in ((0, 100), (B - 100, B)):
        part = mb.rollout_cost_grad(tq[:, lo:hi].contiguous(), tdq[:, lo:hi].contiguous(), tau[..., lo:hi].contiguous(), dt, **kw)
        for a, b in zip(full, part):
            np.testing.assert_array_equal(a[..., lo:hi].cpu().numpy(), b.cpu().numpy())
    assert all(bool(torch.isfinite(x).all()) for x in full)


@pytest.mark.gpu
def test_multi_device_equals_single_device(rb, mb_fr3, oracle_fr3):
    from test_gpu_parity import _two_devices
    mm = rb.Multibody.from_urdf(FR3, devices=_two_devices())
    B = 301
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, 12, 0x5EED0097)
    col = _collision(_fr3_chain(oracle_fr3), q0, 97)
    kw = dict(tip=_tip(97), collision=col, **_weights(7, 97))
    for layout, f in (("soa", lambda x: x), ("aos", _aos)):
        a = mm.rollout_cost(f(q0), f(dq0), f(tau), DT, layout=layout, **kw)
        np.testing.assert_array_equal(a, mb_fr3.rollout_cost(f(q0), f(dq0), f(tau), DT, layout=layout, **kw))
        for x, y in zip(mm.rollout_cost_grad(f(q0), f(dq0), f(tau), DT, layout=layout, **kw),
                        mb_fr3.rollout_cost_grad(f(q0), f(dq0), f(tau), DT, layout=layout, **kw)):
            np.testing.assert_array_equal(x, y)
        np.testing.assert_array_equal(mm.link_poses(f(q0), layout=layout), mb_fr3.link_poses(f(q0), layout=layout))
        np.testing.assert_array_equal(mm.sphere_distance(f(q0), col, layout=layout), mb_fr3.sphere_distance(f(q0), col, layout=layout))
    with pytest.raises(rb.RigidBodyError) as ei:
        mm.rollout_cost_grad(*_dev(q0, dq0, tau), DT, **kw)
    assert ei.value.code == -6
    mm.close()


@pytest.mark.gpu
def test_sphere_on_an_obstacle_centre(rb, mb_fr3, oracle_fr3):
    """A sphere whose world centre is exactly an obstacle's centre (the base link's origin at q = 0 is the base origin):
    finite cost and Phi, and that pair contributes no gradient."""
    q0, dq0 = np.zeros((7, 2)), np.zeros((7, 2))
    tau = np.zeros((2, 7, 2))
    ch = _fr3_chain(oracle_fr3)
    P0 = link_poses_np(ch, q0)[0][1][0]
    col = dict(link=[0], center=[[0.0, 0.0, 0.0]], radius=[0.1], kind=["sphere"], obstacle=[list(P0) + [0.1]], margin=0.05, w=1.0, w_final=1.0)
    d = mb_fr3.sphere_distance(q0, col)
    np.testing.assert_array_equal(d[0], -0.2)
    assert np.isfinite(d).all()
    cost, gt, gq, gdq = mb_fr3.rollout_cost_grad(q0, dq0, tau, DT, collision=col)
    assert np.isfinite(cost).all() and (cost > 0).all()
    off = mb_fr3.rollout_cost_grad(q0, dq0, tau, DT)
    for a, b in zip((gt, gq, gdq), off[1:]):
        _close(a, b)


@pytest.mark.gpu
def test_errors_and_unsupported_chains(rb, mb_fr3, oracle_fr3):
    from rigidbody_rs_b200 import _collision_cost, _lib
    lib = _lib.lib
    z = lambda n, B=4, H=2: (np.zeros((n, B)), np.zeros((n, B)), np.zeros((H, n, B)))
    for mb, ch in (_random(13, 98), _random(6, 99, tree=True)):
        q0, dq0, tau = z(mb.n)
        col = _collision(ch, q0, 98)
        with pytest.raises(rb.RigidBodyError) as ei:
            mb.rollout_cost_grad(q0, dq0, tau, DT, collision=col)
        assert ei.value.code == _lib.RB_ERR_UNSUPPORTED
        assert "12 joints" in str(ei.value)
        assert np.isfinite(mb.rollout_cost(q0, dq0, tau, DT, collision=col)).all()
    mb = mb_fr3
    q0, dq0, tau = z(7)
    good = _collision(_fr3_chain(oracle_fr3), q0, 98)
    p = lambda a: C.c_void_p(a.ctypes.data)
    cost, gt, gq, gdq, out = np.zeros(4), np.zeros((2, 7, 4)), np.zeros((7, 4)), np.zeros((7, 4)), np.zeros((2, 4))
    calls = (lambda cc: lib.multibody_rollout_collision_cost_grad(mb._h, p(q0), p(dq0), p(tau), DT, 2, None, None, cc, p(cost), p(gt), p(gq),
                                                                  p(gdq), 4, 0, 0, 0, None),
             lambda cc: lib.multibody_rollout_collision_cost(mb._h, p(q0), p(dq0), p(tau), DT, 2, None, None, cc, p(cost), None, None, 4, 0, 0, 0, None),
             lambda cc: lib.multibody_sphere_distance_batch(mb._h, p(q0), cc, p(out), 4, 0, 0, 0, None))
    gc, keep = _collision_cost(good)
    for f in calls:
        assert f(C.byref(gc)) == 0
    assert calls[0](None) == 0 and calls[1](None) == 0
    assert calls[2](None) == _lib.RB_ERR_NULL
    bad_arg = [dict(good, link=[7] + list(good["link"][1:])), dict(good, link=[-1] + list(good["link"][1:])),
               dict(good, center=np.where(np.arange(good["center"].size).reshape(-1, 3) == 4, np.nan, good["center"])),
               dict(good, radius=-np.asarray(good["radius"])), dict(good, kind=["sphere", "box", "halfspace", "halfspace"]),
               dict(good, obstacle=np.vstack([good["obstacle"][:3], [0.0, 0.0, 0.0, 1.0]])),
               dict(good, obstacle=np.vstack([good["obstacle"][:3], [0.0, 0.0, 1.0, np.inf]])),
               dict(good, obstacle=np.vstack([[0.0, 0.0, 0.0, -0.1], good["obstacle"][1:]])),
               dict(good, margin=-0.1), dict(good, margin=np.nan), dict(good, w=-1.0), dict(good, w_final=np.inf)]
    for bad in bad_arg:
        cc, keep_bad = _collision_cost(bad)
        for f in calls:
            assert f(C.byref(cc)) == _lib.RB_ERR_ARG, bad
    for field, value in (("n_spheres", -1), ("n_spheres", 257), ("n_obstacles", -1), ("n_obstacles", 65)):
        cc, keep_bad = _collision_cost(good)
        setattr(cc, field, value)
        for f in calls:
            assert f(C.byref(cc)) == _lib.RB_ERR_ARG, field
    for field in ("link", "center", "radius", "kind", "obstacle"):
        cc, keep_bad = _collision_cost(good)
        setattr(cc, field, None)
        for f in calls:
            assert f(C.byref(cc)) == _lib.RB_ERR_NULL, field
    for empty in (dict(good, link=[], center=np.zeros((0, 3)), radius=[]), dict(good, kind=[], obstacle=np.zeros((0, 4)))):
        cc, keep_e = _collision_cost(empty)
        assert calls[2](C.byref(cc)) == _lib.RB_ERR_ARG
        assert calls[1](C.byref(cc)) == 0
    assert lib.multibody_rollout_collision_cost(mb._h, p(q0), p(dq0), p(tau), DT, 2, None, None, C.byref(gc), None, None, None, 4, 0, 0, 0,
                                                None) == _lib.RB_ERR_NULL


@pytest.mark.gpu
def test_not_spd_gives_nan_for_the_bad_trajectories_only(rb):
    from test_rollout_gradients import _spd_where_q1_small
    mb = _spd_where_q1_small(rb)
    B, H = 6, 3
    q0 = np.zeros((2, B)); q0[1, 1::2] = 1.5
    dq0, tau = np.zeros((2, B)), np.zeros((H, 2, B))
    col = dict(link=[0, 1], center=[[0.1, 0.0, 0.0], [0.0, 0.1, 0.0]], radius=[0.1, 0.1], kind=["sphere", "halfspace"],
               obstacle=[[0.1, 0.1, 0.0, 0.1], [0.0, 0.0, 1.0, 0.0]], margin=0.1, w=1.0, w_final=2.0)
    with pytest.raises(rb.NotPositiveDefinite):
        mb.rollout_cost_grad(q0, dq0, tau, 1e-3, collision=col)
    from rigidbody_rs_b200 import _collision_cost, _lib
    lib = _lib.lib
    cc, keep = _collision_cost(col)
    cost, gt, gq, gdq = np.zeros(B), np.zeros((H, 2, B)), np.zeros((2, B)), np.zeros((2, B))
    p = lambda a: C.c_void_p(a.ctypes.data)
    rc = lib.multibody_rollout_collision_cost_grad(mb._h, p(q0), p(dq0), p(tau), 1e-3, H, None, None, C.byref(cc), p(cost), p(gt), p(gq),
                                                   p(gdq), B, 0, 0, 0, None)
    assert rc == _lib.RB_ERR_NOT_SPD
    for g in (cost, gt, gq, gdq):
        assert np.isnan(g[..., 1::2]).all() and np.isfinite(g[..., 0::2]).all()
    good = mb.rollout_cost_grad(q0[:, 0::2].copy(), dq0[:, 0::2].copy(), tau[..., 0::2].copy(), 1e-3, collision=col)
    for a, b in zip((cost, gt, gq, gdq), good):
        np.testing.assert_array_equal(a[..., 0::2], b)


@pytest.mark.gpu
def test_full_size_fr3_65536x64(rb, mb_fr3, oracle_fr3):
    """65 536 trajectories x 64 steps, device-resident: cost and gradients finite, the gradient entry's cost the cost
    entry's bits, and 128 strided trajectories against the checker."""
    import torch
    mb = mb_fr3
    B, H, dt = 65536, 64, 1e-3
    q0, dq0, _ = _fr3_inputs(oracle_fr3, B, 0, 0x5EED0098)
    rng = np.random.default_rng(98)
    tau = rng.uniform(-0.3, 0.3, (H, 7, B)) * oracle_fr3.model.effort[None, :, None]
    w = _weights(7, 98)
    ch = _fr3_chain(oracle_fr3)
    tip = _tip(98, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    col = _collision(ch, q0[:, :512], 98)
    d = _dev(q0, dq0, tau)
    cost = mb.rollout_cost(*d, dt, tip=tip, collision=col, **w)
    res = mb.rollout_cost_grad(*d, dt, tip=tip, collision=col, **w)
    assert all(bool(torch.isfinite(x).all()) for x in res)
    np.testing.assert_array_equal(res[0].cpu().numpy(), cost.cpu().numpy())
    got = [x.cpu().numpy() for x in res]
    del d, res
    torch.cuda.empty_cache()
    idx = np.arange(0, B, B // 128)
    s0, s1, st = q0[:, idx].copy(), dq0[:, idx].copy(), tau[..., idx].copy()
    traj = oracle_fr3.rollout_batch(s0, s1, st, dt)
    _assert_active(ch, traj[0], col)
    _cost_close(got[0][idx], col_cost_np(ch, s0, s1, st, dt, *traj, tip, col, **w))
    for g, want in zip(got[1:], col_cost_grad_np(ch, s0, s1, st, dt, *traj, tip, col, **w)):
        _close(g[..., idx], want)
