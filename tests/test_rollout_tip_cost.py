"""Tip-pose terms of the fused rollout cost and its gradient (include/rigidbody.h multibody_rollout_tip_cost /
multibody_rollout_tip_cost_grad).

The checker: the numpy twin's rollout and its `ChainNP.fwd_kin` (tip orientation and origin) give the cost; its gradient
is `rollout_vjp_np` (tests/test_rollout_gradients.py) fed with the quadratic cost's upstream gradients plus the tip
terms', which come from the twin's `fwd_kin` and `jac` -- not from the world-frame wrench the CUDA kernel projects on
the joint screws.  The CPU test holds the checker against central differences of the whole cost.  Bar on the GPU:
|err| <= 1e-10 * max(1, max|ref|) per trajectory.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import CHAIN32, FR3, TOL
from test_rollout_gradients import (_aos, _chain_inputs, _close, _dev, _fr3_inputs, _np, _per_traj_err, _weights, quad_cost_np,
                                    quad_cost_upstream, rollout_np, rollout_vjp_np)

H_, DT = 16, 2e-3


# ------------------------------------------------------------------------------------------------ the numpy checker
def _tip_arrays(tip):
    g = lambda k, size: np.zeros(size) if tip.get(k) is None else np.asarray(tip[k], dtype=np.float64).reshape(size)
    R_ref = np.eye(3) if tip.get("R_ref") is None else np.asarray(tip["R_ref"], dtype=np.float64).reshape(3, 3)
    return g("offset", 3), g("p_ref", 3), g("w_p", 3), g("w_p_final", 3), R_ref, float(tip.get("w_R", 0.0)), float(tip.get("w_R_final", 0.0))


def tip_terms_np(chain, q, tip):
    """(running, terminal) tip terms of states q [n, B]: sum_k w_p[k] e_k^2 + w_R ||R - R_ref||_F^2 (and the terminal
    weights), x = p + R offset, e = x - p_ref, with (R, p) = the twin's fwd_kin."""
    off, p_ref, w_p, w_pf, R_ref, w_R, w_Rf = _tip_arrays(tip)
    R, p = chain.fwd_kin(np.asarray(q).T)
    e = p + R @ off - p_ref
    dR = ((R - R_ref) ** 2).sum((1, 2))
    return (w_p * e ** 2).sum(1) + w_R * dR, (w_pf * e ** 2).sum(1) + w_Rf * dR


def tip_grad_np(chain, q, tip, a, b):
    """d/dq of a * running + b * terminal tip terms at states q [n, B] -> [n, B], from the twin's fwd_kin and its
    tip-frame Jacobian: dx/dq_j = R (J_lin_j + J_rot_j x offset),  dR/dq_j = [R J_rot_j]x R."""
    off, p_ref, w_p, w_pf, R_ref, w_R, w_Rf = _tip_arrays(tip)
    qb = np.asarray(q).T
    R, p = chain.fwd_kin(qb)
    J = chain.jac(qb)                                                    # [B, 6, n], tip frame
    e = p + R @ off - p_ref                                              # [B, 3]
    W, wr = a * w_p + b * w_pf, a * w_R + b * w_Rf
    dx = np.einsum("bij,bjn->bin", R, J[:, 0:3] + np.cross(J[:, 3:6], off, axisa=1, axisb=0, axisc=1))
    om = np.einsum("bij,bjn->bin", R, J[:, 3:6])                          # world angular rate of each joint
    g = 2.0 * np.einsum("bi,bin->bn", W * e, dx)
    for j in range(chain.n):
        dRj = np.cross(om[:, :, j][:, :, None], R, axis=1)                # column k: om_j x R[:, k]
        g[:, j] += 2.0 * wr * ((R - R_ref) * dRj).sum((1, 2))
    return g.T


def tip_cost_np(chain, q0, dq0, tau, dt, q_traj, dq_traj, tip, **w):
    """multibody_rollout_tip_cost of a stored trajectory: the quadratic cost plus the tip terms, [B]."""
    qH = q_traj[-1] if tau.shape[0] else q0
    run = sum(dt * tip_terms_np(chain, q_traj[t], tip)[0] for t in range(tau.shape[0]))
    return quad_cost_np(q0, dq0, tau, dt, q_traj, dq_traj, **w) + run + tip_terms_np(chain, qH, tip)[1]


def tip_cost_grad_np(chain, q0, dq0, tau, dt, q_traj, dq_traj, tip, **w):
    """(grad_tau, grad_q0, grad_dq0) of tip_cost_np: rollout_vjp_np with the quadratic and the tip upstream gradients."""
    H = tau.shape[0]
    n = np.shape(q0)[0]
    quad = {k: w.get(k) for k in ("q_ref", "w_q", "w_dq", "w_q_final", "w_dq_final")}
    gq, gdq, gqf, gdqf = quad_cost_upstream(q0, dq0, dt, q_traj, dq_traj, **quad)
    gq = gq + np.stack([tip_grad_np(chain, q_traj[t], tip, dt, 0.0) for t in range(H)]) if H else gq
    gqf = gqf + tip_grad_np(chain, q_traj[-1] if H else q0, tip, 0.0, 1.0)
    gt, a_q, a_dq = rollout_vjp_np(chain, q0, dq0, tau, dt, q_traj, dq_traj, gq, gdq, gqf, gdqf)
    w_tau = np.zeros(n) if w.get("w_tau") is None else np.asarray(w["w_tau"])
    return gt + 2.0 * dt * w_tau[None, :, None] * tau, a_q, a_dq


def _tip(seed, pose=None):
    """Tip terms with a non-zero offset, a general target orientation and non-zero orientation weights.  `pose` = (R, p)
    of one reachable state puts the target near the workspace."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    R_ref = Rotation.from_rotvec(rng.normal(size=3)).as_matrix() if pose is None else pose[0] @ Rotation.from_rotvec(0.3 * rng.normal(size=3)).as_matrix()
    p_ref = rng.uniform(-0.5, 0.5, 3) if pose is None else pose[1] + rng.uniform(-0.1, 0.1, 3)
    return dict(offset=rng.uniform(-0.1, 0.1, 3), p_ref=p_ref, w_p=rng.uniform(0.5, 5, 3), w_p_final=rng.uniform(5, 50, 3),
                R_ref=R_ref, w_R=float(rng.uniform(0.1, 2)), w_R_final=float(rng.uniform(1, 10)))


def _fr3_chain(oracle_fr3):
    from oracle.rb_oracle_np import ChainNP
    return ChainNP(oracle_fr3.model)


def _random(n, seed, tree=False):
    """A random chain (oblique axes) or tree: (engine, twin)."""
    import rigidbody_rs_b200 as rb
    from oracle.rb_oracle_np import ChainNP
    from test_host import AXES, _random_chain, _random_tree
    R, t, m, c, Ic = _random_chain(n, seed)
    ax = (AXES * (n // len(AXES) + 1))[:n]
    par = _random_tree(n, seed) if tree else None
    return (rb.Multibody.from_descriptor(R, t, m, c, Ic, axis=ax, parent=par),
            ChainNP.from_arrays(R, t, m, c, Ic, axis=ax, parent=par))


# ------------------------------------------------------------------------------------------------ the checker, on the CPU
@pytest.mark.parametrize("chain", ["fr3", "random5"])
def test_numpy_tip_cost_gradient_matches_finite_differences(oracle_fr3, chain):
    """tip_cost_grad_np against central differences of tip_cost_np (quadratic and tip terms), every component of tau,
    q0 and dq0; H = 8, non-zero offset and orientation weights, oblique axes for the random chain."""
    from oracle.rb_oracle_np import ChainNP
    H, B, dt = 8, 3, 1e-2
    if chain == "fr3":
        ch = _fr3_chain(oracle_fr3)
        q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H, 0x5EED0051)
        roll = lambda a, b, c: oracle_fr3.rollout_batch(a, b, c, dt)
    else:
        from test_host import _random_chain, AXES
        R, t, m, c, Ic = _random_chain(5, 51)
        ch = ChainNP.from_arrays(R, t, m, c, Ic, axis=AXES[:5])
        q0, dq0, tau = _chain_inputs(5, B, H, 52)
        roll = lambda a, b, c: rollout_np(ch, a, b, c, dt)
    w = _weights(ch.n, 53)
    tip = _tip(54)
    cost = lambda a, b, c: tip_cost_np(ch, a, b, c, dt, *roll(a, b, c), tip, **w)
    gt, gq, gdq = tip_cost_grad_np(ch, q0, dq0, tau, dt, *roll(q0, dq0, tau), tip, **w)
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


def test_tip_cost_rejects_unknown_keys():
    from rigidbody_rs_b200 import _tip_cost
    with pytest.raises(ValueError):
        _tip_cost({"w_q": 1.0})
    with pytest.raises(ValueError):
        _tip_cost({"p_ref": [1.0, 2.0]})


# ------------------------------------------------------------------------------------------------ on the B200
def _same_quadratic_bits(mb, q0, dq0, tau, dt, w):
    """tip=None and a tip of zero weights (but a target) both give rollout_cost's bits."""
    ref = mb.rollout_cost(q0, dq0, tau, dt, **w)
    zero = dict(offset=[0.1, 0.2, 0.3], p_ref=[1.0, 2.0, 3.0], R_ref=np.eye(3)[::-1], w_p=np.zeros(3), w_R=0.0)
    np.testing.assert_array_equal(mb.rollout_cost(q0, dq0, tau, dt, tip=None, **w), ref, err_msg=mb.kernel_variant)
    np.testing.assert_array_equal(mb.rollout_cost(q0, dq0, tau, dt, tip=zero, **w), ref, err_msg=mb.kernel_variant)


def _cost_close(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert np.isfinite(got).all()
    err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
    assert err.max() <= TOL, err.max()


@pytest.mark.gpu
def test_fr3_every_family(rb, oracle_fr3):
    """FR3 under every kernel family, B = 64, H = 16: cost and all three gradients against the checker; the gradient
    entry's cost is the cost entry's, bit for bit; the quadratic part alone is rollout_cost's, bit for bit."""
    from test_gpu_parity import _variants
    ch = _fr3_chain(oracle_fr3)
    B = 64
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H_, 0x5EED0061)
    w = _weights(7, 61)
    tip = _tip(62, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    traj = oracle_fr3.rollout_batch(q0, dq0, tau, DT)
    ref_cost = tip_cost_np(ch, q0, dq0, tau, DT, *traj, tip, **w)
    ref = tip_cost_grad_np(ch, q0, dq0, tau, DT, *traj, tip, **w)
    fams = []
    for mb in _variants(rb, FR3):
        fams.append(mb.kernel_variant)
        cost = mb.rollout_cost(q0, dq0, tau, DT, tip=tip, **w)
        _cost_close(cost, ref_cost)
        c2, gt, gq, gdq = mb.rollout_cost_grad(q0, dq0, tau, DT, tip=tip, **w)
        np.testing.assert_array_equal(c2, cost, err_msg=mb.kernel_variant)
        for got, want in zip((gt, gq, gdq), ref):
            _close(got, want)
        _same_quadratic_bits(mb, q0, dq0, tau, DT, w)
    assert fams == ["fr3-specialised", "jit-specialised", "generic-7", "generic-n"]


@pytest.mark.gpu
def test_chain32_every_family(rb, oracle_chain32):
    from test_gpu_parity import _variants
    from oracle.rb_oracle_np import ChainNP
    ch = ChainNP(oracle_chain32.model)
    B, H = 40, 6
    rng = np.random.default_rng(63)
    q0, dq0, tau = rng.uniform(-1, 1, (32, B)), rng.uniform(-0.5, 0.5, (32, B)), rng.uniform(-0.2, 0.2, (H, 32, B))
    w = _weights(32, 63)
    tip = _tip(64, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    ref = tip_cost_np(ch, q0, dq0, tau, DT, *rollout_np(ch, q0, dq0, tau, DT), tip, **w)
    fams = []
    for mb in _variants(rb, CHAIN32):
        fams.append(mb.kernel_variant)
        _cost_close(mb.rollout_cost(q0, dq0, tau, DT, tip=tip, **w), ref)
        _same_quadratic_bits(mb, q0, dq0, tau, DT, w)
    assert fams == ["chain32-specialised", "generic-n"]


@pytest.mark.gpu
@pytest.mark.parametrize("n,tree", [(1, False), (5, False), (12, False), (20, False), (40, False), (5, True), (20, True)])
def test_random_chains_and_trees_cost(rb, n, tree):
    mb, ch = _random(n, 300 + n, tree)
    B, H = 33, 9
    q0, dq0, tau = _chain_inputs(n, B, H, 310 + n)
    w = _weights(n, 320 + n)
    tip = _tip(330 + n)
    ref = tip_cost_np(ch, q0, dq0, tau, DT, *rollout_np(ch, q0, dq0, tau, DT), tip, **w)
    _cost_close(mb.rollout_cost(q0, dq0, tau, DT, tip=tip, **w), ref)
    _same_quadratic_bits(mb, q0, dq0, tau, DT, w)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 5, 12])
def test_random_chains_gradient(rb, n):
    mb, ch = _random(n, 400 + n)
    B = 48
    q0, dq0, tau = _chain_inputs(n, B, H_, 410 + n)
    w = _weights(n, 420 + n)
    tip = _tip(430 + n)
    qt, dqt = mb.rollout(q0, dq0, tau, DT)            # the checker linearises about the engine's trajectory, the twin's to rounding
    assert max(_per_traj_err(a, b).max() for a, b in zip((qt, dqt), rollout_np(ch, q0, dq0, tau, DT))) < TOL
    cost, *got = mb.rollout_cost_grad(q0, dq0, tau, DT, tip=tip, **w)
    _cost_close(cost, tip_cost_np(ch, q0, dq0, tau, DT, qt, dqt, tip, **w))
    np.testing.assert_array_equal(cost, mb.rollout_cost(q0, dq0, tau, DT, tip=tip, **w))
    for a, b in zip(got, tip_cost_grad_np(ch, q0, dq0, tau, DT, qt, dqt, tip, **w)):
        _close(a, b)


@pytest.mark.gpu
def test_autograd_gradcheck(rb, mb_fr3, oracle_fr3):
    import torch
    q0, dq0, tau = _fr3_inputs(oracle_fr3, 3, 3, 0x5EED0065)
    ch = _fr3_chain(oracle_fr3)
    tip = _tip(65, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    w = dict(w_q=np.ones(7), w_tau=np.full(7, 1e-3))
    ins = [x.requires_grad_(True) for x in _dev(q0, dq0, tau)]
    f = lambda a, b, c: mb_fr3.rollout_cost_autograd(a, b, c, 1e-2, tip=tip, **w)
    assert torch.autograd.gradcheck(f, ins)
    cost = f(*ins)
    np.testing.assert_array_equal(cost.detach().cpu().numpy(), mb_fr3.rollout_cost(q0, dq0, tau, 1e-2, tip=tip, **w))
    cost.sum().backward()                                  # a torch optimiser's step: the gradient of the summed cost
    _, gt, gq, gdq = mb_fr3.rollout_cost_grad(q0, dq0, tau, 1e-2, tip=tip, **w)
    for x, want in zip(ins, (gq, gdq, gt)):
        np.testing.assert_array_equal(x.grad.cpu().numpy(), want)
    with torch.no_grad():
        c = mb_fr3.rollout_cost_autograd(*_dev(q0, dq0, tau), 1e-2, tip=tip, **w)
    np.testing.assert_array_equal(c.cpu().numpy(), cost.detach().cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("H", [0, 1, 33])
def test_layouts_memory_and_leading_dimension(rb, mb_fr3, oracle_fr3, H):
    """Host against device and SoA against AoS bit for bit, and a NaN-padded leading dimension through the C ABI."""
    from rigidbody_rs_b200 import _lib, _tip_cost
    lib = _lib.lib
    mb = mb_fr3
    B = 129
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H, 0x5EED0066)
    w = _weights(7, 66)
    tip = _tip(66)
    host = mb.rollout_cost_grad(q0, dq0, tau, DT, tip=tip, **w)
    dev = _np(*mb.rollout_cost_grad(*_dev(q0, dq0, tau), DT, tip=tip, **w))
    aos = mb.rollout_cost_grad(_aos(q0), _aos(dq0), _aos(tau), DT, layout="aos", tip=tip, **w)
    aos_dev = _np(*mb.rollout_cost_grad(*_dev(_aos(q0), _aos(dq0), _aos(tau)), DT, layout="aos", tip=tip, **w))
    for k in range(4):
        np.testing.assert_array_equal(dev[k], host[k])
        np.testing.assert_array_equal(aos[k], host[k] if k == 0 else _aos(host[k]))
        np.testing.assert_array_equal(aos_dev[k], aos[k])
    for c in (mb.rollout_cost(q0, dq0, tau, DT, tip=tip, **w), _np(mb.rollout_cost(*_dev(q0, dq0, tau), DT, tip=tip, **w))[0],
              mb.rollout_cost(_aos(q0), _aos(dq0), _aos(tau), DT, layout="aos", tip=tip, **w)):
        np.testing.assert_array_equal(c, host[0])
    ch = _fr3_chain(oracle_fr3)
    traj = oracle_fr3.rollout_batch(q0, dq0, tau, DT) if H else (np.zeros((0, 7, B)), np.zeros((0, 7, B)))
    _cost_close(host[0], tip_cost_np(ch, q0, dq0, tau, DT, *traj, tip, **w))
    if H == 0:
        _close(host[2], tip_grad_np(ch, q0, tip, 0.0, 1.0) + 2 * w["w_q_final"][:, None] * (q0 - w["q_ref"][:, None]))
    ld = B + 31
    nan = float("nan")
    p = lambda x: C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data) if x is not None else None
    qc, keep = mb._quad_cost(**w)
    tc, keep_tip = _tip_cost(tip)
    for mem in (_lib.RB_MEM_DEVICE, _lib.RB_MEM_HOST):
        def wide(x):
            wd = np.full(x.shape[:-1] + (ld,), nan)
            wd[..., :B] = x
            return _dev(wd)[0] if mem == _lib.RB_MEM_DEVICE else wd
        back = lambda x: x.cpu().numpy() if mem == _lib.RB_MEM_DEVICE else x
        wq, wdq, wtau = (wide(x) for x in (q0, dq0, tau))
        cost, gt, gq, gdq = wide(np.full((1, B), nan))[0], wide(np.full((H, 7, B), nan)), wide(np.full((7, B), nan)), wide(np.full((7, B), nan))
        rc = lib.multibody_rollout_tip_cost_grad(mb._h, p(wq), p(wdq), p(wtau), DT, H, C.byref(qc), C.byref(tc), p(cost), p(gt), p(gq),
                                                 p(gdq), B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(cost)[:B], host[0])
        for got, want in zip((gt, gq, gdq), host[1:]):
            g = back(got)
            np.testing.assert_array_equal(g[..., :B], want)
            assert np.isnan(g[..., B:]).all()
        cost = wide(np.full((1, B), nan))[0]
        rc = lib.multibody_rollout_tip_cost(mb._h, p(wq), p(wdq), p(wtau), DT, H, C.byref(qc), C.byref(tc), p(cost), None, None,
                                            B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(cost)[:B], host[0])


@pytest.mark.gpu
def test_gradient_in_chunks_equals_one_chunk(rb, mb_fr3, oracle_fr3):
    """A batch whose trajectory workspace exceeds one chunk (H = 1000, 10 000 trajectories) gives, per trajectory, the
    bits of a batch small enough for one chunk."""
    import torch
    mb = mb_fr3
    B, H, dt = 10_000, 1000, 1e-3
    q0, dq0, _ = _fr3_inputs(oracle_fr3, B, 0, 0x5EED0067)
    gen = torch.Generator(device="cuda:0").manual_seed(67)
    eff = torch.from_numpy(oracle_fr3.model.effort).to("cuda:0")[None, :, None]
    tau = (torch.rand((H, 7, B), dtype=torch.float64, device="cuda:0", generator=gen) * 2 - 1) * 0.2 * eff
    w = _weights(7, 67)
    tip = _tip(67)
    tq, tdq = _dev(q0, dq0)
    full = mb.rollout_cost_grad(tq, tdq, tau, dt, tip=tip, **w)
    for lo, hi in ((0, 100), (B - 100, B)):
        part = mb.rollout_cost_grad(tq[:, lo:hi].contiguous(), tdq[:, lo:hi].contiguous(), tau[..., lo:hi].contiguous(), dt, tip=tip, **w)
        for a, b in zip(full, part):
            np.testing.assert_array_equal(a[..., lo:hi].cpu().numpy(), b.cpu().numpy())
    assert all(bool(torch.isfinite(x).all()) for x in full)


@pytest.mark.gpu
def test_multi_device_equals_single_device(rb, mb_fr3, oracle_fr3):
    from test_gpu_parity import _two_devices
    mm = rb.Multibody.from_urdf(FR3, devices=_two_devices())
    B = 301
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, 12, 0x5EED0068)
    w = _weights(7, 68)
    tip = _tip(68)
    for layout, f in (("soa", lambda x: x), ("aos", _aos)):
        for call in ("rollout_cost", "rollout_cost_grad"):
            a = getattr(mm, call)(f(q0), f(dq0), f(tau), DT, layout=layout, tip=tip, **w)
            b = getattr(mb_fr3, call)(f(q0), f(dq0), f(tau), DT, layout=layout, tip=tip, **w)
            for x, y in zip(a if call != "rollout_cost" else [a], b if call != "rollout_cost" else [b]):
                np.testing.assert_array_equal(x, y)
    with pytest.raises(rb.RigidBodyError) as ei:
        mm.rollout_cost_grad(*_dev(q0, dq0, tau), DT, tip=tip, **w)
    assert ei.value.code == -6
    mm.close()


@pytest.mark.gpu
def test_errors_and_unsupported_chains(rb, mb_fr3):
    from rigidbody_rs_b200 import _lib, _tip_cost
    lib = _lib.lib
    z = lambda n, B=4, H=2: (np.zeros((n, B)), np.zeros((n, B)), np.zeros((H, n, B)))
    tip = _tip(69)
    for mb in (_random(13, 69)[0], _random(6, 70, tree=True)[0]):
        q0, dq0, tau = z(mb.n)
        with pytest.raises(rb.RigidBodyError) as ei:
            mb.rollout_cost_grad(q0, dq0, tau, DT, tip=tip)
        assert ei.value.code == _lib.RB_ERR_UNSUPPORTED
        assert np.isfinite(mb.rollout_cost(q0, dq0, tau, DT, tip=tip)).all()     # the cost itself serves them
    mb = mb_fr3
    q0, dq0, tau = z(7)
    p = lambda a: C.c_void_p(a.ctypes.data)
    cost, gt, gq, gdq = np.zeros(4), np.zeros((2, 7, 4)), np.zeros((7, 4)), np.zeros((7, 4))
    cg = lambda tc, cst: lib.multibody_rollout_tip_cost_grad(mb._h, p(q0), p(dq0), p(tau), DT, 2, None, tc, cst, p(gt), p(gq), p(gdq), 4, 0, 0, 0, None)
    co = lambda tc, cst: lib.multibody_rollout_tip_cost(mb._h, p(q0), p(dq0), p(tau), DT, 2, None, tc, cst, None, None, 4, 0, 0, 0, None)
    good, keep = _tip_cost(tip)
    for f in (cg, co):
        assert f(C.byref(good), p(cost)) == 0
        assert f(C.byref(good), None) == _lib.RB_ERR_NULL
        assert f(None, p(cost)) == 0                                              # no tip terms, no quadratic terms
        np.testing.assert_array_equal(cost, 0.0)
        for bad in (dict(w_p=[1.0, -1.0, 0.0]), dict(w_p_final=[0.0, np.inf, 0.0]), dict(w_R=-1.0), dict(w_R_final=np.nan),
                    dict(p_ref=[0.0, np.nan, 0.0]), dict(offset=[np.inf, 0.0, 0.0]), dict(R_ref=np.full(9, np.nan))):
            tc, keep_bad = _tip_cost(bad)
            assert f(C.byref(tc), p(cost)) == _lib.RB_ERR_ARG, bad


@pytest.mark.gpu
def test_not_spd_gives_nan_for_the_bad_trajectories_only(rb):
    from test_rollout_gradients import _spd_where_q1_small
    mb = _spd_where_q1_small(rb)
    B, H = 6, 3
    q0 = np.zeros((2, B)); q0[1, 1::2] = 1.5
    dq0, tau = np.zeros((2, B)), np.zeros((H, 2, B))
    w = dict(q_ref=np.full(2, 0.3), w_q=np.ones(2))
    tip = dict(offset=[0.1, 0.0, 0.0], p_ref=[0.0, 0.1, 0.0], w_p=np.ones(3), w_R=0.5, w_R_final=1.0)
    with pytest.raises(rb.NotPositiveDefinite):
        mb.rollout_cost_grad(q0, dq0, tau, 1e-3, tip=tip, **w)
    from rigidbody_rs_b200 import _lib, _tip_cost
    lib = _lib.lib
    qc, keep = mb._quad_cost(**w)
    tc, keep_tip = _tip_cost(tip)
    cost, gt, gq, gdq = np.zeros(B), np.zeros((H, 2, B)), np.zeros((2, B)), np.zeros((2, B))
    p = lambda a: C.c_void_p(a.ctypes.data)
    rc = lib.multibody_rollout_tip_cost_grad(mb._h, p(q0), p(dq0), p(tau), 1e-3, H, C.byref(qc), C.byref(tc), p(cost), p(gt), p(gq), p(gdq),
                                             B, 0, 0, 0, None)
    assert rc == _lib.RB_ERR_NOT_SPD
    for g in (cost, gt, gq, gdq):
        assert np.isnan(g[..., 1::2]).all() and np.isfinite(g[..., 0::2]).all()
    good = mb.rollout_cost_grad(q0[:, 0::2].copy(), dq0[:, 0::2].copy(), tau[..., 0::2].copy(), 1e-3, tip=tip, **w)
    for a, b in zip((cost, gt, gq, gdq), good):
        np.testing.assert_array_equal(a[..., 0::2], b)


@pytest.mark.gpu
def test_full_size_fr3_65536x64(rb, mb_fr3, oracle_fr3):
    """65 536 trajectories x 64 steps, device-resident: cost and gradients finite, the gradient entry's cost the cost
    entry's bits, and 128 strided trajectories against the checker."""
    import torch
    mb = mb_fr3
    B, H, dt = 65536, 64, 1e-3
    lim = oracle_fr3.model
    q0, dq0, _ = _fr3_inputs(oracle_fr3, B, 0, 0x5EED0070)
    rng = np.random.default_rng(70)
    tau = rng.uniform(-0.3, 0.3, (H, 7, B)) * lim.effort[None, :, None]
    w = _weights(7, 70)
    ch = _fr3_chain(oracle_fr3)
    tip = _tip(70, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    d = _dev(q0, dq0, tau)
    cost = mb.rollout_cost(*d, dt, tip=tip, **w)
    res = mb.rollout_cost_grad(*d, dt, tip=tip, **w)
    assert all(bool(torch.isfinite(x).all()) for x in res)
    np.testing.assert_array_equal(res[0].cpu().numpy(), cost.cpu().numpy())
    got = [x.cpu().numpy() for x in res]
    del d, res
    torch.cuda.empty_cache()
    idx = np.arange(0, B, B // 128)
    s0, s1, st = q0[:, idx].copy(), dq0[:, idx].copy(), tau[..., idx].copy()
    traj = oracle_fr3.rollout_batch(s0, s1, st, dt)
    _cost_close(got[0][idx], tip_cost_np(ch, s0, s1, st, dt, *traj, tip, **w))
    for g, want in zip(got[1:], tip_cost_grad_np(ch, s0, s1, st, dt, *traj, tip, **w)):
        _close(g[..., idx], want)
