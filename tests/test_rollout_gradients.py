"""Gradients of rollouts (include/rigidbody.h multibody_rollout_vjp / multibody_rollout_cost_grad).

The checker is rollout_vjp_np below: the backward recursion built on the numpy twin (oracle/rb_oracle_np.py:
complex-step derivatives of the link-frame rnea and the inverse of the twin's crba at every step), not the world-frame
closed forms the CUDA kernel uses; the CPU test holds the checker itself against central finite differences of the
rollout cost.  Bar on the GPU, as for the per-state derivatives: |err| <= 1e-10 * max(1, max|ref|) per trajectory.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import CHAIN32, FR3, TOL

# ------------------------------------------------------------------------------------------------ the numpy checker
# The backward recursion written out with the twin's per-state derivatives (oracle/rb_oracle_np.py ChainNP).
# Layouts as the engine's SoA: q0, dq0 [n, B]; tau and trajectories [H, n, B].  Weights: length-n vectors (None = 0).
def rollout_np(chain, q0, dq0, tau, dt):
    """The engine's semi-implicit Euler rollout (dq += dt qdd; q += dt dq) through the twin's forward dynamics:
    (q_traj, dq_traj), the states after each step."""
    q, dq = np.array(q0, dtype=np.float64).T, np.array(dq0, dtype=np.float64).T
    qt, dqt = [], []
    for t in range(tau.shape[0]):
        dq = dq + dt * chain.forward_dynamics(q, dq, tau[t].T)
        q = q + dt * dq
        qt.append(q.T); dqt.append(dq.T)
    n, B = np.shape(q0)
    return (np.stack(qt), np.stack(dqt)) if qt else (np.zeros((0, n, B)), np.zeros((0, n, B)))


def rollout_vjp_np(chain, q0, dq0, tau, dt, q_traj, dq_traj, g_q_traj=None, g_dq_traj=None, g_q_final=None, g_dq_final=None):
    """Reverse-mode product of the rollout about the given trajectory, with `ChainNP.fd_derivatives` (complex-step
    differentiation of the link-frame rnea, inverse of the twin's crba) at every step:
        a_q = Gqf + Gq[H-1];  a_dq = Gdqf + Gdq[H-1]
        for t = H-1 .. 0:  b = a_dq + dt a_q;  lam = dt b (the adjoint of qdd_t)
            grad_tau[t] = H^-1 lam;  a_q += (d qdd / d q)^T lam;  a_dq = b + (d qdd / d dq)^T lam
            t > 0: a_q += Gq[t-1];  a_dq += Gdq[t-1]
    Returns (grad_tau, grad_q0, grad_dq0)."""
    H = tau.shape[0]
    z = np.zeros(np.shape(q0))
    up = lambda g, t: z if g is None else np.asarray(g[t], dtype=np.float64)
    a_q = (z if g_q_final is None else np.asarray(g_q_final, dtype=np.float64)) + (up(g_q_traj, H - 1) if H else z)
    a_dq = (z if g_dq_final is None else np.asarray(g_dq_final, dtype=np.float64)) + (up(g_dq_traj, H - 1) if H else z)
    grad_tau = np.zeros(np.shape(tau))
    for t in range(H - 1, -1, -1):
        q, dq = (q_traj[t - 1], dq_traj[t - 1]) if t else (q0, dq0)
        Aq, Av, Mi = chain.fd_derivatives(np.asarray(q).T, np.asarray(dq).T, np.asarray(tau[t]).T)     # [B, n, n] each
        b = a_dq + dt * a_q
        lam = dt * b
        grad_tau[t] = np.einsum("bij,ib->jb", Mi, lam)
        a_q = a_q + np.einsum("bij,ib->jb", Aq, lam)
        a_dq = b + np.einsum("bij,ib->jb", Av, lam)
        if t:
            a_q = a_q + up(g_q_traj, t - 1)
            a_dq = a_dq + up(g_dq_traj, t - 1)
    return grad_tau, a_q, a_dq


def _w(v, n):
    return np.zeros(n) if v is None else np.broadcast_to(np.asarray(v, dtype=np.float64), (n,))


def quad_cost_np(q0, dq0, tau, dt, q_traj, dq_traj, q_ref=None, w_q=None, w_dq=None, w_tau=None, w_q_final=None, w_dq_final=None):
    """The quadratic cost of multibody_rollout_cost (include/rigidbody.h RbQuadCost) of a stored trajectory: [B]."""
    n = np.shape(q0)[0]
    c = lambda v: _w(v, n)[:, None]
    qH, dqH = (q_traj[-1], dq_traj[-1]) if tau.shape[0] else (q0, dq0)
    run = sum(dt * ((c(w_q) * (q_traj[t] - c(q_ref)) ** 2).sum(0) + (c(w_dq) * dq_traj[t] ** 2).sum(0) + (c(w_tau) * tau[t] ** 2).sum(0))
              for t in range(tau.shape[0]))
    return run + (c(w_q_final) * (qH - c(q_ref)) ** 2).sum(0) + (c(w_dq_final) * dqH ** 2).sum(0)


def quad_cost_upstream(q0, dq0, dt, q_traj, dq_traj, q_ref=None, w_q=None, w_dq=None, w_q_final=None, w_dq_final=None):
    """Gradients of that cost with respect to the rollout's outputs (g_q_traj, g_dq_traj, g_q_final, g_dq_final):
    Gq[t] = 2 dt w_q (q_{t+1} - q_ref),  Gdq[t] = 2 dt w_dq dq_{t+1},  Gqf = 2 w_q_final (q_H - q_ref),  Gdqf = 2 w_dq_final dq_H."""
    n = np.shape(q0)[0]
    c = lambda v: _w(v, n)[:, None]
    qH, dqH = (q_traj[-1], dq_traj[-1]) if len(q_traj) else (q0, dq0)
    return (2.0 * dt * c(w_q)[None] * (q_traj - c(q_ref)[None]), 2.0 * dt * c(w_dq)[None] * dq_traj,
            2.0 * c(w_q_final) * (qH - c(q_ref)), 2.0 * c(w_dq_final) * dqH)


def rollout_cost_grad_np(chain, q0, dq0, tau, dt, q_traj, dq_traj, q_ref=None, w_q=None, w_dq=None, w_tau=None, w_q_final=None,
                         w_dq_final=None):
    """(grad_tau, grad_q0, grad_dq0) of quad_cost_np: rollout_vjp_np with quad_cost_upstream, plus 2 dt w_tau tau."""
    up = quad_cost_upstream(q0, dq0, dt, q_traj, dq_traj, q_ref, w_q, w_dq, w_q_final, w_dq_final)
    gt, gq, gdq = rollout_vjp_np(chain, q0, dq0, tau, dt, q_traj, dq_traj, *up)
    return gt + 2.0 * dt * _w(w_tau, np.shape(q0)[0])[None, :, None] * tau, gq, gdq


H_, DT = 16, 2e-3
NAMES = ("q_ref", "w_q", "w_dq", "w_tau", "w_q_final", "w_dq_final")


def _weights(n, seed):
    rng = np.random.default_rng(seed)
    return dict(q_ref=rng.uniform(-1, 1, n), w_q=rng.uniform(0, 2, n), w_dq=rng.uniform(0, 1, n), w_tau=rng.uniform(0, 1e-3, n),
                w_q_final=rng.uniform(0, 50, n), w_dq_final=rng.uniform(0, 5, n))


def _fr3_inputs(orc, B, H, seed):
    lim = orc.model
    q = orc.fill(seed, 0, lim.lower, lim.upper, 0, B)
    dq = orc.fill(seed, 1, -lim.velocity, lim.velocity, 0, B)
    tau = np.stack([orc.fill(seed, 4 + t, -lim.effort, lim.effort, t * B, B) for t in range(H)]) if H else np.zeros((0, 7, B))
    return q, dq, tau


def _chain_inputs(n, B, H, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-2, 2, (n, B)), rng.uniform(-1, 1, (n, B)), rng.uniform(-1, 1, (H, n, B))


def _per_traj_err(got, ref):
    """max over everything but the trajectory axis (last), relative to max(1, max|ref|) of that trajectory."""
    got, ref = np.asarray(got), np.asarray(ref)
    ax = tuple(range(got.ndim - 1))
    return np.abs(got - ref).max(ax) / np.maximum(1.0, np.abs(ref).max(ax))


def _close(got, ref, bar=TOL):
    err = _per_traj_err(got, ref)
    assert np.isfinite(np.asarray(got)).all()
    assert err.max() <= bar, err.max()


# ------------------------------------------------------------------------------------------------ the checker, on the CPU
@pytest.mark.parametrize("chain", ["fr3", "random5"])
def test_numpy_vjp_matches_finite_differences_of_the_cost(oracle_fr3, chain):
    """rollout_vjp_np (through rollout_cost_grad_np) against central differences of the rollout's quadratic cost, every
    component of tau, q0 and dq0; H = 8.  The bar is the O(h^2) truncation plus rounding of the difference quotient."""
    from oracle.rb_oracle_np import ChainNP
    H, B, dt = 8, 3, 1e-2
    if chain == "fr3":
        ch = ChainNP(oracle_fr3.model)
        q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H, 0x5EED0031)
        roll = lambda a, b, c: oracle_fr3.rollout_batch(a, b, c, dt)
    else:
        from test_host import _random_chain, AXES
        R, t, m, c, Ic = _random_chain(5, 51)
        ch = ChainNP.from_arrays(R, t, m, c, Ic, axis=AXES[:5])
        q0, dq0, tau = _chain_inputs(5, B, H, 52)
        roll = lambda a, b, c: rollout_np(ch, a, b, c, dt)
    n = ch.n
    w = _weights(n, 53)
    cost = lambda a, b, c: quad_cost_np(a, b, c, dt, *roll(a, b, c), **w)
    gt, gq, gdq = rollout_cost_grad_np(ch, q0, dq0, tau, dt, *roll(q0, dq0, tau), **w)
    args = [q0, dq0, tau]
    for k, g in enumerate((gq, gdq, gt)):
        x = args[k]
        fd = np.zeros_like(x)
        for idx in np.ndindex(x.shape[:-1]):              # every component, all trajectories at once
            h = 1e-6 * max(1.0, np.abs(x[idx]).max())
            up, dn = [a.copy() for a in args], [a.copy() for a in args]
            up[k][idx] += h; dn[k][idx] -= h
            fd[idx] = (cost(*up) - cost(*dn)) / (2 * h)
        err = np.abs(fd - g).max() / max(1.0, np.abs(g).max())
        assert err < 1e-6, (chain, ("q0", "dq0", "tau")[k], err)


# ------------------------------------------------------------------------------------------------ on the B200
def _dev(*xs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(x)).to("cuda:0") for x in xs]


def _np(*xs):
    return [x.cpu().numpy() for x in xs]


def _aos(x):
    """SoA [.., n, B] -> AoS [.., B, n]."""
    return np.ascontiguousarray(np.swapaxes(x, -1, -2))


@pytest.mark.gpu
def test_cost_grad_fr3_every_family(rb, oracle_fr3):
    """FR3 under every kernel family, B = 64, H = 16: all three gradients against the numpy twin, and the cost the same
    bits as rollout_cost on the same engine."""
    from test_gpu_parity import _variants
    from oracle.rb_oracle_np import ChainNP
    B = 64
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H_, 0x5EED0041)
    w = _weights(7, 41)
    ref = rollout_cost_grad_np(ChainNP(oracle_fr3.model), q0, dq0, tau, DT, *oracle_fr3.rollout_batch(q0, dq0, tau, DT), **w)
    fams = []
    for mb in _variants(rb, FR3):
        fams.append(mb.kernel_variant)
        cost, gt, gq, gdq = mb.rollout_cost_grad(q0, dq0, tau, DT, **w)
        np.testing.assert_array_equal(cost, mb.rollout_cost(q0, dq0, tau, DT, **w), err_msg=mb.kernel_variant)
        for got, want in zip((gt, gq, gdq), ref):
            _close(got, want)
    assert fams == ["fr3-specialised", "jit-specialised", "generic-7", "generic-n"]


@pytest.mark.gpu
def test_vjp_is_model_agnostic_and_agrees_with_cost_grad(rb, oracle_fr3):
    """The adjoint kernel is the same code under every family: rollout_vjp of one trajectory gives the same bits
    everywhere.  With the quadratic cost's upstream gradients formed in numpy (plus the direct w_tau term) it agrees
    with cost_grad to 1e-12 relative."""
    from test_gpu_parity import _variants
    B = 64
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H_, 0x5EED0042)
    w = _weights(7, 42)
    mbs = _variants(rb, FR3)
    qt, dqt = mbs[0].rollout(q0, dq0, tau, DT)
    up = quad_cost_upstream(q0, dq0, DT, qt, dqt, w["q_ref"], w["w_q"], w["w_dq"], w["w_q_final"], w["w_dq_final"])
    first = None
    for mb in mbs:
        got = mb.rollout_vjp(q0, dq0, tau, DT, qt, dqt, *up)
        if first is None:
            first = got
        for a, b in zip(got, first):
            np.testing.assert_array_equal(a, b, err_msg=mb.kernel_variant)
    _, gt, gq, gdq = mbs[0].rollout_cost_grad(q0, dq0, tau, DT, **w)
    gt_vjp = first[0] + 2.0 * DT * w["w_tau"][None, :, None] * tau
    for got, want in ((gt, gt_vjp), (gq, first[1]), (gdq, first[2])):
        assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 5, 12])
def test_random_chains_oblique_axes(rb, n):
    from test_host import _random_chain, AXES
    from oracle.rb_oracle_np import ChainNP
    R, t, m, c, Ic = _random_chain(n, 60 + n)
    ax = (AXES + AXES)[:n]
    mb = rb.Multibody.from_descriptor(R, t, m, c, Ic, axis=ax)
    ch = ChainNP.from_arrays(R, t, m, c, Ic, axis=ax)
    B = 48
    q0, dq0, tau = _chain_inputs(n, B, H_, 70 + n)
    qt, dqt = mb.rollout(q0, dq0, tau, DT)           # both sides linearise about the engine's trajectory ...
    twin = rollout_np(ch, q0, dq0, tau, DT)          # ... which is the twin's to rounding
    assert max(_per_traj_err(a, b).max() for a, b in zip((qt, dqt), twin)) < TOL
    rng = np.random.default_rng(n)
    up = (rng.normal(size=qt.shape), rng.normal(size=qt.shape), rng.normal(size=q0.shape), rng.normal(size=q0.shape))
    got = mb.rollout_vjp(q0, dq0, tau, DT, qt, dqt, *up)
    for a, b in zip(got, rollout_vjp_np(ch, q0, dq0, tau, DT, qt, dqt, *up)):
        _close(a, b)
    w = _weights(n, 80 + n)
    _, *got = mb.rollout_cost_grad(q0, dq0, tau, DT, **w)
    for a, b in zip(got, rollout_cost_grad_np(ch, q0, dq0, tau, DT, qt, dqt, **w)):
        _close(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [0, 1, 33])
def test_layouts_memory_and_leading_dimension(rb, mb_fr3, oracle_fr3, H):
    """Host against device and SoA against AoS bit for bit, NaN-padded ld views (padding untouched), n_traj = 129 (a
    ragged block), NULL upstream gradients and NULL outputs."""
    import torch
    from rigidbody_rs_b200 import _lib
    lib = _lib.lib
    mb = mb_fr3
    B = 129
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, H, 0x5EED0043)
    w = _weights(7, 43)
    qt, dqt = mb.rollout(q0, dq0, tau, DT)
    rng = np.random.default_rng(H)
    up = [rng.normal(size=qt.shape), rng.normal(size=qt.shape), rng.normal(size=q0.shape), rng.normal(size=q0.shape)]
    # cost_grad
    host = mb.rollout_cost_grad(q0, dq0, tau, DT, **w)
    dev = _np(*mb.rollout_cost_grad(*_dev(q0, dq0, tau), DT, **w))
    aos = mb.rollout_cost_grad(_aos(q0), _aos(dq0), _aos(tau), DT, layout="aos", **w)
    aos_dev = _np(*mb.rollout_cost_grad(*_dev(_aos(q0), _aos(dq0), _aos(tau)), DT, layout="aos", **w))
    for k in range(4):
        np.testing.assert_array_equal(dev[k], host[k])
        np.testing.assert_array_equal(aos[k], host[k] if k == 0 else _aos(host[k]))
        np.testing.assert_array_equal(aos_dev[k], aos[k])
    if H == 0:                                                 # grad = d terminal cost / d (q0, dq0)
        np.testing.assert_array_equal(host[1], np.zeros((0, 7, B)))
        np.testing.assert_allclose(host[2], 2 * w["w_q_final"][:, None] * (q0 - w["q_ref"][:, None]), rtol=1e-15)
        np.testing.assert_allclose(host[3], 2 * w["w_dq_final"][:, None] * dq0, rtol=1e-15)
    # vjp
    vh = mb.rollout_vjp(q0, dq0, tau, DT, qt, dqt, *up)
    vd = _np(*mb.rollout_vjp(*_dev(q0, dq0, tau), DT, *_dev(qt, dqt, *up)))
    va = mb.rollout_vjp(_aos(q0), _aos(dq0), _aos(tau), DT, _aos(qt), _aos(dqt), *[_aos(u) for u in up], layout="aos")
    for k in range(3):
        np.testing.assert_array_equal(vd[k], vh[k])
        np.testing.assert_array_equal(va[k], _aos(vh[k]))
    if H == 0:
        np.testing.assert_array_equal(vh[1], up[2])
        np.testing.assert_array_equal(vh[2], up[3])
    # NULL upstream = zero upstream; only the final-state gradient given
    zero = [np.zeros_like(u) for u in up]
    a = mb.rollout_vjp(q0, dq0, tau, DT, qt, dqt, None, None, up[2], None)
    b = mb.rollout_vjp(q0, dq0, tau, DT, qt, dqt, zero[0], zero[1], up[2], zero[3])
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    # NaN-padded leading dimension through the C ABI, device and host; NULL outputs leave their buffers alone
    ld = B + 31
    nan = float("nan")
    p = lambda x: C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data) if x is not None else None
    for mem in (_lib.RB_MEM_DEVICE, _lib.RB_MEM_HOST):
        def wide(x):
            wd = np.full(x.shape[:-1] + (ld,), nan)
            wd[..., :B] = x
            return _dev(wd)[0] if mem == _lib.RB_MEM_DEVICE else wd
        blank = lambda *shape: wide(np.full(shape, nan))
        back = lambda x: x.cpu().numpy() if mem == _lib.RB_MEM_DEVICE else x
        wq, wdq, wtau, wqt, wdqt = (wide(x) for x in (q0, dq0, tau, qt, dqt))
        wup = [wide(u) for u in up]
        cost, gt, gq, gdq = blank(1, B)[0], blank(H, 7, B), blank(7, B), blank(7, B)     # cost: n_traj doubles, no ld
        qc, keep = mb._quad_cost(**w)
        rc = lib.multibody_rollout_cost_grad(mb._h, p(wq), p(wdq), p(wtau), DT, H, C.byref(qc), p(cost), p(gt), p(gq), p(gdq),
                                             B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(cost)[:B], host[0])
        for got, want in zip((gt, gq, gdq), host[1:]):
            g = back(got)
            np.testing.assert_array_equal(g[..., :B], want)
            assert np.isnan(g[..., B:]).all()
        gt, gq, gdq = blank(H, 7, B), blank(7, B), blank(7, B)
        rc = lib.multibody_rollout_vjp(mb._h, p(wq), p(wdq), p(wtau), DT, H, p(wqt), p(wdqt), *[p(u) for u in wup], p(gt), None, p(gdq),
                                       B, ld, _lib.RB_LAYOUT_SOA, mem, None)
        assert rc == 0, lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(gt)[..., :B], vh[0])
        assert np.isnan(back(gq)).all()
        np.testing.assert_array_equal(back(gdq)[..., :B], vh[2])
        assert np.isnan(back(gt)[..., B:]).all() and np.isnan(back(gdq)[..., B:]).all()


@pytest.mark.gpu
def test_cost_grad_in_chunks_equals_one_chunk(rb, mb_fr3, oracle_fr3):
    """A batch whose trajectory workspace exceeds one chunk (H = 1000, 10 000 trajectories: 1.1 GB) is cut into
    chunks; every trajectory's results equal those of a batch small enough for one chunk, bit for bit."""
    import torch
    mb = mb_fr3
    B, H, dt = 10_000, 1000, 1e-3
    lim = oracle_fr3.model
    q0, dq0, _ = _fr3_inputs(oracle_fr3, B, 0, 0x5EED0044)
    gen = torch.Generator(device="cuda:0").manual_seed(44)
    eff = torch.from_numpy(lim.effort).to("cuda:0")[None, :, None]
    tau = (torch.rand((H, 7, B), dtype=torch.float64, device="cuda:0", generator=gen) * 2 - 1) * 0.2 * eff
    w = _weights(7, 44)
    tq, tdq = _dev(q0, dq0)
    full = mb.rollout_cost_grad(tq, tdq, tau, dt, **w)
    for lo, hi in ((0, 100), (B - 100, B)):
        part = mb.rollout_cost_grad(tq[:, lo:hi].contiguous(), tdq[:, lo:hi].contiguous(), tau[..., lo:hi].contiguous(), dt, **w)
        for a, b in zip(full, part):
            np.testing.assert_array_equal(a[..., lo:hi].cpu().numpy(), b.cpu().numpy())
    assert all(bool(torch.isfinite(x).all()) for x in full)


@pytest.mark.gpu
def test_autograd_gradcheck(rb, mb_fr3, oracle_fr3):
    import torch
    q0, dq0, tau = _fr3_inputs(oracle_fr3, 3, 3, 0x5EED0045)
    ins = [x.requires_grad_(True) for x in _dev(q0, dq0, tau)]
    assert torch.autograd.gradcheck(lambda a, b, c: mb_fr3.rollout_autograd(a, b, c, 1e-2), ins)
    qt, dqt = mb_fr3.rollout_autograd(*ins, 1e-2)
    np.testing.assert_array_equal(qt.detach().cpu().numpy(), mb_fr3.rollout(q0, dq0, tau, 1e-2)[0])


@pytest.mark.gpu
def test_multi_device_equals_single_device(rb, mb_fr3, oracle_fr3):
    import torch
    from test_gpu_parity import _two_devices
    mm = rb.Multibody.from_urdf(FR3, devices=_two_devices())
    B = 301
    q0, dq0, tau = _fr3_inputs(oracle_fr3, B, 12, 0x5EED0046)
    w = _weights(7, 46)
    qt, dqt = mb_fr3.rollout(q0, dq0, tau, DT)
    up = [np.random.default_rng(46).normal(size=s) for s in (qt.shape, qt.shape, q0.shape, q0.shape)]
    for layout, f in (("soa", lambda x: x), ("aos", _aos)):
        a = mm.rollout_cost_grad(f(q0), f(dq0), f(tau), DT, layout=layout, **w)
        b = mb_fr3.rollout_cost_grad(f(q0), f(dq0), f(tau), DT, layout=layout, **w)
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)
        a = mm.rollout_vjp(f(q0), f(dq0), f(tau), DT, f(qt), f(dqt), *[f(u) for u in up], layout=layout)
        b = mb_fr3.rollout_vjp(f(q0), f(dq0), f(tau), DT, f(qt), f(dqt), *[f(u) for u in up], layout=layout)
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)
    for call in (lambda: mm.rollout_cost_grad(*_dev(q0, dq0, tau), DT, **w),
                 lambda: mm.rollout_vjp(*_dev(q0, dq0, tau), DT, *_dev(qt, dqt))):
        with pytest.raises(rb.RigidBodyError) as ei:
            call()
        assert ei.value.code == -6
    mm.close()


@pytest.mark.gpu
def test_errors_and_unsupported_chains(rb, mb_fr3, oracle_fr3):
    from rigidbody_rs_b200 import _lib
    from test_host import _random_chain, _random_tree
    lib = _lib.lib
    z = lambda n, B=4, H=2: (np.zeros((n, B)), np.zeros((n, B)), np.zeros((H, n, B)))
    R, t, m, c, Ic = _random_chain(13, 90)
    for mb in (rb.Multibody.from_urdf(CHAIN32), rb.Multibody.from_descriptor(R, t, m, c, Ic),
               rb.Multibody.from_descriptor(R[:6], t[:6], m[:6], c[:6], Ic[:6], parent=_random_tree(6, 3))):
        q0, dq0, tau = z(mb.n)
        for call in (lambda: mb.rollout_cost_grad(q0, dq0, tau, DT, w_q=np.ones(mb.n)),
                     lambda: mb.rollout_vjp(q0, dq0, tau, DT, tau, tau)):
            with pytest.raises(rb.RigidBodyError) as ei:
                call()
            assert ei.value.code == _lib.RB_ERR_UNSUPPORTED and "12 joints" in str(ei.value)
    mb = mb_fr3
    q0, dq0, tau = z(7)
    p = lambda a: C.c_void_p(a.ctypes.data)
    out = [np.zeros((2, 7, 4)), np.zeros((7, 4)), np.zeros((7, 4))]
    qc, keep = mb._quad_cost(w_q=np.ones(7))
    cost = np.zeros(4)
    cg = lambda a, b, ct, wts, cst, dt=DT: lib.multibody_rollout_cost_grad(mb._h, a, b, ct, dt, 2, wts, cst, *[p(o) for o in out], 4, 0, 0, 0, None)
    vj = lambda a, b, ct, qt, dqt, dt=DT: lib.multibody_rollout_vjp(mb._h, a, b, ct, dt, 2, qt, dqt, None, None, None, None, *[p(o) for o in out], 4, 0, 0, 0, None)
    assert cg(p(q0), p(dq0), p(tau), C.byref(qc), p(cost)) == 0
    assert vj(p(q0), p(dq0), p(tau), p(tau), p(tau)) == 0
    assert cg(None, p(dq0), p(tau), C.byref(qc), p(cost)) == _lib.RB_ERR_NULL
    assert cg(p(q0), p(dq0), None, C.byref(qc), p(cost)) == _lib.RB_ERR_NULL
    assert cg(p(q0), p(dq0), p(tau), None, p(cost)) == _lib.RB_ERR_NULL
    assert cg(p(q0), p(dq0), p(tau), C.byref(qc), None) == _lib.RB_ERR_NULL
    assert vj(p(q0), None, p(tau), p(tau), p(tau)) == _lib.RB_ERR_NULL
    assert vj(p(q0), p(dq0), p(tau), None, p(tau)) == _lib.RB_ERR_NULL
    assert cg(p(q0), p(dq0), p(tau), C.byref(qc), p(cost), dt=float("inf")) == _lib.RB_ERR_ARG
    assert vj(p(q0), p(dq0), p(tau), p(tau), p(tau), dt=float("nan")) == _lib.RB_ERR_ARG
    bad, keep2 = mb._quad_cost(w_dq=-np.ones(7))
    assert cg(p(q0), p(dq0), p(tau), C.byref(bad), p(cost)) == _lib.RB_ERR_ARG
    with pytest.raises(rb.RigidBodyError):
        mb.rollout_cost_grad(q0, dq0, tau, DT, w_tau=-np.ones(7))


def _spd_where_q1_small(rb):
    """Two joints, the second about the first link's x axis; the second link's (non-physical) inertia diag(0.5, -1, 1)
    makes H_00 = 0.1 + 0.5 cos^2 q_1 - sin^2 q_1: positive definite for |q_1| < 0.68, indefinite near pi/2."""
    R = np.stack([np.eye(3), np.array([[0.0, 0.0, 1.0], [0.0, 1.0, 0.0], [-1.0, 0.0, 0.0]])])
    Ic = np.stack([np.eye(3) * 0.1, np.diag([0.5, -1.0, 1.0])])
    return rb.Multibody.from_descriptor(R, np.zeros((2, 3)), np.ones(2), np.zeros((2, 3)), Ic)


@pytest.mark.gpu
def test_not_spd_gives_nan_for_the_bad_trajectories_only(rb):
    from rigidbody_rs_b200 import _lib
    lib = _lib.lib
    # the chain of test_not_spd_is_reported: every state indefinite
    n = 2
    R = np.tile(np.eye(3), (n, 1, 1)); t = np.zeros((n, 3)); t[1] = [0.1, 0, 0]
    bad = rb.Multibody.from_descriptor(R, t, np.ones(n), np.zeros((n, 3)), np.tile(np.diag([0.1, 0.1, -5.0]), (n, 1, 1)))
    z, zt = np.zeros((2, 4)), np.zeros((3, 2, 4))
    with pytest.raises(rb.NotPositiveDefinite):
        bad.rollout_cost_grad(z, z, zt, 1e-3, w_q=np.ones(2))
    with pytest.raises(rb.NotPositiveDefinite):
        bad.rollout_vjp(z, z, zt, 1e-3, zt, zt, np.ones_like(zt))
    assert bad.rnea(z, z, z).shape == (2, 4)                     # the next call is clean
    # a chain whose mass matrix is indefinite in some configurations only: NaN exactly there
    mb = _spd_where_q1_small(rb)
    B, H = 6, 3
    q0 = np.zeros((2, B)); q0[1, 1::2] = 1.5                      # odd trajectories start (and stay) where H is indefinite
    dq0, tau = np.zeros((2, B)), np.zeros((H, 2, B))
    qc, keep = mb._quad_cost(q_ref=np.full(2, 0.3), w_q=np.ones(2), w_dq_final=np.ones(2))
    cost = np.zeros(B)
    gt, gq, gdq = np.zeros((H, 2, B)), np.zeros((2, B)), np.zeros((2, B))
    p = lambda a: C.c_void_p(a.ctypes.data)
    rc = lib.multibody_rollout_cost_grad(mb._h, p(q0), p(dq0), p(tau), 1e-3, H, C.byref(qc), p(cost), p(gt), p(gq), p(gdq), B, 0, 0, 0, None)
    assert rc == _lib.RB_ERR_NOT_SPD
    for g in (gt, gq, gdq):
        assert np.isnan(g[..., 1::2]).all() and np.isfinite(g[..., 0::2]).all()
    assert np.isnan(cost[1::2]).all() and np.isfinite(cost[0::2]).all()
    good = mb.rollout_cost_grad(q0[:, 0::2].copy(), dq0[:, 0::2].copy(), tau[..., 0::2].copy(), 1e-3, q_ref=np.full(2, 0.3),
                                w_q=np.ones(2), w_dq_final=np.ones(2))
    for a, b in zip((cost, gt, gq, gdq), good):
        np.testing.assert_array_equal(a[..., 0::2], b)


@pytest.mark.gpu
def test_full_size_fr3_65536x64(rb, mb_fr3, oracle_fr3):
    """The size bench.py's rollout runs: 65 536 trajectories x 64 steps through cost_grad, host and device.  All
    gradients finite, host = device bit for bit, and 256 strided trajectories against the numpy twin."""
    import torch
    from oracle.rb_oracle_np import ChainNP
    mb = mb_fr3
    B, H, dt = 65536, 64, 1e-3
    lim = oracle_fr3.model
    q0, dq0, _ = _fr3_inputs(oracle_fr3, B, 0, 0x5EED0047)
    rng = np.random.default_rng(47)
    tau = rng.uniform(-0.3, 0.3, (H, 7, B)) * lim.effort[None, :, None]
    w = _weights(7, 47)
    host = mb.rollout_cost_grad(q0, dq0, tau, dt, **w)
    dev = mb.rollout_cost_grad(*_dev(q0, dq0, tau), dt, **w)
    for a, b in zip(host, dev):
        assert np.isfinite(a).all()
        np.testing.assert_array_equal(b.cpu().numpy(), a)
    del dev
    torch.cuda.empty_cache()
    idx = np.arange(0, B, B // 256)
    s0, s1, st = q0[:, idx].copy(), dq0[:, idx].copy(), tau[..., idx].copy()
    ref = rollout_cost_grad_np(ChainNP(oracle_fr3.model), s0, s1, st, dt, *oracle_fr3.rollout_batch(s0, s1, st, dt), **w)
    for got, want in zip(host[1:], ref):
        _close(got[..., idx], want)
