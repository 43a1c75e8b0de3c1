"""Batched tip pose and inverse kinematics of the tip frame (include/rigidbody.h multibody_tip_pose_batch /
multibody_ik_batch).

The checker `ik_np` replicates the algorithm stated in the header on the numpy twin's `ChainNP.fwd_kin` / `jac`: the same
clamp, the same 6x6 LDL^T of W J J^T W + lambda I, the same lambda schedule and accept rule.  Only the rounding of the
kinematics differs (the kernel accumulates J J^T in the tip frame and rotates it once), so a few iterations agree to
1e-10 * max(1, |ref|) and iteration counts agree exactly.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import CHAIN32, FR3, TOL

SQRT8 = np.sqrt(8.0)


# ------------------------------------------------------------------------------------------------ the numpy checker
def pose_np(chain, q, off):
    """q [B, n] -> (R [B, 3, 3], x = p + R off [B, 3])."""
    R, p = chain.fwd_kin(q)
    return R, p + R @ off


def jac_base_np(chain, q, off, R):
    """Base-frame Jacobian [B, 6, n] of (x, orientation): column j = (z_j x (x - P_j) ; z_j), zero off the tip's branch."""
    J = chain.jac(q)
    lin = J[:, 0:3] + np.cross(J[:, 3:6], off, axisa=1, axisb=0, axisc=1)
    return np.concatenate([R @ lin, R @ J[:, 3:6]], 1)


def objective_np(R, x, pt, Rt, w_p, w_R):
    """(F, squared position error over the weighted axes, ||R - R*||_F^2 (0 when w_R == 0))."""
    e = x - pt
    pos2 = np.where(w_p > 0, e * e, 0.0).sum(1)
    rot2 = ((R - Rt) ** 2).sum((1, 2)) if w_R > 0 else np.zeros(len(x))
    return (w_p * e * e).sum(1) + w_R * rot2, pos2, rot2


def omega_np(R, Rt):
    """omega = 1/2 sum_k R[:, k] x R*[:, k]."""
    return 0.5 * np.cross(R, Rt, axis=1).sum(2)


def rot_angle_np(rot2):
    return 2.0 * np.arcsin(np.minimum(1.0, np.sqrt(rot2) / SQRT8))


def ldlt6_np(A, b):
    """Batched LDL^T solve of 6x6 systems A [B, 6, 6] y = b [B, 6]; ok = every pivot positive."""
    A = A.copy(); y = b.copy()
    ok = np.ones(len(A), bool)
    for j in range(6):
        d = A[:, j, j] - sum(A[:, j, m] * A[:, j, m] * A[:, m, m] for m in range(j)) if j else A[:, j, j].copy()
        ok &= d > 0
        A[:, j, j] = d
        for i in range(j + 1, 6):
            v = A[:, i, j] - sum(A[:, i, m] * A[:, j, m] * A[:, m, m] for m in range(j)) if j else A[:, i, j].copy()
            A[:, i, j] = v / d
    for i in range(1, 6):
        for m in range(i):
            y[:, i] -= A[:, i, m] * y[:, m]
    y /= np.stack([A[:, i, i] for i in range(6)], 1)
    for i in range(4, -1, -1):
        for m in range(i + 1, 6):
            y[:, i] -= A[:, m, i] * y[:, m]
    return y, ok


def step_np(J, pt, x, R, Rt, w_p, w_R, lam):
    """The damped step delta = J^T W (W J J^T W + lambda I)^-1 W e and the pivot flag."""
    sw = np.concatenate([np.sqrt(w_p), np.full(3, np.sqrt(2.0 * w_R))])
    WJ = sw[None, :, None] * J
    A = WJ @ np.swapaxes(WJ, 1, 2) + lam[:, None, None] * np.eye(6)
    e = np.concatenate([pt - x, omega_np(R, Rt) if w_R > 0 else np.zeros_like(x)], 1)
    y, ok = ldlt6_np(A, sw * e)
    return np.einsum("bkn,bk->bn", J, sw * y), ok


def ik_np(chain, q_init, p_t, R_t=None, offset=None, w_p=None, w_R=None, lower=None, upper=None, max_iters=100, tol_p=1e-6,
          tol_R=1e-6, damping=1e-3):
    """The algorithm of multibody_ik_batch.  q_init [B, n], p_t [B, 3], R_t [B, 3, 3].  Returns (q [B, n], pos_err, rot_err,
    iters)."""
    n = chain.n
    B = len(q_init)
    off = np.zeros(3) if offset is None else np.asarray(offset, float)
    w_p = np.ones(3) if w_p is None else np.asarray(w_p, float)
    w_R = (0.0 if R_t is None else 1.0) if w_R is None else float(w_R)
    lo = np.full(n, -np.inf) if lower is None else np.asarray(lower, float)
    hi = np.full(n, np.inf) if upper is None else np.asarray(upper, float)
    Rt = np.zeros((B, 3, 3)) if w_R == 0 else np.asarray(R_t, float).reshape(B, 3, 3)
    fin = np.isfinite(q_init).all(1) & np.isfinite(p_t).all(1) & np.isfinite(Rt).all((1, 2))
    q = np.clip(np.where(fin[:, None], q_init, 0.0), lo, hi)
    R, x = pose_np(chain, q, off)
    F, pos2, rot2 = objective_np(R, x, p_t, Rt, w_p, w_R)
    lam = np.full(B, float(damping))
    iters = np.full(B, -1)
    active = fin.copy()
    with np.errstate(all="ignore"):
        for k in range(max_iters + 1):
            conv = active & (np.sqrt(pos2) <= tol_p) & ((w_R == 0) | (rot_angle_np(rot2) <= tol_R))
            iters[conv] = k
            active &= ~conv
            if k == max_iters or not active.any():
                break
            d, ok = step_np(jac_base_np(chain, q, off, R), p_t, x, R, Rt, w_p, w_R, lam)
            qn = np.clip(np.where(ok[:, None], q + d, q), lo, hi)
            Rn, xn = pose_np(chain, qn, off)
            Fn, pos2n, rot2n = objective_np(Rn, xn, p_t, Rt, w_p, w_R)
            acc = active & ok & (Fn < F)
            rej = active & ~acc
            q[acc], R[acc], x[acc], F[acc], pos2[acc], rot2[acc] = qn[acc], Rn[acc], xn[acc], Fn[acc], pos2n[acc], rot2n[acc]
            lam[acc] = np.maximum(lam[acc] / 10, 1e-12)
            lam[rej] = np.minimum(lam[rej] * 10, 1e12)
    pos, rot = np.sqrt(pos2), (rot_angle_np(rot2) if w_R > 0 else np.zeros(B))
    q[~fin], pos[~fin], rot[~fin] = np.nan, np.nan, np.nan
    return q, pos, rot, iters


# ------------------------------------------------------------------------------------------------ chains
def _fr3_twin():
    from oracle.rb_oracle_np import ChainNP
    from oracle.rb_oracle import Oracle
    return ChainNP(Oracle.from_urdf(FR3).model)


def _random_twin(n, seed, tree=False):
    from oracle.rb_oracle_np import ChainNP
    from test_host import AXES, _random_chain, _random_tree
    R, t, m, c, Ic = _random_chain(n, seed)
    ax = (AXES * (n // len(AXES) + 1))[:n]
    par = _random_tree(n, seed) if tree else None
    return (R, t, m, c, Ic, ax, par), ChainNP.from_arrays(R, t, m, c, Ic, axis=ax, parent=par)


def _chain(rb, name):
    """(engine, twin) of one of the chains the GPU tests use."""
    from oracle.rb_oracle_np import ChainNP
    from oracle.rb_oracle import Oracle
    if name in ("fr3", "chain32"):
        path = FR3 if name == "fr3" else CHAIN32
        return rb.Multibody.from_urdf(path), ChainNP(Oracle.from_urdf(path).model)
    kind, n = name[0], int(name[1:])
    (R, t, m, c, Ic, ax, par), twin = _random_twin(n, 70 + n, tree=kind == "t")
    return rb.Multibody.from_descriptor(R, t, m, c, Ic, axis=ax, parent=par), twin


CHAINS = ["fr3", "chain32", "r1", "r2", "r5", "r12", "r40", "t5", "t20"]
PARITY_CHAINS = ["fr3", "r1", "r2", "r5", "r12", "r40", "t5", "t20"]


def _targets(twin, B, seed, sigma=0.3, lo=None, hi=None):
    """Targets = pose of random q* (inside finite bounds), seeds q* + N(0, sigma^2) clipped; q_init [B, n], p [B, 3], R [B, 3, 3]."""
    rng = np.random.default_rng(seed)
    n = twin.n
    lo = np.full(n, -np.pi) if lo is None else np.where(np.isfinite(lo), lo, -np.pi)
    hi = np.full(n, np.pi) if hi is None else np.where(np.isfinite(hi), hi, np.pi)
    qs = rng.uniform(lo, hi, (B, n))
    R, p = twin.fwd_kin(qs)
    q0 = np.clip(qs + rng.normal(0, sigma, (B, n)), lo, hi)
    return q0, p, R


def _fr3_limits(mb):
    L = mb.limits()
    return L["lower"], L["upper"]


# ------------------------------------------------------------------------------------------------ CPU
def test_push_through_step_equals_normal_equations():
    rng = np.random.default_rng(1)
    for n in (1, 3, 7, 12):
        B = 16
        J = rng.normal(size=(B, 6, n))
        w_p, w_R = rng.uniform(0.1, 3, 3), 0.7
        sw = np.concatenate([np.sqrt(w_p), np.full(3, np.sqrt(2 * w_R))])
        e = rng.normal(size=(B, 6))
        lam = 10.0 ** rng.uniform(-1, 1, B)      # well-conditioned on both sides: the identity is exact, its rounding is not
        WJ = sw[None, :, None] * J
        A6 = WJ @ np.swapaxes(WJ, 1, 2) + lam[:, None, None] * np.eye(6)
        y, ok = ldlt6_np(A6, sw * e)
        assert ok.all()
        d6 = np.einsum("bkn,bk->bn", J, sw * y)
        An = np.swapaxes(WJ, 1, 2) @ WJ + lam[:, None, None] * np.eye(n)
        dn = np.linalg.solve(An, np.einsum("bkn,bk->bn", WJ, sw * e)[..., None])[..., 0]
        assert np.abs(d6 - dn).max() <= 1e-12 * max(1.0, np.abs(dn).max()), n


@pytest.mark.parametrize("chain", ["fr3", "random5"])
def test_gauss_newton_rhs_is_half_the_negative_gradient(built, chain):
    """J^T W^2 e = -1/2 grad F by central differences (tracked point off the tip origin, oblique axes for the random chain)."""
    twin = _fr3_twin() if chain == "fr3" else _random_twin(5, 5)[1]
    rng = np.random.default_rng(2)
    B, n = 4, twin.n
    q = rng.uniform(-1, 1, (B, n))
    off = np.array([0.03, -0.05, 0.1])
    pt = rng.uniform(-0.5, 0.5, (B, 3))
    from scipy.spatial.transform import Rotation
    Rt = Rotation.from_rotvec(rng.normal(size=(B, 3))).as_matrix()
    w_p, w_R = np.array([1.0, 2.0, 0.5]), 0.8
    R, x = pose_np(twin, q, off)
    J = jac_base_np(twin, q, off, R)
    W2 = np.concatenate([w_p, np.full(3, 2 * w_R)])
    e = np.concatenate([pt - x, omega_np(R, Rt)], 1)
    g = np.einsum("bkn,bk->bn", J, W2 * e)
    F = lambda qq: objective_np(*pose_np(twin, qq, off), pt, Rt, w_p, w_R)[0]
    fd = np.zeros_like(q)
    for j in range(n):
        h = 1e-6
        up, dn = q.copy(), q.copy(); up[:, j] += h; dn[:, j] -= h
        fd[:, j] = -0.5 * (F(up) - F(dn)) / (2 * h)
    assert np.abs(fd - g).max() <= 1e-7 * max(1.0, np.abs(g).max())


def test_rotation_angle_formula():
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(3)
    A = Rotation.random(200, random_state=4)
    Dl = Rotation.from_rotvec(rng.normal(size=(200, 3)) * rng.uniform(0, 3.1, (200, 1)))
    Rt, R = A.as_matrix(), (Dl * A).as_matrix()
    want = (Dl).magnitude()
    got = rot_angle_np(((R - Rt) ** 2).sum((1, 2)))
    assert np.abs(got - want).max() < 1e-7


def test_ik_np_converges_on_reachable_fr3_targets(built):
    twin = _fr3_twin()
    q0, p, R = _targets(twin, 64, 5, sigma=0.2)
    q, pos, rot, it = ik_np(twin, q0, p, R)
    assert (it >= 0).mean() >= 0.9
    ok = it >= 0
    assert (pos[ok] <= 1e-6).all() and (rot[ok] <= 1e-6).all()
    R2, x2 = pose_np(twin, q[ok], np.zeros(3))
    assert np.abs(x2 - p[ok]).max() < 2e-6


# ------------------------------------------------------------------------------------------------ on the B200
def _dev(*xs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(x)).to("cuda:0") for x in xs]


def _soa(x):
    return np.ascontiguousarray(np.asarray(x).reshape(len(x), -1).T)


def _close(got, ref, what):
    got, ref = np.asarray(got), np.asarray(ref)
    bad = ~(np.abs(got - ref) <= TOL * np.maximum(1.0, np.abs(ref)))
    bad &= ~(np.isnan(got) & np.isnan(ref))
    assert not bad.any(), (what, int(bad.sum()), np.abs(got - ref)[bad].max() if bad.any() else 0)


def _two_devices():
    import torch
    if torch.cuda.device_count() >= 2:
        return [0, 1]
    os.environ["RIGIDBODY_B200_ALLOW_DUPLICATE_DEVICES"] = "1"
    return [0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CHAINS)
def test_tip_pose_matches_twin(rb, name):
    mb, twin = _chain(rb, name)
    rng = np.random.default_rng(11)
    q = rng.uniform(-np.pi, np.pi, (257, twin.n))
    off = np.array([0.02, -0.07, 0.11])
    R, x = pose_np(twin, q, off)
    ref = np.concatenate([x, R.reshape(-1, 9)], 1).T
    _close(mb.tip_pose(_soa(q), offset=off), ref, name)
    P0 = mb.tip_pose(_soa(q))
    _close(P0[3:], ref[3:], name)
    assert np.abs(P0[:3] - mb.fwd_kin(_soa(q))).max() <= 1e-13 * max(1.0, np.abs(P0[:3]).max())
    x1, R1 = mb.tip_pose(q[0], offset=off)
    _close(np.concatenate([x1, R1.reshape(9)]), ref[:, 0], name)


@pytest.mark.gpu
def test_tip_pose_layouts_memory_and_devices(rb):
    from rigidbody_rs_b200 import _lib
    mb, twin = _chain(rb, "fr3")
    q = _soa(np.random.default_rng(12).uniform(-2, 2, (300, 7)))
    off = [0.0, 0.01, 0.2]
    ref = mb.tip_pose(q, offset=off)
    assert np.array_equal(mb.tip_pose(_dev(q)[0], offset=off).cpu().numpy(), ref)
    assert np.array_equal(mb.tip_pose(q.T.copy(), offset=off, layout="aos"), ref.T)
    assert np.array_equal(mb.tip_pose(_dev(q.T.copy())[0], offset=off, layout="aos").cpu().numpy(), ref.T)
    ld, B = 333, 300
    for mem in (_lib.RB_MEM_HOST, _lib.RB_MEM_DEVICE):
        qp = np.full((7, ld), np.nan); qp[:, :B] = q
        out = np.full((12, ld), -7.0)
        offa = np.asarray(off)
        if mem == _lib.RB_MEM_DEVICE:
            import torch
            qd, od = _dev(qp, out)
            _lib.check(_lib.lib.multibody_tip_pose_batch(mb._h, C.c_void_p(qd.data_ptr()), offa.ctypes.data_as(C.POINTER(C.c_double)),
                                                         C.c_void_p(od.data_ptr()), B, ld, _lib.RB_LAYOUT_SOA, mem, None))
            torch.cuda.synchronize()
            out = od.cpu().numpy()
        else:
            _lib.check(_lib.lib.multibody_tip_pose_batch(mb._h, C.c_void_p(qp.ctypes.data), offa.ctypes.data_as(C.POINTER(C.c_double)),
                                                         C.c_void_p(out.ctypes.data), B, ld, _lib.RB_LAYOUT_SOA, mem, None))
        assert np.array_equal(out[:, :B], ref) and (out[:, B:] == -7.0).all()
    mm = rb.Multibody.from_urdf(FR3, devices=_two_devices())
    assert np.array_equal(mm.tip_pose(q, offset=off), ref)
    assert np.array_equal(mm.tip_pose(q.T.copy(), offset=off, layout="aos"), ref.T)
    with pytest.raises(rb.RigidBodyError):
        mb.tip_pose(q, offset=[0.0, np.inf, 0.0])


def _gpu_ik(mb, q0, p, R, **kw):
    """mb.ik on device SoA arrays -> (q [B, n], pos, rot, iters) as numpy."""
    args = _dev(_soa(q0), _soa(p)) + ([_dev(_soa(R))[0]] if R is not None else [None])
    q, info = mb.ik(args[1], args[2], q_init=args[0], **kw)
    q, info = q.cpu().numpy(), info.cpu().numpy()
    return q.T, info[0], info[1], info[2]


@pytest.mark.gpu
@pytest.mark.parametrize("name", PARITY_CHAINS)
@pytest.mark.parametrize("iters", [0, 1, 2, 5])
def test_ik_matches_numpy_replica(rb, name, iters):
    mb, twin = _chain(rb, name)
    n = twin.n
    B = 256
    q0, p, R = _targets(twin, B, 20 + n, sigma=0.4)
    lo, hi = np.full(n, -2.5), np.full(n, 2.5)
    lo[0], hi[0] = -np.inf, np.inf
    off = np.array([0.01, 0.02, 0.05])
    # Below six joints on the tip's branch W J J^T W is singular and y = (W J J^T W + lambda I)^-1 W e grows like 1/lambda along its null space,
    # which J^T maps to zero only up to the rounding of J: the two kinematics' last-bit differences reach delta amplified
    # by 1/lambda.  A larger initial damping keeps that under the bar over five iterations.
    branch, i = 0, n - 1
    while i >= 0:
        branch, i = branch + 1, twin.parent[i]
    damping = 1e-3 if branch >= 6 else 1.0
    for full in (True, False):
        kw = dict(offset=off, w_p=[1.0, 2.0, 0.5], limits=(lo, hi), max_iters=iters, tol_p=1e-9, tol_R=1e-9, damping=damping)
        Rk = R if full else None
        if full:
            kw["w_R"] = 0.7
        got = _gpu_ik(mb, q0, p, Rk, **kw)
        ref = ik_np(twin, q0, p, Rk, offset=off, w_p=[1.0, 2.0, 0.5], w_R=kw.get("w_R", 0.0), lower=lo, upper=hi, max_iters=iters,
                    tol_p=1e-9, tol_R=1e-9, damping=damping)
        if iters == 0:
            assert np.array_equal(got[0], np.clip(q0, lo, hi))
        same = got[3] == ref[3]
        assert same.mean() >= 0.99, (name, iters, full, same.mean())
        for k, what in enumerate(("q", "pos_err", "rot_err")):
            _close(got[k][same], ref[k][same], (name, iters, full, what))


def _convergence_case(rb, full):
    mb = rb.Multibody.from_urdf(FR3)
    twin = _fr3_twin()
    lo, hi = _fr3_limits(mb)
    B = 65536
    q0, p, R = _targets(twin, B, 31, sigma=0.3, lo=lo, hi=hi)
    return mb, twin, lo, hi, q0, p, (R if full else None)


@pytest.mark.gpu
@pytest.mark.parametrize("full", [True, False])
def test_ik_convergence_fr3(rb, full):
    mb, twin, lo, hi, q0, p, R = _convergence_case(rb, full)
    q, pos, rot, it = _gpu_ik(mb, q0, p, R, max_iters=50)
    _, _, _, it_np = ik_np(twin, q0, p, R, lower=lo, upper=hi, max_iters=50)
    assert ((it >= 0) == (it_np >= 0)).mean() >= 0.999
    assert (it >= 0).mean() >= 0.9, (it >= 0).mean()
    assert (q >= lo).all() and (q <= hi).all()
    Rq, xq = pose_np(twin, q, np.zeros(3))
    pos_t = np.sqrt(((xq - p) ** 2).sum(1))
    assert np.abs(pos - pos_t).max() <= 1e-12
    ok = it >= 0
    assert (pos_t[ok] <= 1e-6 + 1e-12).all()
    if R is not None:
        rot_t = rot_angle_np(((Rq - R) ** 2).sum((1, 2)))
        assert np.abs(rot - rot_t).max() <= 1e-12
        assert (rot_t[ok] <= 1e-6 + 1e-12).all()
    else:
        assert (rot == 0).all()


@pytest.mark.gpu
def test_ik_unreachable_targets(rb):
    mb, twin = _chain(rb, "fr3")
    lo, hi = _fr3_limits(mb)
    rng = np.random.default_rng(41)
    B = 512
    q0 = rng.uniform(lo, hi, (B, 7))
    d = rng.normal(size=(B, 3)); p = 5.0 * d / np.linalg.norm(d, axis=1, keepdims=True)
    from scipy.spatial.transform import Rotation
    R = Rotation.random(B, random_state=42).as_matrix()
    q, pos, rot, it = _gpu_ik(mb, q0, p, R, max_iters=30)
    assert (it == -1).all()
    F0 = objective_np(*pose_np(twin, np.clip(q0, lo, hi), np.zeros(3)), p, R, np.ones(3), 1.0)[0]
    F1 = objective_np(*pose_np(twin, q, np.zeros(3)), p, R, np.ones(3), 1.0)[0]
    assert (F1 <= F0 * (1 + 1e-12)).all()


@pytest.mark.gpu
def test_ik_same_bits_in_every_family(rb):
    twin = _fr3_twin()
    q0, p, R = _targets(twin, 1000, 51)
    res = {}
    saved = {k: os.environ.pop(k, None) for k in ("RIGIDBODY_B200_VARIANT", "RIGIDBODY_B200_JIT")}
    try:
        for v in ("fr3-specialised", "generic-7", "generic-n", "jit-specialised"):
            os.environ["RIGIDBODY_B200_VARIANT"] = v
            mb = rb.Multibody.from_urdf(FR3)
            assert mb.kernel_variant == v
            res[v] = (_gpu_ik(mb, q0, p, R, max_iters=20), mb.tip_pose(_soa(q0), offset=[0.1, 0, 0]))
            mb.close()
    finally:
        os.environ.pop("RIGIDBODY_B200_VARIANT", None)
        for k, v in saved.items():
            if v is not None:
                os.environ[k] = v
    first = res["fr3-specialised"]
    for v, r in res.items():
        for a, b in zip(r[0], first[0]):
            assert np.array_equal(a, b, equal_nan=True), v
        assert np.array_equal(r[1], first[1]), v


@pytest.mark.gpu
def test_ik_layouts_memory_kinds_and_devices(rb):
    from rigidbody_rs_b200 import _lib
    import torch
    mb, twin = _chain(rb, "fr3")
    lo, hi = _fr3_limits(mb)
    B = 777
    q0, p, R = _targets(twin, B, 61, lo=lo, hi=hi)
    kw = dict(max_iters=20, offset=[0, 0, 0.1])
    qd, infod = mb.ik(*_dev(_soa(p), _soa(R)), q_init=_dev(_soa(q0))[0], **kw)
    ref = np.concatenate([qd.cpu().numpy(), infod.cpu().numpy()])
    qh, infoh = mb.ik(_soa(p), _soa(R), q_init=_soa(q0), **kw)
    assert np.array_equal(np.concatenate([qh, infoh]), ref)
    qa, infoa = mb.ik(p, R, q_init=q0, layout="aos", **kw)
    assert np.array_equal(np.concatenate([qa, infoa], 1), ref.T)
    qa, infoa = mb.ik(*_dev(p, R.reshape(B, 9)), q_init=_dev(q0)[0], layout="aos", **kw)
    assert np.array_equal(np.concatenate([qa.cpu().numpy(), infoa.cpu().numpy()], 1), ref.T)
    # padded leading dimension through the C ABI, host and device: the padding is left alone
    ld = B + 45
    offa = np.array([0, 0, 0.1])
    opt = _lib.RbIkOptions(offset=offa.ctypes.data_as(C.POINTER(C.c_double)), w_R=1.0,
                           lower=np.ascontiguousarray(lo).ctypes.data_as(C.POINTER(C.c_double)),
                           upper=np.ascontiguousarray(hi).ctypes.data_as(C.POINTER(C.c_double)),
                           max_iters=20, tol_p=1e-6, tol_R=1e-6, damping=1e-3)
    lo, hi = np.ascontiguousarray(lo), np.ascontiguousarray(hi)
    pad = lambda x: np.concatenate([_soa(x), np.full((_soa(x).shape[0], ld - B), np.nan)], 1)
    for mem in (_lib.RB_MEM_HOST, _lib.RB_MEM_DEVICE):
        ins = [pad(q0), pad(p), pad(R)]
        out = np.full((10, ld), -3.0)
        if mem == _lib.RB_MEM_DEVICE:
            ins, out_t = _dev(*ins), _dev(out)[0]
            ptrs = [C.c_void_p(x.data_ptr()) for x in ins] + [C.c_void_p(out_t.data_ptr())]
        else:
            ptrs = [C.c_void_p(x.ctypes.data) for x in ins] + [C.c_void_p(out.ctypes.data)]
        _lib.check(_lib.lib.multibody_ik_batch(mb._h, *ptrs[:3], C.byref(opt), ptrs[3], B, ld, _lib.RB_LAYOUT_SOA, mem, None))
        if mem == _lib.RB_MEM_DEVICE:
            torch.cuda.synchronize()
            out = out_t.cpu().numpy()
        assert np.array_equal(out[:, :B], ref) and (out[:, B:] == -3.0).all(), mem
    mm = rb.Multibody.from_urdf(FR3, devices=_two_devices())
    qm, infom = mm.ik(_soa(p), _soa(R), q_init=_soa(q0), **kw)
    assert np.array_equal(np.concatenate([qm, infom]), ref)
    with pytest.raises(rb.RigidBodyError) as e:
        mm.ik(*_dev(_soa(p), _soa(R)), q_init=_dev(_soa(q0))[0], **kw)
    assert e.value.code == _lib.RB_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_ik_host_batch_spans_pipeline_chunks(rb):
    """2^20 + 17 FR3 problems from host memory: 29 staged doubles per problem, more than one chunk of the host pipeline."""
    mb, twin = _chain(rb, "fr3")
    lo, hi = _fr3_limits(mb)
    B = (1 << 20) + 17
    rng = np.random.default_rng(71)
    qs = rng.uniform(lo, hi, (B, 7))
    P = mb.tip_pose(_dev(_soa(qs))[0]).cpu().numpy()
    q0 = np.clip(qs + rng.normal(0, 0.3, qs.shape), lo, hi)
    qd, infod = mb.ik(*_dev(P[:3], P[3:]), q_init=_dev(_soa(q0))[0], max_iters=10)
    qh, infoh = mb.ik(P[:3].copy(), P[3:].copy(), q_init=_soa(q0), max_iters=10)
    assert np.array_equal(qh, qd.cpu().numpy()) and np.array_equal(infoh, infod.cpu().numpy())


@pytest.mark.gpu
def test_ik_one_launch_per_device_call(rb):
    mb, twin = _chain(rb, "t5")
    q0, p, R = _targets(twin, 1000, 81)
    args = _dev(_soa(p), _soa(R), _soa(q0))
    c0 = mb.launch_count
    mb.ik(args[0], args[1], q_init=args[2], max_iters=5)
    assert mb.launch_count - c0 == 1
    c0 = mb.launch_count
    mb.tip_pose(args[2])
    assert mb.launch_count - c0 == 1


@pytest.mark.gpu
def test_ik_edge_cases(rb):
    mb, twin = _chain(rb, "fr3")
    import torch
    q, info = mb.ik(torch.empty((3, 0), dtype=torch.float64, device="cuda:0"), q_init=torch.empty((7, 0), dtype=torch.float64, device="cuda:0"))
    assert q.shape == (7, 0) and info.shape == (3, 0)
    q0, p, R = _targets(twin, 4, 91)
    q1, info1 = mb.ik(p[0], R[0], q_init=q0[0])
    ref = ik_np(twin, q0[:1], p[:1], R[:1], lower=_fr3_limits(mb)[0], upper=_fr3_limits(mb)[1])
    assert q1.shape == (7,) and info1.shape == (3,) and info1[2] == ref[3][0]
    q0[1, 2] = np.nan; p[2, 0] = np.inf; R[3, 1, 1] = np.nan
    q, info = mb.ik(_soa(p), _soa(R), q_init=_soa(q0))
    assert np.isnan(q[:, 1:]).all() and np.isnan(info[:2, 1:]).all() and (info[2, 1:] == -1).all()
    assert np.isfinite(q[:, 0]).all()
    # position only: R_target is not needed, and a non-finite entry of a never-read R_target does not matter
    q, info = mb.ik(_soa(p[:1]), q_init=_soa(q0[:1]))
    assert np.isfinite(q).all() and info[1, 0] == 0.0


@pytest.mark.gpu
def test_ik_error_codes(rb):
    from rigidbody_rs_b200 import _lib
    mb, twin = _chain(rb, "fr3")
    q0, p, R = _targets(twin, 8, 101)
    qa, pa, Ra = _soa(q0), _soa(p), _soa(R)
    out = np.empty((10, 8))
    n = 7
    arr = lambda v: np.ascontiguousarray(v, dtype=np.float64)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))

    def call(R_ptr=True, **kw):
        base = dict(w_R=1.0, max_iters=10, tol_p=1e-6, tol_R=1e-6, damping=1e-3)
        keep = []
        for k in ("offset", "w_p", "lower", "upper"):
            if k in kw:
                a = arr(kw.pop(k)); keep.append(a); base[k] = dp(a)
        base.update(kw)
        opt = _lib.RbIkOptions(**base)
        return _lib.lib.multibody_ik_batch(mb._h, C.c_void_p(qa.ctypes.data), C.c_void_p(pa.ctypes.data),
                                           C.c_void_p(Ra.ctypes.data) if R_ptr else None, C.byref(opt), C.c_void_p(out.ctypes.data), 8, 0,
                                           _lib.RB_LAYOUT_SOA, _lib.RB_MEM_HOST, None)
    assert call() == _lib.RB_OK
    ARG = _lib.RB_ERR_ARG
    assert call(w_p=[1, -1, 1]) == ARG
    assert call(w_p=[1, np.nan, 1]) == ARG
    assert call(w_R=-1.0) == ARG
    assert call(w_R=np.inf) == ARG
    assert call(lower=np.full(n, np.nan)) == ARG
    assert call(lower=np.full(n, 1.0), upper=np.full(n, 0.0)) == ARG
    assert call(max_iters=-1) == ARG
    assert call(tol_p=-1e-3) == ARG
    assert call(tol_R=-1e-3) == ARG
    assert call(damping=1e-13) == ARG
    assert call(damping=2e12) == ARG
    assert call(damping=np.nan) == ARG
    assert call(offset=[0, np.inf, 0]) == ARG
    assert call(R_ptr=False) == _lib.RB_ERR_NULL
    assert call(R_ptr=False, w_R=0.0) == _lib.RB_OK
    assert call(lower=np.full(n, -np.inf), upper=np.full(n, np.inf)) == _lib.RB_OK
    assert _lib.lib.multibody_ik_batch(mb._h, C.c_void_p(qa.ctypes.data), C.c_void_p(pa.ctypes.data), C.c_void_p(Ra.ctypes.data), None,
                                       C.c_void_p(out.ctypes.data), 8, 0, _lib.RB_LAYOUT_SOA, _lib.RB_MEM_HOST, None) == _lib.RB_ERR_NULL


@pytest.mark.gpu
def test_ik_python_defaults_and_side_stream(rb):
    import torch
    mb, twin = _chain(rb, "fr3")
    L = mb.limits()
    lo, hi = L["lower"].copy(), L["upper"].copy()
    q0, p, R = _targets(twin, 64, 111, lo=lo, hi=hi)
    # q_init=None: the midpoint of the (finite) bounds
    q, info = mb.ik(_soa(p), _soa(R), max_iters=3)
    ref = ik_np(twin, np.repeat((0.5 * (lo + hi))[None], 64, 0), p, R, lower=lo, upper=hi, max_iters=3)
    same = info[2] == ref[3]
    _close(q.T[same], ref[0][same], "midpoint start")
    # joints whose bounds are empty (lower >= upper: what the URDF parser reports for continuous joints) are unbounded
    # with limits=True; the others keep theirs
    (Rr, t, m, c, Ic, ax, par), tw5 = _random_twin(5, 3)
    m5 = rb.Multibody.from_descriptor(Rr, t, m, c, Ic, axis=ax)
    L5 = m5.limits()
    L5["lower"][[0, 3]] = 0.0
    L5["upper"][[0, 3]] = 0.0
    m5.limits = lambda: L5
    q05, p5, R5 = _targets(tw5, 32, 7, sigma=0.5)
    q5, info5 = m5.ik(_soa(p5), _soa(R5), q_init=_soa(q05), max_iters=4)
    lo5, hi5 = L5["lower"].copy(), L5["upper"].copy()
    lo5[[0, 3]], hi5[[0, 3]] = -np.inf, np.inf
    ref5 = ik_np(tw5, q05, p5, R5, lower=lo5, upper=hi5, max_iters=4)
    same = info5[2] == ref5[3]
    _close(q5.T[same], ref5[0][same], "unbounded")
    # torch tensors on a side stream
    s = torch.cuda.Stream()
    args = _dev(_soa(p), _soa(R), _soa(q0))
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        qs, infos = mb.ik(args[0], args[1], q_init=args[2], max_iters=10)
        P = mb.tip_pose(qs)
    s.synchronize()
    qh, infoh = mb.ik(_soa(p), _soa(R), q_init=_soa(q0), max_iters=10)
    assert np.array_equal(qs.cpu().numpy(), qh) and np.array_equal(infos.cpu().numpy(), infoh)
    assert np.array_equal(P.cpu().numpy(), mb.tip_pose(qh))
