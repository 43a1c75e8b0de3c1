"""CPU tests of the oracle itself (no GPU): what pins the oracle, since the reference pins nothing (SURVEY.md 4, 8c)."""
import ctypes as C

import numpy as np
import pytest

from conftest import FR3, CHAIN32, ROOT, TOL, load_golden, state_err
from oracle.rb_oracle import Oracle, parse_urdf
from oracle.rb_oracle_np import ChainNP, rnea_mp


@pytest.fixture(scope="module")
def np_fr3():
    return ChainNP(parse_urdf(FR3))


def test_urdf_pairing_matches_survey_table(oracle_fr3):
    """from_urdf's zip-by-document-order pairing (multibody.rs:70-75) keeps exactly the 7 revolute joints, each
    with its own child link's inertia (SURVEY.md 2.1 table)."""
    m = oracle_fr3.model
    assert m.n == 7 and m.names == [f"fr3_joint{k}" for k in range(1, 8)]
    np.testing.assert_array_equal(m.mass, [4.970684, 0.646926, 3.228604, 3.587895, 1.225946, 1.666555, 0.735522])
    np.testing.assert_array_equal(m.xyz[4], [-0.0825, 0.384, 0.0])
    np.testing.assert_array_equal(m.rpy[:, 0], [0, -np.pi / 2, np.pi / 2, np.pi / 2, -np.pi / 2, np.pi / 2, np.pi / 2])
    np.testing.assert_array_equal(m.com[1], [-0.003141, -0.02872, 0.003495])     # double space in the source xyz
    np.testing.assert_array_equal(m.effort, [87, 87, 87, 87, 12, 12, 12])


def test_dynamics_only_urdf_equals_reference_urdf():
    """assets/fr3.urdf loads to exactly the model the reference's robot description gives (stored in
    tests/golden/fr3_reference_model.json)."""
    a, b = load_golden("fr3_reference_model.json"), parse_urdf(FR3)
    for k in ("axis", "xyz", "rpy", "mass", "com", "inertia6", "lower", "upper", "velocity", "effort"):
        np.testing.assert_array_equal(np.array(a[k]), getattr(b, k))
    assert a["names"] == b.names


def test_survey_known_answers(oracle_fr3):
    """SURVEY.md 8c KATs (independent numpy restatement made during the survey)."""
    k = load_golden("survey_kat.json")
    for key in ("rnea_zero", "main_cpp", "generic"):
        c = k[key]
        tau = oracle_fr3.rnea(c["q"], c["dq"], c["ddq"])
        np.testing.assert_allclose(tau, c["tau"], rtol=0, atol=2e-12)
    c = k["main_cpp"]
    H = oracle_fr3.crba(c["q"])
    np.testing.assert_allclose(np.diag(H), c["crba_diag"], rtol=1e-12)
    np.testing.assert_allclose([H[0, 1], H[1, 3], H[5, 6]], [c["H01"], c["H13"], c["H56"]], rtol=1e-12)
    assert np.all(np.tril(H, -1) == 0.0)                     # reference leaves the strict lower triangle at 0
    np.testing.assert_allclose(oracle_fr3.fwd_kin(np.zeros(7)), k["fwd_kin_zero"], atol=1e-15)


@pytest.mark.parametrize("name,urdf", [("fr3_oracle.json", FR3), ("chain32_oracle.json", CHAIN32)])
def test_frozen_oracle_vectors(name, urdf, built):
    g = load_golden(name)
    o = Oracle.from_urdf(urdf)
    q, dq, ddq, tau = (np.array(g[k]) for k in ("q", "dq", "ddq", "tau_in"))
    assert state_err(o.rnea_batch(q, dq, ddq, layout="aos"), np.array(g["rnea"]), 1).max() < 1e-13
    assert state_err(o.forward_dynamics_batch(q, dq, tau, layout="aos"), np.array(g["fd"]), 1).max() < 1e-11
    assert state_err(o.crba_batch(q[:8], layout="aos"), np.array(g["crba_colmajor"]), 1).max() < 1e-13


@pytest.mark.parametrize("urdf", [FR3, CHAIN32])
def test_reference_shaped_oracle_equals_matrix_form(urdf, built):
    """Evidence (1) of SURVEY.md 8c: quaternion/(m,c,I_c) path == matrix/10-parameter path."""
    m = parse_urdf(urdf)
    o, c = Oracle(m), ChainNP(m)
    n, B = m.n, 1500
    rng = np.random.default_rng(1)
    q, dq, ddq = rng.uniform(-np.pi, np.pi, (B, n)), rng.uniform(-2, 2, (B, n)), rng.uniform(-10, 10, (B, n))
    tau = rng.uniform(-50, 50, (B, n))
    assert state_err(o.rnea_batch(q, dq, ddq, layout="aos"), c.rnea(q, dq, ddq), 1).max() < 1e-12
    Ho = o.crba_batch(q, layout="aos").reshape(B, n, n).transpose(0, 2, 1)
    assert np.abs(Ho - c.crba(q)).max() < 1e-11
    assert state_err(o.forward_dynamics_batch(q, dq, tau, layout="aos"), c.forward_dynamics(q, dq, tau), 1).max() < 1e-9
    J = np.stack([o.jac(x) for x in q[:40]])
    assert np.abs(J - c.jac(q[:40])).max() < 1e-12
    p = np.stack([o.fwd_kin(x) for x in q[:40]])
    assert np.abs(p - c.fwd_kin(q[:40])[1]).max() < 1e-12


def test_identities(oracle_fr3, np_fr3):
    """Evidence (2)-(5) of SURVEY.md 8c."""
    n, B = 7, 800
    rng = np.random.default_rng(2)
    q, dq, ddq = rng.uniform(-np.pi, np.pi, (B, n)), rng.uniform(-2, 2, (B, n)), rng.uniform(-10, 10, (B, n))
    tau = oracle_fr3.rnea_batch(q, dq, ddq, layout="aos")
    Hu = oracle_fr3.crba_batch(q, layout="aos").reshape(B, n, n).transpose(0, 2, 1)
    H = Hu + np.triu(Hu, 1).transpose(0, 2, 1)
    bias = oracle_fr3.rnea_batch(q, dq, np.zeros_like(q), layout="aos")
    assert np.abs(np.einsum("bij,bj->bi", H, ddq) + bias - tau).max() < 1e-12          # (2)
    back = oracle_fr3.forward_dynamics_batch(q, dq, tau, layout="aos")
    assert state_err(back, ddq, 1).max() < 1e-11                                        # (3)
    assert np.linalg.eigvalsh(H).min() > 0                                              # (4)
    grav = oracle_fr3.rnea_batch(q, np.zeros_like(q), np.zeros_like(q), layout="aos")   # (5) tau_g = dU/dq
    eps = 1e-6
    for i in range(n):
        e = np.zeros(n); e[i] = eps
        dU = (np_fr3.potential_energy(q + e) - np_fr3.potential_energy(q - e)) / (2 * eps)
        assert np.abs(dU - grav[:, i]).max() < 1e-6


def test_mpmath_bounds_rounding_error(oracle_fr3, np_fr3):
    """Evidence (7): both fp64 restatements sit within 1e-12 of a 40-digit evaluation."""
    rng = np.random.default_rng(3)
    for _ in range(3):
        q, dq, ddq = rng.uniform(-np.pi, np.pi, 7), rng.uniform(-2, 2, 7), rng.uniform(-10, 10, 7)
        t = rnea_mp(oracle_fr3.model, q, dq, ddq)
        s = max(1.0, np.abs(t).max())
        assert np.abs(oracle_fr3.rnea(q, dq, ddq) - t).max() / s < 1e-12
        assert np.abs(np_fr3.rnea(q, dq, ddq)[0] - t).max() / s < 1e-12


def test_mpmath_forward_dynamics_truth(oracle_fr3, oracle_chain32, np_fr3):
    """The forward-dynamics truth (fd_mp: H column by column from the 40-digit recursion, 40-digit solve) against both
    fp64 restatements: the C oracle's LL^T and the twin's numpy solve sit within 8 cond(H) eps of it (the bar of
    conftest.fd_bound), and the truth itself satisfies rnea(q, dq, qdd) = tau to 1e-25."""
    from conftest import fd_bound
    from oracle.rb_oracle_np import _rnea_mp, fd_mp
    rng = np.random.default_rng(5)
    for o, K, lim in ((oracle_fr3, 4, 80.0), (oracle_chain32, 1, 50.0)):
        n = o.model.n
        for _ in range(K):
            q, dq, tau = rng.uniform(-np.pi, np.pi, n), rng.uniform(-2, 2, n), rng.uniform(-lim, lim, n)
            x, cond = fd_mp(o.model, q, dq, tau, return_cond=True)
            err = np.abs(o.forward_dynamics(q, dq, tau) - x).max() / max(1.0, np.abs(x).max())
            assert err <= fd_bound(cond) and err < 1e-11, (n, err, cond)
            if n == 7:
                errn = np.abs(np_fr3.forward_dynamics(q, dq, tau)[0] - x).max() / max(1.0, np.abs(x).max())
                assert errn <= fd_bound(cond), (errn, cond)
            back = _rnea_mp(o.model, q, dq, x, 40)          # residual of the (fp64-rounded) truth: rounding of x only
            res = max(abs(float(back[i]) - tau[i]) for i in range(n))
            assert res < 1e-9 * max(1.0, np.abs(tau).max())


def test_reference_convention_tests_restated(oracle_fr3):
    """rigidbody/src/spatial.rs:283-382 restated against the oracle's building blocks, with the reference's own
    epsilons and the same asserts it leaves enabled."""
    lib = oracle_fr3.lib
    from oracle.rb_oracle import C as _C

    class Q(C.Structure):
        _fields_ = [("i", C.c_double), ("j", C.c_double), ("k", C.c_double), ("w", C.c_double)]

    class Iso(C.Structure):
        _fields_ = [("rot", Q), ("t", C.c_double * 3)]

    class SV(C.Structure):
        _fields_ = [("lin", C.c_double * 3), ("rot", C.c_double * 3)]

    lib.rbo_quat_from_scaled_axis.restype = Q
    lib.rbo_iso_inverse.restype = Iso
    lib.rbo_iso_inverse.argtypes = [Iso]
    lib.rbo_motion_transform.restype = SV
    lib.rbo_force_transform.restype = SV
    v3 = lambda *a: (C.c_double * 3)(*a)

    # coord_transforms (:283-300): rotation about -z by pi/2 equals the hand Rz(theta) matrix; x -> -y
    th = np.pi / 2
    rot = lib.rbo_quat_from_scaled_axis(v3(0, 0, -th))
    R = (C.c_double * 9)()
    lib.rbo_quat_to_matrix(rot, R)
    np.testing.assert_allclose(np.array(R).reshape(3, 3),
                               [[np.cos(th), np.sin(th), 0], [-np.sin(th), np.cos(th), 0], [0, 0, 1]], atol=1e-5)
    out = v3(0, 0, 0)
    lib.rbo_quat_rotate(rot, v3(1, 0, 0), out)
    np.testing.assert_allclose(list(out), [0, -1, 0], atol=1e-5)

    def feather(fn, T, vec6):   # 6x6 matrices are [rot; lin]-ordered (spatial.rs:137-149)
        X = (C.c_double * 36)()
        fn(C.byref(T), X)
        r = np.array(X).reshape(6, 6) @ vec6
        return r[3:], r[:3]     # lin, rot

    # vel_transform (:302-340)
    v = SV(v3(0, 1, 0), v3(1, 0, 0))
    v6 = np.array([1, 0, 0, 0, 1, 0.0])
    X1 = Iso(Q(0, 0, 0, 1), v3(0, 1, 0))
    v1 = lib.rbo_motion_transform(C.byref(v), C.byref(X1))
    lin_f, rot_f = feather(lib.rbo_plucker_motion, lib.rbo_iso_inverse(X1), v6)
    np.testing.assert_allclose(list(v1.rot), rot_f, atol=1e-4)        # (:324; the lin assert :325 is commented out)
    X2 = Iso(lib.rbo_quat_from_scaled_axis(v3(0, 0, th)), v3(0, 0, 0))
    v2 = lib.rbo_motion_transform(C.byref(v), C.byref(X2))
    lin_f, rot_f = feather(lib.rbo_plucker_motion, lib.rbo_iso_inverse(X2), v6)
    np.testing.assert_allclose(list(v2.rot), rot_f, atol=1e-4)        # :338
    np.testing.assert_allclose(list(v2.lin), lin_f, atol=1e-4)        # :339

    # force_transform (:342-382)
    f = SV(v3(0, 1, 0), v3(1, 0, 0))
    f6 = np.array([1, 0, 0, 0, 1, 0.0])
    X1 = Iso(Q(0, 0, 0, 1), v3(1, 0, 0))
    f1 = lib.rbo_force_transform(C.byref(f), C.byref(X1))
    lin_f, rot_f = feather(lib.rbo_plucker_force, X1, f6)
    np.testing.assert_allclose(list(f1.rot), rot_f, atol=1e-4)        # :364
    np.testing.assert_allclose(list(f1.lin), lin_f, atol=1e-4)        # :365
    X2 = Iso(lib.rbo_quat_from_scaled_axis(v3(0, 0, th)), v3(0.3, 0.5, 0))
    f2 = lib.rbo_force_transform(C.byref(f), C.byref(X2))
    lin_f, rot_f = feather(lib.rbo_plucker_force, lib.rbo_iso_inverse(X2), f6)
    np.testing.assert_allclose(list(f2.lin), lin_f, atol=1e-4)        # :381 (the rot assert :380 is commented out)


def test_sampler_is_counter_based(oracle_fr3):
    a = oracle_fr3.fill(0x5EED0001, 0, -1.0, 1.0, 0, 1000)
    b = oracle_fr3.fill(0x5EED0001, 0, -1.0, 1.0, 400, 100)
    np.testing.assert_array_equal(a[:, 400:500], b)                    # any shard regenerates its slice
    assert np.all(a >= -1.0) and np.all(a < 1.0) and abs(a.mean()) < 0.05
    c = oracle_fr3.fill(0x5EED0001, 1, -1.0, 1.0, 0, 1000)
    assert not np.array_equal(a, c)
    aos = oracle_fr3.fill(0x5EED0001, 0, -1.0, 1.0, 0, 1000, layout="aos")
    np.testing.assert_array_equal(aos.T, a)


def test_rollout_oracle_consistency(oracle_fr3):
    rng = np.random.default_rng(4)
    q0, dq0 = rng.uniform(-1, 1, 7), rng.uniform(-1, 1, 7)
    tau = rng.uniform(-5, 5, (5, 7))
    qt, dqt = oracle_fr3.rollout(q0, dq0, tau, 1e-3)
    q, dq = q0.copy(), dq0.copy()
    for t in range(5):
        qdd = oracle_fr3.forward_dynamics(q, dq, tau[t])
        dq = dq + 1e-3 * qdd
        q = q + 1e-3 * dq
        np.testing.assert_allclose(qt[t], q, rtol=0, atol=1e-15)
        np.testing.assert_allclose(dqt[t], dq, rtol=0, atol=1e-15)
