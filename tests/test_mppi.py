"""One MPPI iteration per call (include/rigidbody.h multibody_mppi_step).

The checker restates the header: `mppi_noise_np` is the counter-based normal sampler, `samples_np` the clamped samples,
`weights_np` and `update_np` the softmin weights and the weighted mean, and `mppi_step_np` composes them with the existing
numpy checkers of the rollout cost (`rollout_np`, `quad_cost_np`, `tip_cost_np`, `col_cost_np`).  The CPU tests hold the
sampler to a standard normal and the weights to their invariants.  On the GPU: the samples match the sampler to 1e-13, each
cost is the rollout cost entry's on the returned samples bit for bit, the weights and the update match the formulas applied
to the returned costs and samples to 1e-13, and every layout, memory kind, chunking and multi-device handle gives the same
bits.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import CHAIN32, FR3, TOL
from test_collision_cost import _collision, col_cost_np
from test_rollout_gradients import _aos, _chain_inputs, _dev, _fr3_inputs, _np, _weights, quad_cost_np, rollout_np
from test_rollout_tip_cost import _fr3_chain, _random, _tip, tip_cost_np

GOLDEN = 0x9E3779B97F4A7C15
M64 = (1 << 64) - 1
DT = 2e-3
BAR = 1e-13


# ------------------------------------------------------------------------------------------------ the numpy checker
def mppi_noise_np(seed, s, K, H, n):
    """eps [len(s), H, n] of the global sample indices s (sample k = s mod K of problem s // K): counter
    c = (s H + t) n + i, z = splitmix64(seed + GOLDEN (c + 1)), eps = sqrt(-2 ln u1) cos(2 pi u2); 0 for k = 0."""
    s = np.asarray(s, dtype=np.uint64)
    c = (s[:, None, None] * np.uint64(H) + np.arange(H, dtype=np.uint64)[None, :, None]) * np.uint64(n) \
        + np.arange(n, dtype=np.uint64)[None, None, :]
    with np.errstate(over="ignore"):
        z = np.uint64(seed & M64) + np.uint64(GOLDEN) * (c + np.uint64(1))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    u1 = ((z >> np.uint64(32)).astype(np.float64) + 0.5) * 2.0 ** -32
    u2 = (z & np.uint64(0xFFFFFFFF)).astype(np.float64) * 2.0 ** -32
    eps = np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)
    eps[s % np.uint64(K) == 0] = 0.0
    return eps


def samples_np(u_nom, sigma, lower, upper, seed, K, p_first=0):
    """tau [H, n, P K] (SoA, sample k of problem p at column p K + k) of u_nom [H, n, P]."""
    H, n, P = u_nom.shape
    eps = mppi_noise_np(seed, np.arange(p_first * K, (p_first + P) * K), K, H, n)           # [P K, H, n]
    x = np.repeat(u_nom, K, axis=2) + np.asarray(sigma, dtype=np.float64)[None, :, None] * eps.transpose(1, 2, 0)
    return np.minimum(np.maximum(x, np.asarray(lower)[None, :, None]), np.asarray(upper)[None, :, None])


def weights_np(cost, lam):
    """(w [P, K], eta [P]) of costs [P, K]: w = exp(-(c - m) / lambda) over the finite costs (0 otherwise), m their min."""
    cost = np.asarray(cost, dtype=np.float64)
    fin = np.isfinite(cost)
    m = np.where(fin, cost, np.inf).min(1, keepdims=True)
    with np.errstate(invalid="ignore", over="ignore"):
        w = np.where(fin, np.exp(-(cost - m) / lam), 0.0)
    return w, w.sum(1)


def update_np(w, eta, tau):
    """u_new [H, n, P] = sum_k w tau / eta of the samples tau [H, n, P K]."""
    H, n, PK = tau.shape
    P, K = w.shape
    with np.errstate(invalid="ignore", divide="ignore"):
        return (tau.reshape(H, n, P, K) * w[None, None]).sum(-1) / eta[None, None]


def mppi_step_np(cost_fn, q0, dq0, u_nom, sigma, lower, upper, K, lam, seed):
    """(u_new, cost [P, K], sample weights [P, K], samples) composed from the checkers; cost_fn(q0, dq0, tau) -> [B]."""
    P = np.shape(q0)[1]
    tau = samples_np(u_nom, sigma, lower, upper, seed, K)
    cost = cost_fn(np.repeat(q0, K, axis=1), np.repeat(dq0, K, axis=1), tau).reshape(P, K)
    w, eta = weights_np(cost, lam)
    with np.errstate(invalid="ignore"):
        return update_np(w, eta, tau), cost, w / eta[:, None], tau


def _fr3_cost_fn(orc, ch, dt, tip=None, col=None, **w):
    def f(q0, dq0, tau):
        traj = orc.rollout_batch(q0, dq0, tau, dt) if tau.shape[0] else (np.zeros((0,) + q0.shape), np.zeros((0,) + q0.shape))
        if col is not None:
            return col_cost_np(ch, q0, dq0, tau, dt, *traj, tip or {}, col, **w)
        if tip is not None:
            return tip_cost_np(ch, q0, dq0, tau, dt, *traj, tip, **w)
        return quad_cost_np(q0, dq0, tau, dt, *traj, **w)
    return f


def _effort_bounds(orc):
    eff = orc.model.effort
    return np.where(eff > 0, -eff, -np.inf), np.where(eff > 0, eff, np.inf)


# ------------------------------------------------------------------------------------------------ the checker, on the CPU
def test_noise_is_standard_normal():
    """10^6 draws (K = 4001 samples of H = 25 steps and n = 10 joints, sample 0 left out): a KS test against N(0, 1), the
    mean and the variance, and no correlation between neighbouring samples, steps and joints."""
    K, H, n = 4001, 25, 10
    eps = mppi_noise_np(0x5EED00A1, np.arange(1, K), K, H, n)                 # [K - 1, H, n]
    from scipy import stats
    x = eps.reshape(-1)
    N = x.size
    assert N == 1_000_000
    assert stats.kstest(x, "norm").pvalue > 1e-3
    assert abs(x.mean()) < 5.0 / np.sqrt(N)
    assert abs(x.var() - 1.0) < 5.0 * np.sqrt(2.0 / N)
    for a, b in ((eps[1:], eps[:-1]), (eps[:, 1:], eps[:, :-1]), (eps[:, :, 1:], eps[:, :, :-1])):
        r = np.corrcoef(a.reshape(-1), b.reshape(-1))[0, 1]
        assert abs(r) < 5.0 / np.sqrt(a.size), r


def test_noise_of_sample_zero_is_exactly_zero():
    K, H, n = 17, 6, 7
    eps = mppi_noise_np(123, np.arange(5 * K), K, H, n)
    assert (eps[::K] == 0.0).all()
    assert (eps.reshape(5, K, H, n)[:, 1:] != 0.0).all()


def test_weights_invariants():
    """A constant added to every cost leaves the weights unchanged; lambda -> 0 gives the best sample, lambda -> inf the
    plain mean; a non-finite cost gets weight 0 and a problem without a finite cost gets NaN."""
    rng = np.random.default_rng(0xA2)
    P, K, H, n = 3, 50, 4, 5
    cost = rng.uniform(0, 10, (P, K))
    tau = rng.normal(size=(H, n, P * K))
    w, eta = weights_np(cost, 0.7)
    w2, eta2 = weights_np(cost + 123.25, 0.7)
    np.testing.assert_allclose(w2 / eta2[:, None], w / eta[:, None], rtol=1e-12)
    w, eta = weights_np(cost, 1e-9)
    best = cost.argmin(1)
    np.testing.assert_array_equal(w / eta[:, None], np.eye(K)[best])
    np.testing.assert_allclose(update_np(w, eta, tau), tau.reshape(H, n, P, K)[:, :, np.arange(P), best], rtol=0, atol=0)
    w, eta = weights_np(cost, 1e300)
    np.testing.assert_allclose(update_np(w, eta, tau), tau.reshape(H, n, P, K).mean(-1), rtol=1e-12)
    cost[0, 3], cost[1, :] = np.nan, np.inf
    w, eta = weights_np(cost, 0.7)
    assert w[0, 3] == 0.0 and np.isfinite(update_np(w, eta, tau)[:, :, 0]).all()
    assert eta[1] == 0.0 and np.isnan(update_np(w, eta, tau)[:, :, 1]).all()


def test_step_np_on_fr3(oracle_fr3):
    """The composed checker on FR3: sample 0 is clamp(u_nom) with its rollout cost; sigma = 0 returns clamp(u_nom); the
    samples lie within the bounds."""
    ch = _fr3_chain(oracle_fr3)
    P, K, H = 2, 6, 3
    q0, dq0, u_nom = _fr3_inputs(oracle_fr3, P, H, 0x5EED00A3)
    u_nom = 1.5 * u_nom
    lo, hi = _effort_bounds(oracle_fr3)
    w = _weights(7, 0xA3)
    f = _fr3_cost_fn(oracle_fr3, ch, DT, **w)
    clamp = np.clip(u_nom, lo[None, :, None], hi[None, :, None])
    assert (clamp != u_nom).any()
    u_new, cost, sw, tau = mppi_step_np(f, q0, dq0, u_nom, np.full(7, 5.0), lo, hi, K, 0.5, 7)
    assert ((tau >= lo[None, :, None]) & (tau <= hi[None, :, None])).all()
    np.testing.assert_array_equal(tau[:, :, ::K], clamp)
    np.testing.assert_array_equal(cost[:, 0], f(q0, dq0, clamp))
    np.testing.assert_allclose(sw.sum(1), 1.0, rtol=1e-14)
    u0, *_ = mppi_step_np(f, q0, dq0, u_nom, np.zeros(7), lo, hi, K, 0.5, 7)
    np.testing.assert_allclose(u0, clamp, rtol=1e-15, atol=0)


# ------------------------------------------------------------------------------------------------ on the B200
def _sample_err(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    return float((np.abs(got - ref) / np.maximum(1.0, np.abs(ref))).max())


def _check_formulas(u_new, cost, sw, smp, lam):
    """sample_weights and u_new against weights_np / update_np applied to the returned costs and samples."""
    w, eta = weights_np(cost, lam)
    with np.errstate(invalid="ignore"):
        ref_sw = w / eta[:, None]
    ok = np.isfinite(ref_sw)
    assert (np.isnan(sw) == ~ok).all()
    assert _sample_err(sw[ok], ref_sw[ok]) <= BAR
    ref_u = update_np(w, eta, smp)
    if ref_u.size:
        ok = np.isfinite(ref_u)
        assert (np.isnan(u_new) == ~ok).all()
        assert _sample_err(u_new[ok], ref_u[ok]) <= BAR


def _cost_bits(mb, q0, dq0, dt, K, cost, smp, **kw):
    """cost [P, K] is the rollout cost entry's on the returned samples with q0, dq0 repeated K times, bit for bit."""
    ref = mb.rollout_cost(np.repeat(q0, K, axis=1), np.repeat(dq0, K, axis=1), smp, dt, **kw)
    np.testing.assert_array_equal(np.asarray(cost).reshape(-1), ref, err_msg=mb.kernel_variant)


def _fr3_case(oracle_fr3, P, K, H, seed, scale=1.5):
    q0, dq0, u_nom = _fr3_inputs(oracle_fr3, P, H, seed)
    return q0, dq0, scale * u_nom


@pytest.mark.gpu
def test_samples_match_the_sampler(rb, mb_fr3, oracle_fr3):
    """FR3, P = 3, K = 37, H = 5: the samples are samples_np's to 1e-13; sample 0 is clamp(u_nom) exactly; every sample
    lies within the bounds (the default ones: +-effort); sigma = 0 gives u_new = clamp(u_nom)."""
    P, K, H = 3, 37, 5
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00B1)
    lo, hi = _effort_bounds(oracle_fr3)
    sigma = 0.4 * oracle_fr3.model.effort
    u_new, cost, sw, smp = mb_fr3.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.3, 11, samples=True, **_weights(7, 0xB1))
    assert smp.shape == (H, 7, P * K) and cost.shape == (P, K) and sw.shape == (P, K) and u_new.shape == u_nom.shape
    ref = samples_np(u_nom, sigma, lo, hi, 11, K)
    assert _sample_err(smp, ref) <= BAR
    clamp = np.clip(u_nom, lo[None, :, None], hi[None, :, None])
    assert (clamp != u_nom).any() and (smp == lo[None, :, None]).any() and (smp == hi[None, :, None]).any()
    np.testing.assert_array_equal(smp[:, :, ::K], clamp)
    assert ((smp >= lo[None, :, None]) & (smp <= hi[None, :, None])).all()
    slack = 1e-15 * np.abs(hi)[None, :, None]
    assert ((u_new >= lo[None, :, None] - slack) & (u_new <= hi[None, :, None] + slack)).all()
    _check_formulas(u_new, cost, sw, smp, 0.3)
    u0, *_ = mb_fr3.mppi_step(q0, dq0, u_nom, DT, 0.0, K, 0.3, 11, **_weights(7, 0xB1))
    np.testing.assert_allclose(u0, clamp, rtol=1e-15, atol=0)
    # explicit bounds and unbounded samples
    lo2, hi2 = -0.5 * oracle_fr3.model.effort, 0.25 * oracle_fr3.model.effort
    *_, smp2 = mb_fr3.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.3, 11, limits=(lo2, hi2), samples=True)
    assert _sample_err(smp2, samples_np(u_nom, sigma, lo2, hi2, 11, K)) <= BAR
    *_, smp3 = mb_fr3.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.3, 11, limits=None, samples=True)
    assert _sample_err(smp3, samples_np(u_nom, sigma, np.full(7, -np.inf), np.full(7, np.inf), 11, K)) <= BAR


@pytest.mark.gpu
def test_against_the_composed_checker(rb, mb_fr3, oracle_fr3):
    """FR3 with quadratic, tip and collision terms, P = 4, K = 24, H = 8: costs, sample weights and u_new against
    mppi_step_np on the oracle's rollouts (costs to 1e-10, weights and u_new to 1e-9 relative: the weights amplify
    the costs' rounding by |c - m| / lambda)."""
    P, K, H = 4, 24, 8
    ch = _fr3_chain(oracle_fr3)
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00B2, scale=0.3)
    lo, hi = _effort_bounds(oracle_fr3)
    sigma, lam = 0.1 * oracle_fr3.model.effort, 50.0
    w = _weights(7, 0xB2)
    tip = _tip(0xB2, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    col = _collision(ch, q0, 0xB2)
    got = mb_fr3.mppi_step(q0, dq0, u_nom, DT, sigma, K, lam, 5, tip=tip, collision=col, samples=True, **w)
    ref = mppi_step_np(_fr3_cost_fn(oracle_fr3, ch, DT, tip=tip, col=col, **w), q0, dq0, u_nom, sigma, lo, hi, K, lam, 5)
    assert _sample_err(got[3], ref[3]) <= BAR
    assert _sample_err(got[1], ref[1]) <= TOL
    assert _sample_err(got[2], ref[2]) <= 1e-9
    assert _sample_err(got[0], ref[0]) <= 1e-9
    assert (np.abs(col_cost_np(ch, q0, dq0, u_nom, DT, *oracle_fr3.rollout_batch(q0, dq0, u_nom, DT), {}, col))
            > 0).any()
    _check_formulas(*got, lam)


@pytest.mark.gpu
def test_cost_is_the_rollout_cost_every_family_and_term_set(rb, oracle_fr3):
    """Under every FR3 family, with quadratic terms only, with tip terms and with collision terms: each cost is
    rollout_cost's (multibody_rollout_cost, _tip_cost, _collision_cost) on the returned samples, bit for bit; the samples
    are the same bits under every family."""
    from test_gpu_parity import _variants
    P, K, H = 3, 29, 7
    ch = _fr3_chain(oracle_fr3)
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00B3, scale=0.3)
    w = _weights(7, 0xB3)
    terms = [dict(), dict(tip=_tip(0xB3)), dict(tip=_tip(0xB3), collision=_collision(ch, q0, 0xB3))]
    sigma = 0.2 * oracle_fr3.model.effort
    fams, ref_smp = [], None
    for mb in _variants(rb, FR3):
        fams.append(mb.kernel_variant)
        for kw in terms:
            u_new, cost, sw, smp = mb.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.5, 3, samples=True, **kw, **w)
            _cost_bits(mb, q0, dq0, DT, K, cost, smp, **kw, **w)
            _check_formulas(u_new, cost, sw, smp, 0.5)
            if ref_smp is None:
                ref_smp = smp
            np.testing.assert_array_equal(smp, ref_smp)
    assert fams == ["fr3-specialised", "jit-specialised", "generic-7", "generic-n"]


@pytest.mark.gpu
def test_chain32_every_family(rb, oracle_chain32):
    from oracle.rb_oracle_np import ChainNP
    from test_gpu_parity import _variants
    ch = ChainNP(oracle_chain32.model)
    P, K, H = 2, 19, 5
    rng = np.random.default_rng(0xB4)
    q0, dq0, u_nom = rng.uniform(-1, 1, (32, P)), rng.uniform(-0.5, 0.5, (32, P)), rng.uniform(-0.2, 0.2, (H, 32, P))
    kw = dict(tip=_tip(0xB4), collision=_collision(ch, q0, 0xB4, spheres_per_link=2), **_weights(32, 0xB4))
    fams = []
    for mb in _variants(rb, CHAIN32):
        fams.append(mb.kernel_variant)
        u_new, cost, sw, smp = mb.mppi_step(q0, dq0, u_nom, DT, 0.1, K, 0.5, 4, limits=None, samples=True, **kw)
        assert _sample_err(smp, samples_np(u_nom, np.full(32, 0.1), np.full(32, -np.inf), np.full(32, np.inf), 4, K)) <= BAR
        _cost_bits(mb, q0, dq0, DT, K, cost, smp, **kw)
        _check_formulas(u_new, cost, sw, smp, 0.5)
    assert fams == ["chain32-specialised", "generic-n"]


@pytest.mark.gpu
@pytest.mark.parametrize("n,tree", [(1, False), (2, False), (7, False), (17, False), (40, False), (6, True), (20, True)])
def test_random_chains_and_trees(rb, n, tree):
    mb, ch = _random(n, 0xB50 + n, tree)
    P, K, H = 3, 11, 6
    q0, dq0, u_nom = _chain_inputs(n, P, H, 0xB60 + n)
    kw = dict(tip=_tip(0xB70 + n), collision=_collision(ch, q0, 0xB80 + n, spheres_per_link=2), **_weights(n, 0xB90 + n))
    u_new, cost, sw, smp = mb.mppi_step(q0, dq0, u_nom, DT, 0.3, K, 1.0, n, limits=(-1.5, 1.5), samples=True, **kw)
    assert _sample_err(smp, samples_np(u_nom, np.full(n, 0.3), np.full(n, -1.5), np.full(n, 1.5), n, K)) <= BAR
    _cost_bits(mb, q0, dq0, DT, K, cost, smp, **kw)
    _check_formulas(u_new, cost, sw, smp, 1.0)
    assert np.isfinite(u_new).all()


def _c_call(mb, opt, q0, dq0, u_nom, H, u_new, cost, sw, smp, P, ld, layout, mem, stream=None, qc=None, tc=None, cc=None, dt=DT):
    from rigidbody_rs_b200 import _lib
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data)
    return _lib.lib.multibody_mppi_step(mb._h, p(q0), p(dq0), p(u_nom), dt, H, qc, tc, cc, opt, p(u_new), p(cost), p(sw), p(smp), P, ld,
                                        layout, mem, stream)


def _opt(n, K, lam=0.5, seed=9, sigma=None, lower=None, upper=None):
    from rigidbody_rs_b200 import _lib
    keep = [np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (n,))) if v is not None else None
            for v in (0.5 if sigma is None else sigma, lower, upper)]
    dp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))
    return _lib.RbMppiOptions(sigma=dp(keep[0]), lower=dp(keep[1]), upper=dp(keep[2]), temperature=lam, n_samples=K, seed=seed), keep


@pytest.mark.gpu
@pytest.mark.parametrize("H", [0, 1, 9])
def test_determinism_layouts_memory_and_leading_dimension(rb, mb_fr3, oracle_fr3, H):
    """Same seed, same bits; another seed, other samples; SoA and AoS, host and device, and a NaN-padded ld through the C
    ABI give the same bits; padded columns are not written."""
    from rigidbody_rs_b200 import _lib
    mb = mb_fr3
    P, K = 5, 33
    ch = _fr3_chain(oracle_fr3)
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00B6)
    kw = dict(tip=_tip(0xB6), collision=_collision(ch, q0, 0xB6), **_weights(7, 0xB6))
    sigma = 0.3 * oracle_fr3.model.effort
    host = mb.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.4, 21, samples=True, **kw)
    again = mb.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.4, 21, samples=True, **kw)
    for a, b in zip(host, again):
        np.testing.assert_array_equal(a, b)
    other = mb.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.4, 22, samples=True, **kw)
    if H:                                     # samples at a bound, and sample 0, are the same under both seeds
        free = (np.abs(host[3]) < oracle_fr3.model.effort[None, :, None]) & (np.arange(P * K) % K != 0)[None, None, :]
        assert (other[3] != host[3])[free].all()
    dev = _np(*mb.mppi_step(*_dev(q0, dq0, u_nom), DT, sigma, K, 0.4, 21, samples=True, **kw))
    aos = mb.mppi_step(_aos(q0), _aos(dq0), _aos(u_nom), DT, sigma, K, 0.4, 21, layout="aos", samples=True, **kw)
    aos_dev = _np(*mb.mppi_step(*_dev(_aos(q0), _aos(dq0), _aos(u_nom)), DT, sigma, K, 0.4, 21, layout="aos", samples=True, **kw))
    for k in range(4):
        np.testing.assert_array_equal(dev[k], host[k])
        for a in (aos, aos_dev):
            np.testing.assert_array_equal(a[k], _aos(host[k]) if k in (0, 3) else host[k])
    # without samples the step keeps them in its workspace (another leading dimension): the same bits
    for got, is_aos in ((mb.mppi_step(q0, dq0, u_nom, DT, sigma, K, 0.4, 21, **kw), False),
                        (_np(*mb.mppi_step(*_dev(q0, dq0, u_nom), DT, sigma, K, 0.4, 21, **kw)), False),
                        (mb.mppi_step(_aos(q0), _aos(dq0), _aos(u_nom), DT, sigma, K, 0.4, 21, layout="aos", **kw), True)):
        np.testing.assert_array_equal(got[0], _aos(host[0]) if is_aos else host[0])
        np.testing.assert_array_equal(got[1], host[1])
        np.testing.assert_array_equal(got[2], host[2])
    if H == 0:
        np.testing.assert_array_equal(host[2], np.full((P, K), 1.0 / K))
        _cost_bits(mb, q0, dq0, DT, K, host[1], np.zeros((0, 7, P * K)), **kw)
        np.testing.assert_array_equal(host[1], np.repeat(host[1][:, :1], K, axis=1))
    # padded leading dimension of the per-problem arrays; the samples stay dense
    ld = P + 7
    nan = float("nan")
    qc, keep = mb._quad_cost(**_weights(7, 0xB6))
    from rigidbody_rs_b200 import _collision_cost, _tip_cost
    tc, keep_t = _tip_cost(kw["tip"])
    cc, keep_c = _collision_cost(kw["collision"])
    eff = oracle_fr3.model.effort
    opt, keep_o = _opt(7, K, 0.4, 21, sigma, -eff, eff)
    for mem in (_lib.RB_MEM_DEVICE, _lib.RB_MEM_HOST):
        def wide(x):
            wd = np.full(x.shape[:-1] + (ld,), nan)
            wd[..., :P] = x
            return _dev(wd)[0] if mem == _lib.RB_MEM_DEVICE else wd
        z = lambda shape: _dev(np.full(shape, nan))[0] if mem == _lib.RB_MEM_DEVICE else np.full(shape, nan)
        back = lambda x: x.cpu().numpy() if mem == _lib.RB_MEM_DEVICE else x
        u_new, cost, sw, smp = wide(np.full((H, 7, P), nan)), z(P * K), z(P * K), z((H, 7, P * K))
        rc = _c_call(mb, C.byref(opt), wide(q0), wide(dq0), wide(u_nom), H, u_new, cost, sw, smp, P, ld, _lib.RB_LAYOUT_SOA, mem,
                     qc=C.byref(qc), tc=C.byref(tc), cc=C.byref(cc))
        assert rc == 0, _lib.lib.multibody_last_error()
        mb.sync()
        np.testing.assert_array_equal(back(u_new)[..., :P], host[0])
        assert np.isnan(back(u_new)[..., P:]).all()
        np.testing.assert_array_equal(back(cost), host[1].reshape(-1))
        np.testing.assert_array_equal(back(sw), host[2].reshape(-1))
        np.testing.assert_array_equal(back(smp), host[3])


@pytest.mark.gpu
def test_multi_device_equals_single_device(rb, mb_fr3, oracle_fr3):
    from test_gpu_parity import _two_devices
    mm = rb.Multibody.from_urdf(FR3, devices=_two_devices())
    ch = _fr3_chain(oracle_fr3)
    for P in (7, 1):
        K, H = 13, 6
        q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00B7 + P)
        kw = dict(tip=_tip(0xB7), collision=_collision(ch, q0, 0xB7), **_weights(7, 0xB7))
        for layout, f in (("soa", lambda x: x), ("aos", _aos)):
            a = mm.mppi_step(f(q0), f(dq0), f(u_nom), DT, 20.0, K, 0.5, 77, layout=layout, samples=True, **kw)
            b = mb_fr3.mppi_step(f(q0), f(dq0), f(u_nom), DT, 20.0, K, 0.5, 77, layout=layout, samples=True, **kw)
            for x, y in zip(a, b):
                np.testing.assert_array_equal(x, y)
    with pytest.raises(rb.RigidBodyError) as ei:
        mm.mppi_step(*_dev(q0, dq0, u_nom), DT, 20.0, K, 0.5, 77)
    assert ei.value.code == -6
    mm.close()


@pytest.mark.gpu
def test_chunks_equal_one_problem_calls(rb, mb_fr3, oracle_fr3):
    """P = 4, K = 8192, H = 1000 takes two chunks of two problems (10 launches); each problem's results equal a one-problem
    call's bits.  The one-problem call of problem p uses seed + GOLDEN p K H n, which gives it the batch's counters."""
    import torch
    mb = mb_fr3
    P, K, H, n = 4, 8192, 1000, 7
    q0, dq0, _ = _fr3_inputs(oracle_fr3, P, 0, 0x5EED00B8)
    gen = torch.Generator(device="cuda:0").manual_seed(0xB8)
    eff = torch.from_numpy(oracle_fr3.model.effort).to("cuda:0")[None, :, None]
    u_nom = (torch.rand((H, n, P), dtype=torch.float64, device="cuda:0", generator=gen) * 2 - 1) * 0.2 * eff
    kw = dict(tip=_tip(0xB8), **_weights(7, 0xB8))
    tq, tdq = _dev(q0, dq0)
    sigma = 0.05 * oracle_fr3.model.effort
    l0 = mb.launch_count
    full = mb.mppi_step(tq, tdq, u_nom, 1e-3, sigma, K, 0.5, 1234, **kw)
    torch.cuda.synchronize()
    assert mb.launch_count - l0 == 10
    for p in range(P):
        seed = (1234 + GOLDEN * p * K * H * n) & M64
        one = mb.mppi_step(tq[:, p:p + 1].contiguous(), tdq[:, p:p + 1].contiguous(), u_nom[..., p:p + 1].contiguous(), 1e-3, sigma, K, 0.5,
                           seed, **kw)
        np.testing.assert_array_equal(full[0][..., p:p + 1].cpu().numpy(), one[0].cpu().numpy())
        np.testing.assert_array_equal(full[1][p:p + 1].cpu().numpy(), one[1].cpu().numpy())
        np.testing.assert_array_equal(full[2][p:p + 1].cpu().numpy(), one[2].cpu().numpy())
    assert bool(torch.isfinite(full[0]).all())
    # with samples the rollout reads them in place in one chunk; without, two chunks of the workspace: the same bits,
    # on the device and from the host
    with_s = mb.mppi_step(tq, tdq, u_nom, 1e-3, sigma, K, 0.5, 1234, samples=True, **kw)
    for a, b in zip(full, with_s[:3]):
        np.testing.assert_array_equal(a.cpu().numpy(), b.cpu().numpy())
    del with_s
    torch.cuda.empty_cache()
    hq0, hdq0, hu = q0, dq0, u_nom.cpu().numpy()
    no_s = mb.mppi_step(hq0, hdq0, hu, 1e-3, sigma, K, 0.5, 1234, **kw)
    for a, b in zip(full, no_s):
        np.testing.assert_array_equal(a.cpu().numpy(), b)
    yes_s = mb.mppi_step(hq0, hdq0, hu, 1e-3, sigma, K, 0.5, 1234, samples=True, **kw)
    for a, b in zip(no_s, yes_s[:3]):
        np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_host_call_stages_only_what_it_returns(rb, mb_fr3, oracle_fr3):
    """A host call of P = 1 024 problems of K = 65 536 samples and H = 64 steps without `samples`: its samples (240 GB)
    are neither returned nor staged, and the step runs in chunks of the workspace.  Problems 0 and P - 1 are one-problem
    calls' bits (with the seeds that give them the batch's counters)."""
    mb = mb_fr3
    P, K, H, n = 1024, 65536, 64, 7
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00BB, scale=0.3)
    sigma = 0.1 * oracle_fr3.model.effort
    w = _weights(7, 0xBB)
    u_new, cost, sw = mb.mppi_step(q0, dq0, u_nom, 1e-3, sigma, K, 10.0, 55, **w)
    assert np.isfinite(u_new).all() and np.isfinite(cost).all()
    for p in (0, P - 1):
        seed = (55 + GOLDEN * p * K * H * n) & M64
        one = mb.mppi_step(q0[:, p:p + 1].copy(), dq0[:, p:p + 1].copy(), u_nom[..., p:p + 1].copy(), 1e-3, sigma, K, 10.0, seed, **w)
        np.testing.assert_array_equal(u_new[..., p:p + 1], one[0])
        np.testing.assert_array_equal(cost[p:p + 1], one[1])
        np.testing.assert_array_equal(sw[p:p + 1], one[2])


@pytest.mark.gpu
def test_edge_cases_and_launch_counts(rb, mb_fr3, oracle_fr3):
    """H = 0 (no u_new, uniform weights, the terminal cost), K = 1 (u_new = clamp(u_nom) bit for bit), P = 0; launches per
    chunk: sampler, rollout, weights and the two update stages (3 with H = 0), plus the transposes of AoS calls."""
    import torch
    mb = mb_fr3
    P, K, H = 3, 8, 4
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00B9)
    w = _weights(7, 0xB9)
    lo, hi = _effort_bounds(oracle_fr3)
    u1, c1, s1 = mb.mppi_step(q0, dq0, u_nom, DT, 30.0, 1, 0.5, 3, **w)
    np.testing.assert_array_equal(u1, np.clip(u_nom, lo[None, :, None], hi[None, :, None]))
    np.testing.assert_array_equal(s1, np.ones((P, 1)))
    u0, c0, s0 = mb.mppi_step(q0, dq0, u_nom[:0], DT, 30.0, K, 0.5, 3, **w)
    assert u0.shape == (0, 7, P)
    np.testing.assert_array_equal(s0, np.full((P, K), 1.0 / K))
    np.testing.assert_array_equal(c0, np.repeat(mb.rollout_cost(q0, dq0, u_nom[:0], DT, **w)[:, None], K, axis=1))
    e = mb.mppi_step(np.zeros((7, 0)), np.zeros((7, 0)), np.zeros((H, 7, 0)), DT, 30.0, K, 0.5, 3, samples=True, **w)
    assert e[0].shape == (H, 7, 0) and e[1].shape == (0, K) and e[3].shape == (H, 7, 0)
    d = _dev(q0, dq0, u_nom)
    for h, per in ((H, 5), (0, 3)):
        l0 = mb.launch_count
        mb.mppi_step(d[0], d[1], d[2][:h], DT, 30.0, K, 0.5, 3, **w)
        torch.cuda.synchronize()
        assert mb.launch_count - l0 == per
        l0 = mb.launch_count
        mb.mppi_step(q0, dq0, u_nom[:h], DT, 30.0, K, 0.5, 3, **w)
        assert mb.launch_count - l0 == per
    l0 = mb.launch_count
    mb.mppi_step(_aos(q0), _aos(dq0), _aos(u_nom), DT, 30.0, K, 0.5, 3, layout="aos", samples=True, **w)
    assert mb.launch_count - l0 == 5 + (2 + H) + 2 * H


@pytest.mark.gpu
def test_non_spd_samples_and_non_finite_problems(rb):
    """On a chain whose mass matrix is indefinite for |q_1| >= 0.68: the host call returns RB_ERR_NOT_SPD and still writes
    every output; a sample that meets it costs NaN and weighs 0; a problem with no finite cost, or a non-finite q0, gets NaN
    in u_new and its weights; a device call sets the status word."""
    from rigidbody_rs_b200 import _lib
    from test_rollout_gradients import _spd_where_q1_small
    mb = _spd_where_q1_small(rb)
    P, K, H, dt = 4, 256, 2, 0.1
    q0 = np.zeros((2, P)); q0[1] = [0.0, 0.4, 0.75, 0.0]; q0[0, 3] = np.nan
    dq0 = np.zeros((2, P))
    u_nom = np.zeros((H, 2, P))
    u_new, cost, sw, smp = (np.full(s, -1.0) for s in ((H, 2, P), P * K, P * K, (H, 2, P * K)))
    opt, keep = _opt(2, K, 1.0, 5, sigma=300.0)        # q_1 after one step spreads over about +-10 dt^2 / (unit inertia)
    qc, keep_w = mb._quad_cost(w_q=np.ones(2))
    rc = _c_call(mb, C.byref(opt), q0, dq0, u_nom, H, u_new, cost, sw, smp, P, 0, _lib.RB_LAYOUT_SOA, _lib.RB_MEM_HOST,
                 qc=C.byref(qc), dt=dt)
    assert rc == _lib.RB_ERR_NOT_SPD
    cost, sw = cost.reshape(P, K), sw.reshape(P, K)
    _check_formulas(u_new, cost, sw, smp, 1.0)
    fin = np.isfinite(cost)
    mixed = fin.any(1) & ~fin.all(1)
    assert mixed.any(), fin.sum(1)
    assert (sw[mixed][~fin[mixed]] == 0.0).all()
    assert np.isfinite(u_new[..., mixed]).all()
    for p in (2, 3):
        assert not fin[p].any() and np.isnan(u_new[..., p]).all() and np.isnan(sw[p]).all()
    import torch
    mb.sync()
    mb.mppi_step(*_dev(q0, dq0, u_nom), dt, 300.0, K, 1.0, 5, w_q=np.ones(2))
    torch.cuda.synchronize()
    with pytest.raises(rb.NotPositiveDefinite):
        mb.sync()


@pytest.mark.gpu
def test_error_codes(rb, mb_fr3):
    from rigidbody_rs_b200 import _lib
    mb = mb_fr3
    P, K, H = 2, 4, 3
    q0, dq0, u_nom = np.zeros((7, P)), np.zeros((7, P)), np.zeros((H, 7, P))
    u_new, cost = np.zeros((H, 7, P)), np.zeros(P * K)
    S, A = _lib.RB_LAYOUT_SOA, _lib.RB_MEM_HOST
    ok, keep = _opt(7, K)
    call = lambda opt, **kv: _c_call(mb, opt, kv.get("q0", q0), kv.get("dq0", dq0), kv.get("u_nom", u_nom), kv.get("H", H),
                                     kv.get("u_new", u_new), cost, None, None, kv.get("P", P), kv.get("ld", 0), kv.get("layout", S),
                                     kv.get("mem", A))
    assert call(C.byref(ok)) == 0
    assert call(None) == _lib.RB_ERR_NULL
    no_sigma = _lib.RbMppiOptions(temperature=1.0, n_samples=K)
    assert call(C.byref(no_sigma)) == _lib.RB_ERR_NULL
    for name in ("q0", "dq0", "u_nom", "u_new"):
        assert call(C.byref(ok), **{name: None}) == _lib.RB_ERR_NULL, name
    assert call(C.byref(ok), u_nom=None, u_new=None, H=0) == 0
    for name in ("q0", "dq0"):                # H = 0 still needs the start state when costs are asked for
        assert call(C.byref(ok), u_nom=None, u_new=None, H=0, **{name: None}) == _lib.RB_ERR_NULL, name
    bad = [_opt(7, 0), _opt(7, -3), _opt(7, K, lam=0.0), _opt(7, K, lam=-1.0), _opt(7, K, lam=float("inf")), _opt(7, K, lam=float("nan")),
           _opt(7, K, sigma=-0.1), _opt(7, K, sigma=float("nan")), _opt(7, K, sigma=float("inf")),
           _opt(7, K, lower=float("nan")), _opt(7, K, upper=float("nan")), _opt(7, K, lower=1.0, upper=0.5)]
    for o, keep_b in bad:
        assert call(C.byref(o)) == _lib.RB_ERR_ARG
    for kv in (dict(layout=7), dict(mem=7), dict(H=-1), dict(ld=1)):
        assert call(C.byref(ok), **kv) == _lib.RB_ERR_ARG, kv
    assert _lib.lib.multibody_mppi_step(mb._h, None, None, None, float("nan"), H, None, None, None, C.byref(ok), None, None, None, None, 0, 0, S,
                                        A, None) == _lib.RB_ERR_ARG
    assert _lib.lib.multibody_mppi_step(None, None, None, None, DT, H, None, None, None, C.byref(ok), None, None, None, None, 0, 0, S, A,
                                        None) == _lib.RB_ERR_NULL
    assert call(C.byref(ok), P=0, q0=None, dq0=None, u_nom=None, u_new=None) == 0
    with pytest.raises(rb.RigidBodyError):
        mb.mppi_step(q0, dq0, u_nom, DT, 0.5, K, 0.5, 1, w_q=-np.ones(7))
    with pytest.raises(rb.RigidBodyError):
        mb.mppi_step(q0, dq0, u_nom, DT, 0.5, K, 0.5, 1, collision=dict(link=[9], center=np.zeros((1, 3)), radius=[0.1], kind=["sphere"],
                                                                         obstacle=np.zeros((1, 4)), w=1.0))


@pytest.mark.gpu
@pytest.mark.parametrize("P,K", [(1, 65536), (64, 1024)])
def test_full_size_fr3(rb, mb_fr3, oracle_fr3, P, K):
    """FR3, H = 64, device-resident, with tip and collision terms: the costs are rollout_cost's on the returned samples
    bit for bit, 256 strided samples match the sampler, 128 strided costs match the checker on the oracle's rollouts, and
    the weights and u_new match the formulas applied to the returned costs and samples."""
    import torch
    mb = mb_fr3
    H, dt = 64, 1e-3
    ch = _fr3_chain(oracle_fr3)
    q0, dq0, u_nom = _fr3_case(oracle_fr3, P, K, H, 0x5EED00BA + P, scale=0.3)
    w = _weights(7, 0xBA)
    tip = _tip(0xBA, pose=tuple(x[0] for x in ch.fwd_kin(q0[:, :1].T)))
    col = _collision(ch, q0, 0xBA)
    kw = dict(tip=tip, collision=col, **w)
    sigma, lam = 0.1 * oracle_fr3.model.effort, 5.0
    d = _dev(q0, dq0, u_nom)
    u_new, cost, sw, smp = mb.mppi_step(*d, dt, sigma, K, lam, 99, samples=True, **kw)
    ref = mb.rollout_cost(d[0].repeat_interleave(K, 1).contiguous(), d[1].repeat_interleave(K, 1).contiguous(), smp, dt, **kw)
    np.testing.assert_array_equal(cost.reshape(-1).cpu().numpy(), ref.cpu().numpy())
    del ref
    u_new, cost, sw = u_new.cpu().numpy(), cost.cpu().numpy(), sw.cpu().numpy()
    smp_h = smp.cpu().numpy()
    del smp, d
    torch.cuda.empty_cache()
    assert np.isfinite(cost).all()
    _check_formulas(u_new, cost, sw, smp_h, lam)
    lo, hi = _effort_bounds(oracle_fr3)
    idx = np.arange(0, P * K, P * K // 256)
    eps = mppi_noise_np(99, idx, K, H, 7)
    x = u_nom[:, :, idx // K] + sigma[None, :, None] * eps.transpose(1, 2, 0)
    assert _sample_err(smp_h[:, :, idx], np.clip(x, lo[None, :, None], hi[None, :, None])) <= BAR
    idx = np.arange(0, P * K, P * K // 128)
    s0, s1, st = q0[:, idx // K], dq0[:, idx // K], smp_h[:, :, idx].copy()
    traj = oracle_fr3.rollout_batch(s0, s1, st, dt)
    assert _sample_err(cost.reshape(-1)[idx], col_cost_np(ch, s0, s1, st, dt, *traj, tip, col, **w)) <= TOL
