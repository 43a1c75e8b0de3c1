"""Which kernel family serves which chain, which kernels serve the entries a family leaves to the run-time-n family,
and how many launches each entry point issues.

The other GPU tests hold every family to the oracle within a tolerance; these pin the dispatch itself:
  * the family `RIGIDBODY_B200_VARIANT` / `RIGIDBODY_B200_JIT` select for each kind of chain, or the status and
    message the constructor returns;
  * entries the chain32 and jit-long families do not have give exactly the bits of a generic-n engine of the same
    chain, and in the two-launch path of rnea_fd the tau half is the engine's own rnea;
  * the multibody_gpu_launch_count delta of one call per entry point, family by family.
"""
import os

import numpy as np
import pytest

from conftest import CHAIN32, FR3
from test_host import _random_chain, _random_tree

pytestmark = pytest.mark.gpu

ARG, UNSUPPORTED = -2, -6
NAMES = ["auto", "fr3-specialised", "chain32-specialised", "jit-specialised", "jit-long", "generic-7", "generic-n",
         "no-such-family"]


def _chain(name):
    """(constructor keyword arguments, is a tree) of one test chain."""
    if name == "fr3":
        return dict(urdf=FR3), False
    if name == "chain32":
        return dict(urdf=CHAIN32), False
    kind, n = name.split()
    n = int(n)
    if kind == "serial":
        R, t, m, c, Ic = _random_chain(n, 300 + n)
        return dict(arrays=(R, t * min(1.0, 8.0 / n), m, c, Ic)), False      # reach (and cond(H)) as for short chains
    seed = {5: 1, 20: 3}[n]
    ax = np.random.default_rng(seed).normal(size=(n, 3))
    return dict(arrays=_random_chain(n, 70 + seed), axis=ax, parent=_random_tree(n, seed)), True


def _make(rb, name, variant=None, jit=None):
    """An engine for chain `name`, built with the two selection variables set as given (None = unset)."""
    spec, _ = _chain(name)
    saved = {k: os.environ.pop(k, None) for k in ("RIGIDBODY_B200_VARIANT", "RIGIDBODY_B200_JIT")}
    try:
        if variant is not None:
            os.environ["RIGIDBODY_B200_VARIANT"] = variant
        if jit is not None:
            os.environ["RIGIDBODY_B200_JIT"] = jit
        if "urdf" in spec:
            return rb.Multibody.from_urdf(spec["urdf"])
        return rb.Multibody.from_descriptor(*spec["arrays"], axis=spec.get("axis"), parent=spec.get("parent"))
    finally:
        for k, v in saved.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


@pytest.fixture(scope="module", autouse=True)
def _private_jit_cache(tmp_path_factory):
    """One kernel cache for the module: every chain is compiled once, whatever $HOME is."""
    old = os.environ.get("RIGIDBODY_B200_CACHE")
    os.environ["RIGIDBODY_B200_CACHE"] = str(tmp_path_factory.mktemp("jit_cache"))
    yield
    os.environ.pop("RIGIDBODY_B200_CACHE", None)
    if old is not None:
        os.environ["RIGIDBODY_B200_CACHE"] = old


# chain -> (family of `auto`, family of `auto` with RIGIDBODY_B200_JIT=0, the explicit names that succeed)
SELECTION = {
    "fr3": ("fr3-specialised", "fr3-specialised", {"fr3-specialised", "jit-specialised", "generic-7", "generic-n"}),
    "chain32": ("chain32-specialised", "chain32-specialised", {"chain32-specialised", "jit-long", "generic-n"}),
    "serial 5": ("jit-specialised", "generic-n", {"jit-specialised", "generic-n"}),
    "serial 7": ("jit-specialised", "generic-7", {"jit-specialised", "generic-7", "generic-n"}),
    "serial 20": ("jit-long", "generic-n", {"jit-long", "generic-n"}),
    "serial 40": ("generic-n", "generic-n", {"generic-n"}),
    "tree 5": ("jit-specialised", "generic-n", {"jit-specialised", "generic-n"}),
    "tree 20": ("generic-n", "generic-n", {"generic-n"}),
}

REFUSALS = {
    "fr3-specialised": "RIGIDBODY_B200_VARIANT=fr3-specialised but the chain is not the compiled-in FR3 model",
    "chain32-specialised": "RIGIDBODY_B200_VARIANT=chain32-specialised but the chain is not the compiled-in 32-joint model",
    "jit-specialised": "RIGIDBODY_B200_VARIANT=jit-specialised needs a chain of at most 18 joints",
    "jit-long": "RIGIDBODY_B200_VARIANT=jit-long serves chains of 19..32 joints",
    "generic-7": "RIGIDBODY_B200_VARIANT=generic-7 needs a 7-joint chain",
}


def _refusal(name, tree):
    """(status, message) the constructor returns for a name that cannot serve the chain."""
    if tree and name not in ("jit-specialised", "generic-n"):
        # an unknown name on a tree is refused like a serial-only family, not as an unknown name
        return UNSUPPORTED, f"RIGIDBODY_B200_VARIANT={name} serves serial chains only; trees run on jit-specialised or generic-n"
    if name not in REFUSALS:
        return ARG, f"unknown RIGIDBODY_B200_VARIANT '{name}'"
    return UNSUPPORTED, REFUSALS[name]


@pytest.mark.parametrize("chain", list(SELECTION))
def test_family_selection_table(rb, chain):
    auto, auto_nojit, explicit = SELECTION[chain]
    tree = _chain(chain)[1]
    bad = []
    for jit in (None, "0"):
        for name in NAMES:
            if name == "auto":
                want = auto if jit is None else auto_nojit
            else:
                want = name if name in explicit else None
            try:
                mb = _make(rb, chain, name, jit)
            except rb.RigidBodyError as e:
                code, msg = _refusal(name, tree)
                if want is not None or e.code != code or str(e) != f"[{code}] {msg}":
                    bad.append((name, jit, want, str(e)))
                continue
            got, note = mb.kernel_variant, mb._note()
            mb.close()
            if got != want or (tree and "kinematic tree" not in note):
                bad.append((name, jit, want, got, note))
    assert not bad, bad


# ---------------------------------------------------------------- entries served by the run-time-n family
B_RAGGED = 1000 + 37
H_ROLL = 3


def _inputs(n, B, seed):
    rng = np.random.default_rng(seed)
    q, dq, ddq, tau = rng.uniform(-2, 2, (B, n)), rng.uniform(-1, 1, (B, n)), rng.uniform(-5, 5, (B, n)), rng.uniform(-5, 5, (B, n))
    tau_h = rng.uniform(-5, 5, (H_ROLL, B, n))
    return q, dq, ddq, tau, tau_h


def _as(place, x):
    """AoS host array -> the layout and memory of `place` ('aos host' or 'soa device')."""
    if place == "aos host":
        return np.ascontiguousarray(x)
    import torch
    x = np.swapaxes(x, -1, -2)                                 # [.., B, n] -> [.., n, B]
    return torch.from_numpy(np.ascontiguousarray(x)).to("cuda:0")


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


@pytest.mark.parametrize("place", ["soa device", "aos host"])
@pytest.mark.parametrize("chain,family,fallback", [
    ("chain32", "chain32-specialised", ("fd", "fwd_kin", "jac", "rollout", "rollout_cost")),
    ("serial 20", "jit-long", ("fd", "rollout", "rollout_cost")),
], ids=["chain32", "jit-long"])
def test_fallback_entries_are_the_generic_n_kernels(rb, chain, family, fallback, place):
    mb = _make(rb, chain)
    gen = _make(rb, chain, "generic-n")
    assert mb.kernel_variant == family and gen.kernel_variant == "generic-n"
    n = mb.n
    q, dq, ddq, tau, tau_h = (_as(place, x) for x in _inputs(n, B_RAGGED, 7))
    lay = "aos" if place == "aos host" else "soa"
    w = np.linspace(0.5, 2.0, n)
    entries = {
        "fd": lambda m: m.forward_dynamics(q, dq, tau, layout=lay),
        "fwd_kin": lambda m: m.fwd_kin(q, layout=lay),
        "jac": lambda m: m.jac(q, layout=lay),
        "rollout": lambda m: m.rollout(q, dq, tau_h, 1e-3, layout=lay, final=True),
        "rollout_cost": lambda m: m.rollout_cost(q, dq, tau_h, 1e-3, w_q=w, w_dq=0.1 * w, w_tau=1e-3 * w, w_q_final=3 * w,
                                                 layout=lay),
    }
    for name in fallback:
        a, b = entries[name](mb), entries[name](gen)
        a, b = (a, b) if isinstance(a, tuple) else ((a,), (b,))
        for x, y in zip(a, b):
            np.testing.assert_array_equal(_np(x), _np(y), err_msg=f"{family} {name} {place}")
    # rnea_fd has no fused kernel here: tau from the family's own rnea, qdd from the generic-n forward dynamics
    both = _np(mb.rnea_fd(q, dq, ddq, tau, layout=lay))
    t_half, a_half = (both[:, :n], both[:, n:]) if lay == "aos" else (both[:n], both[n:])
    np.testing.assert_array_equal(t_half, _np(mb.rnea(q, dq, ddq, layout=lay)), err_msg=f"{family} rnea_fd tau {place}")
    np.testing.assert_array_equal(a_half, _np(gen.forward_dynamics(q, dq, tau, layout=lay)), err_msg=f"{family} rnea_fd qdd {place}")


# ---------------------------------------------------------------- launch counts
# One call of each entry point.  SoA (device or one host chunk): one launch, two for rnea_fd where the family has no
# fused kernel.  AoS device batches: families without in-kernel AoS staging transpose each input and the output
# (n_in + 2); the rollouts stage through transposes for every family (2 + H in, 2H out of the trajectory).
# fp32 entries exist on the register-resident families only (None = RB_ERR_UNSUPPORTED).
_WITH_AOS = {"soa device": dict(rnea=1, fd=1, rnea_fd=1, crba=1, fwd_kin=1, jac=1, rollout=1, rollout_cost=1, rnea_f32=1, fd_f32=1),
             "aos device": dict(rnea=1, fd=1, rnea_fd=6, crba=3, fwd_kin=3, jac=3, rollout=9, rollout_cost=5),
             "soa host": dict(rnea=1, fd=1, rnea_fd=1, crba=1, fwd_kin=1, jac=1, rollout=1, rollout_cost=1)}
_NO_AOS = {"soa device": dict(rnea=1, fd=1, rnea_fd=2, crba=1, fwd_kin=1, jac=1, rollout=1, rollout_cost=1, rnea_f32=None, fd_f32=None),
           "aos device": dict(rnea=5, fd=5, rnea_fd=7, crba=3, fwd_kin=3, jac=3, rollout=9, rollout_cost=5),
           "soa host": dict(rnea=1, fd=1, rnea_fd=2, crba=1, fwd_kin=1, jac=1, rollout=1, rollout_cost=1)}
LAUNCHES = {
    ("fr3", None, None): ("fr3-specialised", _WITH_AOS),
    ("serial 5", None, None): ("jit-specialised", _WITH_AOS),
    ("serial 7", None, "0"): ("generic-7", _WITH_AOS),
    ("chain32", None, None): ("chain32-specialised", _NO_AOS),
    ("serial 20", None, None): ("jit-long", _NO_AOS),
    ("serial 40", None, None): ("generic-n", _NO_AOS),
}


@pytest.mark.parametrize("key", list(LAUNCHES), ids=lambda k: LAUNCHES[k][0])
def test_launch_counts(rb, key):
    import torch
    family, want = LAUNCHES[key]
    mb = _make(rb, *key)
    assert mb.kernel_variant == family
    n, B, H = mb.n, 1037, 2
    q, dq, ddq, tau, _ = _inputs(n, B, 11)
    tau_h = np.random.default_rng(12).uniform(-5, 5, (H, B, n))
    w = np.linspace(0.5, 2.0, n)
    got = {}
    for place in want:
        lay = "aos" if place.startswith("aos") else "soa"
        if lay == "aos":
            x = [np.ascontiguousarray(a) for a in (q, dq, ddq, tau, tau_h)]
        else:
            x = [np.ascontiguousarray(np.swapaxes(a, -1, -2)) for a in (q, dq, ddq, tau, tau_h)]
        if place.endswith("device"):
            x = [torch.from_numpy(a).to("cuda:0") for a in x]
        xq, xdq, xddq, xtau, xh = x
        calls = {
            "rnea": lambda: mb.rnea(xq, xdq, xddq, layout=lay),
            "fd": lambda: mb.forward_dynamics(xq, xdq, xtau, layout=lay),
            "rnea_fd": lambda: mb.rnea_fd(xq, xdq, xddq, xtau, layout=lay),
            "crba": lambda: mb.crba(xq, layout=lay),
            "fwd_kin": lambda: mb.fwd_kin(xq, layout=lay),
            "jac": lambda: mb.jac(xq, layout=lay),
            "rollout": lambda: mb.rollout(xq, xdq, xh, 1e-3, layout=lay),
            "rollout_cost": lambda: mb.rollout_cost(xq, xdq, xh, 1e-3, w_q=w, w_dq=w, layout=lay),
            "rnea_f32": lambda: mb.rnea(xq.float(), xdq.float(), xddq.float()),
            "fd_f32": lambda: mb.forward_dynamics(xq.float(), xdq.float(), xtau.float()),
        }
        for entry in want[place]:
            l0 = mb.launch_count
            try:
                calls[entry]()
                got[place, entry] = mb.launch_count - l0
            except rb.RigidBodyError as e:
                got[place, entry] = None if e.code == UNSUPPORTED and mb.launch_count == l0 else str(e)
        mb.sync()
    expect = {(p, e): v for p, d in want.items() for e, v in d.items()}
    assert got == expect, {k: (got[k], expect[k]) for k in expect if got.get(k) != expect[k]}
