"""ctypes front end of the CPU ORACLE (test infrastructure, NOT product code).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this.  PARITY UNPINNED -- see oracle/rb_oracle.h for what pins the oracle instead.

Also holds the oracle-side URDF reader, an independent mirror of what the reference does at load
time (xurdf 0.2.5 document-order `links` / `joints`, then `Multibody::from_urdf`'s zip + "fixed"
filter, rigidbody/src/multibody.rs:65-77, and `RevoluteJoint::from_xurdf_joint`,
rigidbody/src/joint.rs:53-68).  The product has its own loader in C++ (csrc/urdf.cpp); tests compare
the two.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
import xml.etree.ElementTree as ET
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
MAX_N = 64


# --------------------------------------------------------------------------- URDF (oracle side)
def _floats(s, n, default=0.0):
    if s is None:
        return [default] * n
    v = [float(x) for x in s.split()]
    assert len(v) == n, s
    return v


@dataclass
class ModelArrays:
    """What `from_urdf` keeps: one row per surviving (joint, link) pair, in document order."""
    n: int
    axis: np.ndarray      # [n,3]
    xyz: np.ndarray       # [n,3]  joint origin translation
    rpy: np.ndarray       # [n,3]  joint origin roll/pitch/yaw
    mass: np.ndarray      # [n]
    com: np.ndarray       # [n,3]
    inertia6: np.ndarray  # [n,6]  ixx ixy ixz iyy iyz izz about the COM
    lower: np.ndarray     # [n] joint limits (for sampling synthetic states only)
    upper: np.ndarray
    velocity: np.ndarray
    effort: np.ndarray
    names: list


def parse_urdf(path) -> ModelArrays:
    root = ET.parse(path).getroot()
    links, joints = [], []
    for el in root:                      # direct children only, document order (xurdf)
        if el.tag == "link":
            inert = el.find("inertial")
            if inert is None:            # xurdf: Inertial::default()
                links.append(dict(mass=0.0, com=[0.0] * 3, inertia6=[0.0] * 6))
            else:
                org = inert.find("origin")
                ine = inert.find("inertia")
                links.append(dict(
                    mass=float(inert.find("mass").get("value")),
                    com=_floats(org.get("xyz") if org is not None else None, 3),
                    inertia6=[float(ine.get(k)) for k in ("ixx", "ixy", "ixz", "iyy", "iyz", "izz")]))
        elif el.tag == "joint":
            org = el.find("origin")
            ax = el.find("axis")
            lim = el.find("limit")
            joints.append(dict(
                name=el.get("name"), type=el.get("type"),
                xyz=_floats(org.get("xyz") if org is not None else None, 3),
                rpy=_floats(org.get("rpy") if org is not None else None, 3),
                axis=_floats(ax.get("xyz") if ax is not None else None, 3) if ax is not None else [1.0, 0.0, 0.0],
                lower=float(lim.get("lower", 0.0)) if lim is not None else 0.0,
                upper=float(lim.get("upper", 0.0)) if lim is not None else 0.0,
                velocity=float(lim.get("velocity", 0.0)) if lim is not None else 0.0,
                effort=float(lim.get("effort", 0.0)) if lim is not None else 0.0))
    keep = [(j, l) for j, l in zip(joints, links) if "fixed" not in j["type"]]   # multibody.rs:70-71
    f = lambda key, src: np.array([p[src][key] for p in keep], dtype=np.float64)
    return ModelArrays(
        n=len(keep), axis=f("axis", 0), xyz=f("xyz", 0), rpy=f("rpy", 0),
        mass=f("mass", 1), com=f("com", 1), inertia6=f("inertia6", 1),
        lower=f("lower", 0), upper=f("upper", 0), velocity=f("velocity", 0), effort=f("effort", 0),
        names=[p[0]["name"] for p in keep])


# --------------------------------------------------------------------------- library
def build(fast: bool = False, out_dir: str | None = None) -> str:
    """Compile the oracle with the committed recipe (oracle/Makefile); returns the .so path.  The -march=native
    build (`fast`) goes to `out_dir`, which the caller creates afresh: it is specific to this host, and the tree it
    would otherwise land in may be read-only."""
    if not fast:
        subprocess.run(["make", "-s", "-C", _HERE, "librb_oracle.so"], check=True)
        return os.path.join(_HERE, "librb_oracle.so")
    path = os.path.join(out_dir, "librb_oracle_fast.so")
    subprocess.run(["make", "-s", "-C", _HERE, "FAST_SO=" + path, path], check=True)
    return path


class _MB(C.Structure):
    # opaque, sized generously: rbo_multibody = int + MAX_N * rbo_joint(3+7+1+3+9+9 doubles)
    _fields_ = [("raw", C.c_double * (2 + MAX_N * 32))]


_dp = C.POINTER(C.c_double)


def _p(a):
    return a.ctypes.data_as(_dp)


class Oracle:
    """One loaded model.  All arrays float64; batch layout 'soa' = [n][B], 'aos' = [B][n]."""

    def __init__(self, model: ModelArrays, fast: bool = False):
        if fast:
            with tempfile.TemporaryDirectory(prefix="rb_oracle_") as d:
                lib = C.CDLL(build(True, d))         # stays loaded after its directory is gone
        else:
            lib = C.CDLL(build())
        self.lib = lib
        self.model = model
        self.n = model.n
        lib.rbo_multibody_init.restype = C.c_int
        lib.rbo_forward_dynamics.restype = C.c_int
        lib.rbo_forward_dynamics_batch.restype = C.c_int
        lib.rbo_rollout.restype = C.c_int
        lib.rbo_max_threads.restype = C.c_int
        lib.rbo_sample.restype = C.c_double
        lib.rbo_sample.argtypes = [C.c_uint64, C.c_uint, C.c_uint, C.c_uint64, C.c_double, C.c_double]
        self.mb = _MB()
        c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        self._keep = [c(model.axis), c(model.xyz), c(model.rpy), c(model.mass), c(model.com), c(model.inertia6)]
        rc = lib.rbo_multibody_init(C.byref(self.mb), C.c_int(self.n), *[_p(a) for a in self._keep])
        if rc != 0:
            raise ValueError("rbo_multibody_init failed")

    @classmethod
    def from_urdf(cls, path, fast: bool = False):
        return cls(parse_urdf(path), fast)

    # ---- single state (FFI-shaped: rigidbody_bindings/src/lib.rs:15-70)
    def rnea(self, q, dq, ddq):
        q, dq, ddq = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, dq, ddq))
        tau = np.empty(self.n)
        self.lib.rbo_rnea(C.byref(self.mb), _p(q), _p(dq), _p(ddq), _p(tau))
        return tau

    def crba(self, q):
        q = np.ascontiguousarray(q, dtype=np.float64)
        H = np.empty(self.n * self.n)
        self.lib.rbo_crba(C.byref(self.mb), _p(q), _p(H))
        return H.reshape(self.n, self.n).T.copy()     # column-major -> H[r, c]

    def fwd_kin(self, q):
        q = np.ascontiguousarray(q, dtype=np.float64)
        out = np.empty(3)
        self.lib.rbo_fwd_kin(C.byref(self.mb), _p(q), _p(out))
        return out

    def jac(self, q):
        q = np.ascontiguousarray(q, dtype=np.float64)
        J = np.empty(6 * self.n)
        self.lib.rbo_jac(C.byref(self.mb), _p(q), _p(J))
        return J.reshape(self.n, 6).T.copy()          # column-major 6 x n -> J[r, c]

    def forward_dynamics(self, q, dq, tau):
        q, dq, tau = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, dq, tau))
        qdd = np.empty(self.n)
        rc = self.lib.rbo_forward_dynamics(C.byref(self.mb), _p(q), _p(dq), _p(tau), _p(qdd))
        if rc != 0:
            raise FloatingPointError("mass matrix not positive definite")
        return qdd

    def rollout(self, q0, dq0, tau, dt):
        """tau [H][n] -> (q_traj [H][n], dq_traj [H][n])."""
        q0, dq0, tau = (np.ascontiguousarray(x, dtype=np.float64) for x in (q0, dq0, tau))
        Hn = tau.shape[0]
        qt = np.empty((Hn, self.n)); dqt = np.empty((Hn, self.n))
        rc = self.lib.rbo_rollout(C.byref(self.mb), _p(q0), _p(dq0), _p(tau), C.c_double(dt), C.c_int(Hn), _p(qt), _p(dqt))
        if rc != 0:
            raise FloatingPointError("mass matrix not positive definite")
        return qt, dqt

    # ---- batches
    @staticmethod
    def _B(x, n, layout):
        x = np.ascontiguousarray(x, dtype=np.float64)
        return x, (x.shape[1] if layout == "soa" else x.shape[0])

    def rnea_batch(self, q, dq, ddq, layout="soa", threads=0):
        q, B = self._B(q, self.n, layout)
        dq, _ = self._B(dq, self.n, layout); ddq, _ = self._B(ddq, self.n, layout)
        tau = np.empty_like(q)
        self.lib.rbo_rnea_batch(C.byref(self.mb), _p(q), _p(dq), _p(ddq), _p(tau), C.c_size_t(B),
                                C.c_int(layout == "soa"), C.c_int(threads))
        return tau

    def forward_dynamics_batch(self, q, dq, tau, layout="soa", threads=0):
        q, B = self._B(q, self.n, layout)
        dq, _ = self._B(dq, self.n, layout); tau, _ = self._B(tau, self.n, layout)
        qdd = np.empty_like(q)
        rc = self.lib.rbo_forward_dynamics_batch(C.byref(self.mb), _p(q), _p(dq), _p(tau), _p(qdd), C.c_size_t(B),
                                                 C.c_int(layout == "soa"), C.c_int(threads))
        if rc != 0:
            raise FloatingPointError("mass matrix not positive definite")
        return qdd

    def crba_batch(self, q, layout="soa", threads=0):
        """SoA -> [n*n][B] (entry k = r + n*c), AoS -> [B][n*n] column-major."""
        q, B = self._B(q, self.n, layout)
        shape = (self.n * self.n, B) if layout == "soa" else (B, self.n * self.n)
        H = np.empty(shape)
        self.lib.rbo_crba_batch(C.byref(self.mb), _p(q), _p(H), C.c_size_t(B), C.c_int(layout == "soa"), C.c_int(threads))
        return H

    def rollout_batch(self, q0, dq0, tau, dt):
        """q0,dq0 [n][B]; tau [H][n][B] -> q_traj, dq_traj [H][n][B] (python loop over trajectories: small B only)."""
        Hn, n, B = tau.shape
        qt = np.empty((Hn, n, B)); dqt = np.empty((Hn, n, B))
        for b in range(B):
            a, c = self.rollout(q0[:, b], dq0[:, b], np.ascontiguousarray(tau[:, :, b]), dt)
            qt[:, :, b] = a; dqt[:, :, b] = c
        return qt, dqt

    def max_threads(self):
        return int(self.lib.rbo_max_threads())

    # ---- sampler
    def fill(self, seed, field, lo, hi, first, count, layout="soa"):
        lo = np.ascontiguousarray(np.broadcast_to(lo, (self.n,)), dtype=np.float64)
        hi = np.ascontiguousarray(np.broadcast_to(hi, (self.n,)), dtype=np.float64)
        out = np.empty((self.n, count) if layout == "soa" else (count, self.n))
        self.lib.rbo_fill(_p(out), C.c_uint64(seed), C.c_uint(field), C.c_int(self.n), _p(lo), _p(hi),
                          C.c_size_t(first), C.c_size_t(count), C.c_size_t(count), C.c_int(layout == "soa"))
        return out
