"""rigidbody_rs_b200 -- host-side mirror of the reference's `Multibody` API over the B200 engine.

The reference exposes one type, `rigidbody::multibody::Multibody` (rigidbody/src/multibody.rs:32,64-175), with
`from_urdf`, `rnea`, `crba`, `fwd_kin`, `jac`; its FFI crate (rigidbody_bindings/src/lib.rs) wraps each for one
state.  This module keeps those names and argument meanings and accepts either one state (a length-n vector,
exactly the reference call) or a batch.  Every call goes through the C ABI in include/rigidbody.h into
hand-written sm_100a kernels; nothing here computes dynamics in Python and nothing falls back to the CPU.

Batches:
  * layout="soa": arrays shaped [n, B] (joint-major; the engine's native, coalesced layout)
  * layout="aos": arrays shaped [B, n] (the reference's double[7], repeated)
  * numpy arrays are host memory (copied in and out, pipelined); torch CUDA float64 tensors are used in place
    on the current torch stream (asynchronous; no copy).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (NotPositiveDefinite, RigidBodyError, RB_LAYOUT_AOS, RB_LAYOUT_SOA, RB_MEM_DEVICE, RB_MEM_HOST,
                   check, lib)

__all__ = ["Multibody", "RigidBodyError", "NotPositiveDefinite", "host_empty"]


def _is_torch(x):
    return type(x).__module__.startswith("torch")


class _Arg:
    """Pointer + placement of one array argument."""

    def __init__(self, x, name):
        self.torch = _is_torch(x)
        if self.torch:
            import torch
            if x.dtype != torch.float64:
                raise TypeError(f"{name}: torch tensors must be float64 (Real = f64, rigidbody/src/lib.rs:15); "
                                f"float32 is accepted by rnea / forward_dynamics only (fp32 mode)")
            if not x.is_contiguous():
                raise ValueError(f"{name}: tensor must be contiguous")
            self.device = x.device
            self.cuda = x.is_cuda
            self.arr = x
            self.ptr = x.data_ptr()
            self.shape = tuple(x.shape)
        else:
            a = np.ascontiguousarray(x, dtype=np.float64)
            self.cuda = False
            self.arr = a
            self.ptr = a.ctypes.data
            self.shape = a.shape


def host_empty(shape):
    """A float64 numpy array backed by pinned host memory (multibody_host_alloc), for full-rate PCIe copies."""
    n = int(np.prod(shape))
    p = C.c_void_p()
    check(lib.multibody_host_alloc(C.byref(p), n * 8))
    buf = (C.c_double * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.float64).reshape(shape)
    _PINNED[arr.ctypes.data] = p.value
    return arr


_PINNED = {}


def host_free(arr):
    p = _PINNED.pop(arr.ctypes.data, None)
    if p is not None:
        lib.multibody_host_free(C.c_void_p(p))


class Multibody:
    """A kinematic chain resident on one B200.  Mirrors rigidbody::multibody::Multibody."""

    def __init__(self, handle, owns=True):
        self._h = handle
        self._owns = owns
        self.n = lib.multibody_gpu_n_joints(handle)
        self.device = lib.multibody_gpu_device(handle)
        self.kernel_variant = lib.multibody_gpu_kernel_variant(handle).decode()

    # ---- construction (multibody.rs:65-77)
    @classmethod
    def from_urdf(cls, path, device=0, devices=None):
        """`devices` (a list of CUDA ordinals) builds ONE engine over several GPUs (multibody_gpu_new_multi_from_urdf):
        host batches are cut into contiguous slices, one per device; device tensors then go to `peer(i)`."""
        h = C.c_void_p()
        if devices is not None:
            arr = (C.c_int * len(devices))(*[int(d) for d in devices])
            check(lib.multibody_gpu_new_multi_from_urdf(str(path).encode(), arr, len(devices), C.byref(h)))
        else:
            check(lib.multibody_gpu_new_from_urdf(str(path).encode(), int(device), C.byref(h)))
        return cls(h)

    @property
    def n_devices(self):
        return lib.multibody_gpu_n_devices(self._h)

    def peer(self, index):
        """The single-device engine of device slot `index` of a multi-device engine (owned by this object)."""
        h = lib.multibody_gpu_peer(self._h, int(index))
        if not h:
            check(_lib.RB_ERR_ARG)
        m = Multibody(C.c_void_p(h), owns=False)
        m._parent = self          # keeps the owner alive
        return m

    def copy_peak(self, h2d_bytes, d2h_bytes, reps=3):
        """Bare pinned-copy ceiling of the host path (multibody_gpu_measure_copy_peak): (h2d GB/s, d2h GB/s), both
        directions at once, summed over the devices of the engine."""
        a, b = C.c_double(), C.c_double()
        check(lib.multibody_gpu_measure_copy_peak(self._h, int(h2d_bytes), int(d2h_bytes), int(reps), C.byref(a), C.byref(b)))
        return a.value, b.value

    @classmethod
    def from_descriptor(cls, parent_rot, parent_trans, mass, com, inertia_com, gravity=(0.0, 0.0, 9.81),
                        axis=None, parent=None, device=0):
        """Flattened chain descriptor (include/rigidbody.h RbChainDesc): what the Rust side extracts from
        Multibody::iter() (multibody.rs:79-81; joint.rs:26-31; inertia.rs:12-17)."""
        f = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        R, t, m, c, Ic = f(parent_rot), f(parent_trans), f(mass), f(com), f(inertia_com)
        n = int(m.shape[0])
        d = _lib.RbChainDesc()
        d.n_joints = n
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        keep = [R, t, m, c, Ic]
        d.parent_rot, d.parent_trans, d.mass, d.com, d.inertia_com = dp(R), dp(t), dp(m), dp(c), dp(Ic)
        if axis is not None:
            ax = f(axis); keep.append(ax); d.axis = dp(ax)
        if parent is not None:
            pa = np.ascontiguousarray(parent, dtype=np.int32); keep.append(pa)
            d.parent = pa.ctypes.data_as(C.POINTER(C.c_int32))
        d.gravity[:] = list(gravity)
        h = C.c_void_p()
        check(lib.multibody_gpu_new(C.byref(d), int(device), C.byref(h)))
        return cls(h)

    def close(self):
        if self._h is not None and self._owns:
            lib.multibody_gpu_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- introspection
    def model(self):
        n = self.n
        R, t, m, h, I = np.empty((n, 3, 3)), np.empty((n, 3)), np.empty(n), np.empty((n, 3)), np.empty((n, 6))
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        check(lib.multibody_gpu_get_model(self._h, dp(R), dp(t), dp(m), dp(h), dp(I)))
        return dict(parent_rot=R, parent_trans=t, mass=m, h=h, inertia_origin=I)

    def limits(self):
        L = _lib.RbJointLimits()
        check(lib.multibody_gpu_get_limits(self._h, C.byref(L)))
        return {k: np.array(getattr(L, k)[: self.n]) for k in ("lower", "upper", "velocity", "effort")}

    def _note(self):
        """Why this kernel family serves the chain (e.g. 'kernels compiled with NVRTC')."""
        return lib.multibody_gpu_family_note(self._h).decode()

    @property
    def launch_count(self):
        return int(lib.multibody_gpu_launch_count(self._h))

    def sync(self):
        check(lib.multibody_gpu_sync(self._h))

    def fp64_peak_tflops(self, millis=50):
        out = C.c_double()
        check(lib.multibody_gpu_measure_fp64_peak(self._h, int(millis), C.byref(out)))
        return out.value

    # ---- argument plumbing
    def _prep(self, arrays, names, layout, per_state_in):
        args = [_Arg(a, nm) for a, nm in zip(arrays, names)]
        cuda = args[0].cuda
        if any(a.cuda != cuda for a in args):
            raise ValueError("all arrays of one call must live in the same place (all host or all CUDA)")
        a0 = args[0]
        single = len(a0.shape) == 1
        if single:
            B, lay = 1, RB_LAYOUT_AOS
            for a, per in zip(args, per_state_in):
                if a.shape != (per,):
                    raise ValueError(f"expected a vector of length {per}, got shape {a.shape}")
        else:
            if layout not in ("soa", "aos"):
                raise ValueError("layout must be 'soa' ([n, B]) or 'aos' ([B, n])")
            lay = RB_LAYOUT_SOA if layout == "soa" else RB_LAYOUT_AOS
            B = a0.shape[1] if layout == "soa" else a0.shape[0]
            for a, per in zip(args, per_state_in):
                want = (per, B) if layout == "soa" else (B, per)
                if a.shape != want:
                    raise ValueError(f"expected shape {want} for layout '{layout}', got {a.shape}")
        return args, cuda, single, B, lay

    def _out(self, like, cuda, single, B, lay, per_state_out, out):
        shape = (per_state_out,) if single else ((per_state_out, B) if lay == RB_LAYOUT_SOA else (B, per_state_out))
        if out is not None:
            o = _Arg(out, "out")
            if o.shape != shape or o.cuda != cuda:
                raise ValueError(f"out must have shape {shape} and live with the inputs")
            if not o.torch and o.arr is not out:
                raise ValueError("out must be a contiguous float64 array")
            return o
        if cuda:
            import torch
            return _Arg(torch.empty(shape, dtype=torch.float64, device=like.device), "out")
        return _Arg(np.empty(shape, dtype=np.float64), "out")

    @staticmethod
    def _stream(cuda, like):
        if not cuda:
            return None
        import torch
        return C.c_void_p(torch.cuda.current_stream(like.device).cuda_stream)

    def _call(self, fn, arrays, names, per_in, per_out, layout, out):
        args, cuda, single, B, lay = self._prep(arrays, names, layout, per_in)
        o = self._out(args[0], cuda, single, B, lay, per_out, out)
        if cuda and args[0].device.index not in (None, self.device):
            raise ValueError(f"tensors are on cuda:{args[0].device.index}, engine is on cuda:{self.device}")
        mem = RB_MEM_DEVICE if cuda else RB_MEM_HOST
        check(fn(self._h, *[C.c_void_p(a.ptr) for a in args], C.c_void_p(o.ptr), B, 0, lay, mem,
                 self._stream(cuda, args[0])))
        return o.arr

    def _call_f32(self, fn, a, b, c, out):
        """fp32 mode: CUDA float32 tensors shaped [n, B] only (include/rigidbody.h multibody_*_batch_f32)."""
        import torch
        n = self.n
        ts = (a, b, c)
        if not all(_is_torch(t) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and tuple(t.shape) == tuple(a.shape) for t in ts) \
                or a.dim() != 2 or a.shape[0] != n:
            raise ValueError("fp32 mode takes contiguous CUDA float32 tensors shaped [n, B] (layout 'soa')")
        if out is None:
            out = torch.empty_like(a)
        B = a.shape[1]
        check(fn(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(c.data_ptr()), C.c_void_p(out.data_ptr()),
                 B, B, C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)))
        return out

    @staticmethod
    def _is_f32(x):
        if not _is_torch(x):
            return False
        import torch
        return x.dtype == torch.float32

    # ---- the reference's operations, batched
    def rnea(self, q, dq, ddq, layout="soa", out=None):
        """tau = ID(q, dq, ddq)  (multibody.rs:111-153 after get_transforms :83-85; FFI lib.rs:15-30)."""
        n = self.n
        if self._is_f32(q):
            return self._call_f32(lib.multibody_rnea_batch_f32, q, dq, ddq, out)
        return self._call(lib.multibody_rnea_batch, (q, dq, ddq), ("q", "dq", "ddq"), (n, n, n), n, layout, out)

    def forward_dynamics(self, q, dq, tau, layout="soa", out=None):
        """qdd = chol_solve(sym(crba(q)), tau - rnea(q, dq, 0))  (SURVEY.md 3.3; not a reference function)."""
        n = self.n
        if self._is_f32(q):
            return self._call_f32(lib.multibody_forward_dynamics_batch_f32, q, dq, tau, out)
        return self._call(lib.multibody_forward_dynamics_batch, (q, dq, tau), ("q", "dq", "tau"), (n, n, n), n, layout, out)

    def rnea_fd(self, q, dq, ddq, tau, layout="soa", out=None):
        """tau_out = rnea(q, dq, ddq) and qdd = forward_dynamics(q, dq, tau) of the same states in one call
        (include/rigidbody.h multibody_rnea_fd_batch): q and dq are transferred once.  Returns the packed result,
        soa [2n, B] (rows 0..n-1 tau, n..2n-1 qdd) or aos [B, 2n]; one state -> (tau, qdd)."""
        n = self.n
        D = self._call(lib.multibody_rnea_fd_batch, (q, dq, ddq, tau), ("q", "dq", "ddq", "tau"), (n, n, n, n), 2 * n, layout, out)
        if len(D.shape) == 1:
            return D[:n], D[n:]
        return D

    def rnea_derivatives(self, q, dq, ddq, layout="soa", out=None):
        """Analytical d tau / d q and d tau / d dq of tau = rnea(q, dq, ddq), packed as the C ABI returns them
        (include/rigidbody.h multibody_rnea_derivatives_batch): 2 n*n entries per state, block b entry r + n*c.
        soa -> [2*n*n, B]; aos -> [B, 2*n*n]; one state -> the pair of [n, n] matrices (D[r, c] = d tau_r / d x_c)."""
        n = self.n
        D = self._call(lib.multibody_rnea_derivatives_batch, (q, dq, ddq), ("q", "dq", "ddq"), (n, n, n), 2 * n * n, layout, out)
        if len(D.shape) == 1:
            return tuple(D[b * n * n:(b + 1) * n * n].reshape(n, n).T for b in range(2))
        return D

    def fd_derivatives(self, q, dq, tau, layout="soa", out=None):
        """Analytical d qdd / d q, d qdd / d dq and H^-1 = d qdd / d tau of qdd = forward_dynamics(q, dq, tau):
        3 n*n entries per state, same packing as `rnea_derivatives`; one state -> three [n, n] matrices."""
        n = self.n
        D = self._call(lib.multibody_fd_derivatives_batch, (q, dq, tau), ("q", "dq", "tau"), (n, n, n), 3 * n * n, layout, out)
        if len(D.shape) == 1:
            return tuple(D[b * n * n:(b + 1) * n * n].reshape(n, n).T for b in range(3))
        return D

    def crba(self, q, layout="soa", out=None):
        """Joint-space mass matrix, reference convention (multibody.rs:155-174; FFI lib.rs:32-43): n*n entries per
        state, entry r + n*c, upper triangle + diagonal filled, strict lower 0.  One state -> [n, n] matrix H[r, c]."""
        n = self.n
        H = self._call(lib.multibody_crba_batch, (q,), ("q",), (n,), n * n, layout, out)
        if len(H.shape) == 1:
            return H.reshape(n, n).T.copy() if not _is_torch(H) else H.reshape(n, n).T.contiguous()
        return H

    def fwd_kin(self, q, layout="soa", out=None):
        """Tip translation (multibody.rs:87-93; FFI lib.rs:46-57)."""
        return self._call(lib.multibody_fwd_kin_batch, (q,), ("q",), (self.n,), 3, layout, out)

    def jac(self, q, layout="soa", out=None):
        """Tip-frame Jacobian, 6n entries per state, entry r + 6*c (multibody.rs:95-108; FFI lib.rs:60-70).
        One state -> [6, n] matrix."""
        n = self.n
        J = self._call(lib.multibody_jac_batch, (q,), ("q",), (n,), 6 * n, layout, out)
        if len(J.shape) == 1:
            return J.reshape(n, 6).T.copy() if not _is_torch(J) else J.reshape(n, 6).T.contiguous()
        return J

    def tip_pose(self, q, offset=None, layout="soa", out=None):
        """Pose of the tip frame (the frame of `jac`) and of a tracked point `offset` (3 values in the tip frame, None = 0)
        in the base frame (include/rigidbody.h multibody_tip_pose_batch): 12 entries per state, x = p + R offset then R
        row-major.  soa -> [12, B]; aos -> [B, 12]; one state -> (x [3], R [3, 3])."""
        args, cuda, single, B, lay = self._prep((q,), ("q",), layout, (self.n,))
        o = self._out(args[0], cuda, single, B, lay, 12, out)
        off = None if offset is None else np.ascontiguousarray(np.broadcast_to(offset, (3,)), dtype=np.float64)
        check(lib.multibody_tip_pose_batch(self._h, C.c_void_p(args[0].ptr), None if off is None else off.ctypes.data_as(C.POINTER(C.c_double)),
                                           C.c_void_p(o.ptr), B, 0, lay, RB_MEM_DEVICE if cuda else RB_MEM_HOST, self._stream(cuda, args[0])))
        P = o.arr
        return (P[:3], P[3:].reshape(3, 3)) if single else P

    def link_poses(self, q, layout="soa", out=None):
        """Pose of every link's frame (the descriptor / URDF joint frame of joint l's child link) in the base frame
        (include/rigidbody.h multibody_link_poses_batch): 12 entries per link per state, P_l then R_l row-major, link-major.
        soa -> [12 n, B]; aos -> [B, 12 n]; one state -> (P [n, 3], R [n, 3, 3])."""
        n = self.n
        P = self._call(lib.multibody_link_poses_batch, (q,), ("q",), (n,), 12 * n, layout, out)
        if len(P.shape) == 1:
            P = P.reshape(n, 12)
            return P[:, :3], P[:, 3:].reshape(n, 3, 3)
        return P

    def sphere_distance(self, q, collision, layout="soa", out=None):
        """Per state min_{k,o} d_ko and the unweighted penalty Phi(q) of a collision model (include/rigidbody.h
        multibody_sphere_distance_batch).  `collision` as for `rollout_cost`.  soa -> [2, B]; aos -> [B, 2]; one state ->
        (min d, Phi)."""
        args, cuda, single, B, lay = self._prep((q,), ("q",), layout, (self.n,))
        o = self._out(args[0], cuda, single, B, lay, 2, out)
        if cuda and args[0].device.index not in (None, self.device):
            raise ValueError(f"tensors are on cuda:{args[0].device.index}, engine is on cuda:{self.device}")
        cc, keep = _collision_cost(collision)
        check(lib.multibody_sphere_distance_batch(self._h, C.c_void_p(args[0].ptr), C.byref(cc), C.c_void_p(o.ptr), B, 0, lay,
                                                  RB_MEM_DEVICE if cuda else RB_MEM_HOST, self._stream(cuda, args[0])))
        D = o.arr
        return (float(D[0]), float(D[1])) if single else D

    def ik(self, p_target, R_target=None, q_init=None, offset=None, w_p=None, w_R=None, limits=True, max_iters=100, tol_p=1e-6,
           tol_R=1e-6, damping=1e-3, layout="soa"):
        """Inverse kinematics of the tip frame, one damped least-squares problem per entry (include/rigidbody.h
        multibody_ik_batch, where the algorithm is stated): finds q with tip point x(q) = p + R offset at `p_target` and,
        when `R_target` is given, orientation R(q) at `R_target`.
        soa: p_target [3, B], R_target [9, B] (row-major entries), q_init [n, B];  aos: [B, 3], [B, 9] or [B, 3, 3], [B, n];
        one problem: p_target [3], R_target [3, 3].  w_R defaults to 1 with R_target and 0 without; w_p (3 values) to 1.
        limits=True takes `limits()` (a joint whose URDF bounds are empty, lower >= upper as for continuous joints, is
        unbounded); None = unbounded; or a (lower, upper) pair of length-n vectors.  q_init=None starts at the midpoint of
        finite bounds, else 0.  Returns (q, info): q shaped like q_init, info rows (pos_err, rot_err, iters) shaped [3, B]
        (soa), [B, 3] (aos) or [3]; iters = -1 marks a problem that did not converge."""
        n = self.n
        w_R = (0.0 if R_target is None else 1.0) if w_R is None else float(w_R)
        if w_R > 0.0 and R_target is None:
            raise ValueError("ik: w_R > 0 needs R_target")
        if limits is True:
            L = self.limits()
            lo, hi = L["lower"].copy(), L["upper"].copy()
            empty = ~(lo < hi)
            lo[empty], hi[empty] = -np.inf, np.inf
        elif limits is None:
            lo, hi = np.full(n, -np.inf), np.full(n, np.inf)
        else:
            lo, hi = (np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (n,))) for v in limits)
        a_p = _Arg(p_target, "p_target")
        single = len(a_p.shape) == 1
        if q_init is None:
            mid = np.where(np.isfinite(lo) & np.isfinite(hi), 0.5 * (lo + hi), 0.0)
            B = 1 if single else (a_p.shape[1] if layout == "soa" else a_p.shape[0])
            q0 = mid if single else (np.repeat(mid[:, None], B, 1) if layout == "soa" else np.repeat(mid[None, :], B, 0))
            if a_p.torch:
                import torch
                q0 = torch.as_tensor(np.ascontiguousarray(q0), device=a_p.device)
            q_init = q0
        arrays, names, per = [q_init, p_target], ["q_init", "p_target"], [n, 3]
        if w_R > 0.0:
            R = R_target
            if single:
                R = R.reshape(9)
            elif layout == "aos" and len(tuple(R.shape)) == 3:
                R = R.reshape(R.shape[0], 9)
            arrays.append(R); names.append("R_target"); per.append(9)
        args, cuda, single, B, lay = self._prep(arrays, names, layout, per)
        if cuda and args[0].device.index not in (None, self.device):
            raise ValueError(f"tensors are on cuda:{args[0].device.index}, engine is on cuda:{self.device}")
        o = self._out(args[0], cuda, single, B, lay, n + 3, None)
        vec = lambda v: None if v is None else np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (3,)))
        off, wp = vec(offset), vec(w_p)
        dp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))
        opt = _lib.RbIkOptions(offset=dp(off), w_p=dp(wp), w_R=w_R, lower=dp(lo), upper=dp(hi), max_iters=int(max_iters),
                               tol_p=float(tol_p), tol_R=float(tol_R), damping=float(damping))
        ptr = [C.c_void_p(a.ptr) for a in args] + [None] * (3 - len(args))
        check(lib.multibody_ik_batch(self._h, *ptr, C.byref(opt), C.c_void_p(o.ptr), B, 0, lay,
                                     RB_MEM_DEVICE if cuda else RB_MEM_HOST, self._stream(cuda, args[0])))
        D = o.arr
        if single or lay == RB_LAYOUT_SOA:
            return D[:n], D[n:]
        return D[:, :n], D[:, n:]

    def rollout(self, q0, dq0, tau, dt, layout="soa", trajectory=True, final=False):
        """Semi-implicit Euler rollout through forward dynamics (SURVEY.md a14).
        soa: q0, dq0 [n, B], tau [H, n, B];  aos: q0, dq0 [B, n], tau [H, B, n].
        Returns (q_traj, dq_traj) shaped like tau, and/or (q_final, dq_final) shaped like q0."""
        a_q, a_dq, a_tau, B, H, lay, new = self._rollout_args(q0, dq0, tau, layout, "rollout")
        cuda = a_q.cuda

        qt = new(a_tau.shape) if trajectory else None
        dqt = new(a_tau.shape) if trajectory else None
        qf = new(a_q.shape) if final else None
        dqf = new(a_q.shape) if final else None
        ptr = lambda a: C.c_void_p(a.ptr) if a is not None else None
        check(lib.multibody_rollout(self._h, ptr(a_q), ptr(a_dq), ptr(a_tau), float(dt), int(H), ptr(qt), ptr(dqt),
                                    ptr(qf), ptr(dqf), B, 0, lay, RB_MEM_DEVICE if cuda else RB_MEM_HOST,
                                    self._stream(cuda, a_q)))
        res = []
        if trajectory:
            res += [qt.arr, dqt.arr]
        if final:
            res += [qf.arr, dqf.arr]
        return tuple(res)

    def rollout_cost(self, q0, dq0, tau, dt, q_ref=None, w_q=None, w_dq=None, w_tau=None, w_q_final=None, w_dq_final=None,
                     layout="soa", final=False, tip=None, collision=None):
        """Fused rollout + quadratic running/terminal cost (one scalar per trajectory; include/rigidbody.h
        multibody_rollout_cost).  Shapes as `rollout`; weights are length-n vectors (None = zeros).  `tip`: a mapping
        with the keys of RbTipCost (offset, p_ref, w_p, w_p_final: 3 values; R_ref: 3x3; w_R, w_R_final: scalars;
        missing = the struct's NULL / 0) adds the tip-pose terms (multibody_rollout_tip_cost).  `collision`: a mapping with
        the keys of RbCollisionCost (link [S], center [S, 3], radius [S], kind [O] of "sphere" / "halfspace", obstacle [O, 4],
        margin, w, w_final) adds the collision-sphere terms (multibody_rollout_collision_cost)."""
        a_q, a_dq, a_tau, B, H, lay, new = self._rollout_args(q0, dq0, tau, layout, "rollout_cost")
        cuda = a_q.cuda
        qc, keep = self._quad_cost(q_ref, w_q, w_dq, w_tau, w_q_final, w_dq_final)
        cost = new((B,))
        qf = new(a_q.shape) if final else None
        dqf = new(a_q.shape) if final else None
        ptr = lambda a: C.c_void_p(a.ptr) if a is not None else None
        head = (self._h, ptr(a_q), ptr(a_dq), ptr(a_tau), float(dt), int(H), C.byref(qc))
        tail = (ptr(cost), ptr(qf), ptr(dqf), B, 0, lay, RB_MEM_DEVICE if cuda else RB_MEM_HOST, self._stream(cuda, a_q))
        if collision is not None:
            tc, keep_tip = _tip_cost(tip or {})
            cc, keep_col = _collision_cost(collision)
            check(lib.multibody_rollout_collision_cost(*head, C.byref(tc), C.byref(cc), *tail))
        elif tip is None:
            check(lib.multibody_rollout_cost(*head, *tail))
        else:
            tc, keep_tip = _tip_cost(tip)
            check(lib.multibody_rollout_tip_cost(*head, C.byref(tc), *tail))
        return (cost.arr, qf.arr, dqf.arr) if final else cost.arr

    def rollout_cost_grad(self, q0, dq0, tau, dt, q_ref=None, w_q=None, w_dq=None, w_tau=None, w_q_final=None, w_dq_final=None,
                          layout="soa", tip=None, collision=None):
        """`rollout_cost` and its gradient (include/rigidbody.h multibody_rollout_cost_grad): returns (cost, grad_tau,
        grad_q0, grad_dq0), the cost bit for bit `rollout_cost`'s, grad_tau shaped like tau, grad_q0 / grad_dq0 like q0.
        `tip` and `collision` as for `rollout_cost` (multibody_rollout_tip_cost_grad,
        multibody_rollout_collision_cost_grad).  Serial chains of at most 12 joints."""
        a_q, a_dq, a_tau, B, H, lay, new = self._rollout_args(q0, dq0, tau, layout, "rollout_cost_grad")
        cuda = a_q.cuda
        qc, keep = self._quad_cost(q_ref, w_q, w_dq, w_tau, w_q_final, w_dq_final)
        cost, gt, gq, gdq = new((B,)), new(a_tau.shape), new(a_q.shape), new(a_q.shape)
        head = (self._h, C.c_void_p(a_q.ptr), C.c_void_p(a_dq.ptr), C.c_void_p(a_tau.ptr), float(dt), int(H), C.byref(qc))
        tail = (C.c_void_p(cost.ptr), C.c_void_p(gt.ptr), C.c_void_p(gq.ptr), C.c_void_p(gdq.ptr),
                B, 0, lay, RB_MEM_DEVICE if cuda else RB_MEM_HOST, self._stream(cuda, a_q))
        if collision is not None:
            tc, keep_tip = _tip_cost(tip or {})
            cc, keep_col = _collision_cost(collision)
            check(lib.multibody_rollout_collision_cost_grad(*head, C.byref(tc), C.byref(cc), *tail))
        elif tip is None:
            check(lib.multibody_rollout_cost_grad(*head, *tail))
        else:
            tc, keep_tip = _tip_cost(tip)
            check(lib.multibody_rollout_tip_cost_grad(*head, C.byref(tc), *tail))
        return cost.arr, gt.arr, gq.arr, gdq.arr

    def rollout_cost_autograd(self, q0, dq0, tau, dt, tip=None, collision=None, **weights):
        """`rollout_cost` as a differentiable torch function: q0, dq0 [n, B] and tau [H, n, B] are CUDA float64 tensors
        (layout 'soa'); returns cost [B].  The forward pass runs `rollout_cost_grad` (`rollout_cost` when no input requires
        a gradient); the backward pass scales the stored gradients by the upstream gradient of each trajectory's cost.
        `tip`, `collision` and the weights as for `rollout_cost`."""
        return _rollout_cost_function().apply(self, q0, dq0, tau, float(dt), tip, collision, weights)

    def mppi_step(self, q0, dq0, u_nom, dt, sigma, n_samples, temperature, seed, limits=True, layout="soa", tip=None, collision=None,
                  samples=False, **weights):
        """One MPPI iteration for each of P problems (include/rigidbody.h multibody_mppi_step, where the sampler, the weights
        and the update are stated): K = n_samples torque sequences around each nominal sequence, drawn on the device from
        `seed` (sample 0 is the nominal one) and clamped to the bounds, costed with the fused rollout cost, and averaged with
        softmin weights of temperature lambda.  The cost terms are `rollout_cost`'s: the weights (q_ref, w_q, ...), `tip`
        and `collision`.  soa: q0, dq0 [n, P], u_nom [H, n, P];  aos: [P, n], [P, n], [H, P, n].  sigma: n values or one.
        limits=True bounds the samples by +-limits()["effort"] (a joint with effort <= 0 is unbounded); None = unbounded; or
        a (lower, upper) pair.  Returns (u_new shaped like u_nom, cost [P, K], sample_weights [P, K]), and with samples=True
        also the samples [H, n, P K] (soa) or [H, P K, n] (aos), sample k of problem p at p K + k."""
        a_q, a_dq, a_u, P, H, lay, new = self._rollout_args(q0, dq0, u_nom, layout, "mppi_step")
        cuda = a_q.cuda
        if cuda and a_q.device.index not in (None, self.device):
            raise ValueError(f"tensors are on cuda:{a_q.device.index}, engine is on cuda:{self.device}")
        n, K = self.n, int(n_samples)
        vec = lambda v: np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (n,)))
        if limits is True:
            eff = self.limits()["effort"]
            lo, hi = np.where(eff > 0, -eff, -np.inf), np.where(eff > 0, eff, np.inf)
        elif limits is None:
            lo, hi = np.full(n, -np.inf), np.full(n, np.inf)
        else:
            lo, hi = (vec(v) for v in limits)
        sg = vec(sigma)
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        opt = _lib.RbMppiOptions(sigma=dp(sg), lower=dp(lo), upper=dp(hi), temperature=float(temperature), n_samples=K,
                                 seed=int(seed) & 0xFFFFFFFFFFFFFFFF)
        qc, keep = self._quad_cost(**weights)
        tc, keep_tip = _tip_cost(tip or {}) if tip is not None or collision is not None else (None, None)
        cc, keep_col = _collision_cost(collision) if collision is not None else (None, None)
        Kp = max(K, 0)
        u_new, cost, sw = new(a_u.shape), new((P, Kp)), new((P, Kp))
        smp = new((H, n, P * Kp) if lay == RB_LAYOUT_SOA else (H, P * Kp, n)) if samples else None
        ptr = lambda a: C.c_void_p(a.ptr) if a is not None else None
        ref = lambda s: C.byref(s) if s is not None else None
        check(lib.multibody_mppi_step(self._h, ptr(a_q), ptr(a_dq), ptr(a_u), float(dt), int(H), C.byref(qc), ref(tc), ref(cc), C.byref(opt),
                                      ptr(u_new), ptr(cost), ptr(sw), ptr(smp), P, 0, lay, RB_MEM_DEVICE if cuda else RB_MEM_HOST,
                                      self._stream(cuda, a_q)))
        res = (u_new.arr, cost.arr, sw.arr)
        return res + (smp.arr,) if samples else res

    def rollout_vjp(self, q0, dq0, tau, dt, q_traj, dq_traj, g_q_traj=None, g_dq_traj=None, g_q_final=None, g_dq_final=None,
                    layout="soa"):
        """Vector-Jacobian product of `rollout` (include/rigidbody.h multibody_rollout_vjp): given the trajectory `rollout`
        returned for these inputs and upstream gradients of (q_traj, dq_traj, q_final, dq_final) (None = zero), returns
        (grad_tau, grad_q0, grad_dq0).  Serial chains of at most 12 joints."""
        a_q, a_dq, a_tau, B, H, lay, new = self._rollout_args(q0, dq0, tau, layout, "rollout_vjp")
        cuda = a_q.cuda

        def arg(x, name, shape):
            if x is None:
                return None
            a = _Arg(x, name)
            if a.shape != shape or a.cuda != cuda:
                raise ValueError(f"rollout_vjp: {name} must have shape {shape} and live with q0")
            return a
        ins = [arg(q_traj, "q_traj", a_tau.shape), arg(dq_traj, "dq_traj", a_tau.shape), arg(g_q_traj, "g_q_traj", a_tau.shape),
               arg(g_dq_traj, "g_dq_traj", a_tau.shape), arg(g_q_final, "g_q_final", a_q.shape), arg(g_dq_final, "g_dq_final", a_q.shape)]
        gt, gq, gdq = new(a_tau.shape), new(a_q.shape), new(a_q.shape)
        ptr = lambda a: C.c_void_p(a.ptr) if a is not None else None
        check(lib.multibody_rollout_vjp(self._h, ptr(a_q), ptr(a_dq), ptr(a_tau), float(dt), int(H), *[ptr(a) for a in ins],
                                        ptr(gt), ptr(gq), ptr(gdq), B, 0, lay, RB_MEM_DEVICE if cuda else RB_MEM_HOST,
                                        self._stream(cuda, a_q)))
        return gt.arr, gq.arr, gdq.arr

    def rollout_autograd(self, q0, dq0, tau, dt):
        """`rollout` as a differentiable torch function: q0, dq0 [n, B] and tau [H, n, B] are CUDA float64 tensors (layout
        'soa'); returns (q_traj, dq_traj) [H, n, B], whose backward pass is `rollout_vjp` on the current stream."""
        return _rollout_function().apply(self, q0, dq0, tau, float(dt))

    # ---- argument plumbing of the rollout entries
    def _rollout_args(self, q0, dq0, tau, layout, what):
        """Checks (q0, dq0, tau) against `layout`; returns their _Args, B, H, the layout code and an allocator of outputs
        that live with them."""
        a_q, a_dq, a_tau = _Arg(q0, "q0"), _Arg(dq0, "dq0"), _Arg(tau, "tau")
        cuda = a_q.cuda
        if a_dq.cuda != cuda or a_tau.cuda != cuda:
            raise ValueError("all arrays of one call must live in the same place")
        n = self.n
        if layout == "soa":
            B = a_q.shape[1]; H = a_tau.shape[0]
            ok = a_q.shape == (n, B) and a_dq.shape == (n, B) and a_tau.shape == (H, n, B)
            lay = RB_LAYOUT_SOA
        elif layout == "aos":
            B = a_q.shape[0]; H = a_tau.shape[0]
            ok = a_q.shape == (B, n) and a_dq.shape == (B, n) and a_tau.shape == (H, B, n)
            lay = RB_LAYOUT_AOS
        else:
            raise ValueError("layout must be 'soa' or 'aos'")
        if not ok:
            raise ValueError(f"{what}: inconsistent shapes")

        def new(shape):
            if cuda:
                import torch
                return _Arg(torch.empty(shape, dtype=torch.float64, device=a_q.device), "out")
            return _Arg(np.empty(shape, dtype=np.float64), "out")
        return a_q, a_dq, a_tau, B, H, lay, new

    def _quad_cost(self, q_ref=None, w_q=None, w_dq=None, w_tau=None, w_q_final=None, w_dq_final=None):
        """An RbQuadCost over length-n weight vectors (None = zeros) and the arrays it points into (keep them alive)."""
        qc = _lib.RbQuadCost()
        keep = []
        for name, v in (("q_ref", q_ref), ("w_q", w_q), ("w_dq", w_dq), ("w_tau", w_tau), ("w_q_final", w_q_final), ("w_dq_final", w_dq_final)):
            if v is not None:
                a = np.ascontiguousarray(np.broadcast_to(v, (self.n,)), dtype=np.float64); keep.append(a)
                setattr(qc, name, a.ctypes.data_as(C.POINTER(C.c_double)))
        return qc, keep

    # ---- device-side sampler (bench / tests)
    def fill(self, out, seed, field, lo, hi, first_index=0):
        """Fill a CUDA float64 tensor [n, B] with the counter-based sampler of SURVEY.md 8d."""
        o = _Arg(out, "out")
        if not o.cuda or len(o.shape) != 2 or o.shape[0] != self.n:
            raise ValueError("fill: out must be a CUDA float64 tensor shaped [n, B]")
        lo = np.ascontiguousarray(np.broadcast_to(lo, (self.n,)), dtype=np.float64)
        hi = np.ascontiguousarray(np.broadcast_to(hi, (self.n,)), dtype=np.float64)
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        check(lib.multibody_gpu_fill(self._h, C.c_void_p(o.ptr), int(seed), int(field), dp(lo), dp(hi),
                                     int(first_index), o.shape[1], o.shape[1], self._stream(True, o)))
        return out


_TIP_KEYS = {"offset": 3, "p_ref": 3, "w_p": 3, "w_p_final": 3, "R_ref": 9}


def _tip_cost(tip):
    """An RbTipCost from a mapping with its keys (missing = NULL / 0) and the arrays it points into (keep them alive)."""
    unknown = set(tip) - set(_TIP_KEYS) - {"w_R", "w_R_final"}
    if unknown:
        raise ValueError(f"tip: unknown keys {sorted(unknown)}")
    tc = _lib.RbTipCost()
    keep = []
    for name, size in _TIP_KEYS.items():
        if tip.get(name) is not None:
            a = np.ascontiguousarray(np.asarray(tip[name], dtype=np.float64).reshape(-1))
            if a.size != size:
                raise ValueError(f"tip: {name} must have {size} values")
            keep.append(a)
            setattr(tc, name, a.ctypes.data_as(C.POINTER(C.c_double)))
    tc.w_R = float(tip.get("w_R", 0.0))
    tc.w_R_final = float(tip.get("w_R_final", 0.0))
    return tc, keep


_COLLISION_KINDS = {"sphere": _lib.RB_OBSTACLE_SPHERE, "halfspace": _lib.RB_OBSTACLE_HALFSPACE}


def _collision_cost(col):
    """An RbCollisionCost from a mapping with its keys (link, center [S, 3], radius, kind of "sphere" / "halfspace",
    obstacle [O, 4], margin, w, w_final; missing = empty / 0) and the arrays it points into (keep them alive).  The values
    themselves are checked by the library."""
    unknown = set(col) - {"link", "center", "radius", "kind", "obstacle", "margin", "w", "w_final"}
    if unknown:
        raise ValueError(f"collision: unknown keys {sorted(unknown)}")
    link = np.ascontiguousarray(np.asarray(col.get("link", ()), dtype=np.int32).reshape(-1))
    S = link.size
    center = np.ascontiguousarray(np.asarray(col.get("center", np.zeros((S, 3))), dtype=np.float64).reshape(-1))
    radius = np.ascontiguousarray(np.asarray(col.get("radius", np.zeros(S)), dtype=np.float64).reshape(-1))
    if center.size != 3 * S or radius.size != S:
        raise ValueError("collision: center must be [S, 3] and radius [S] for the S entries of link")
    kinds = [k if isinstance(k, (int, np.integer)) else _COLLISION_KINDS.get(k, -1) for k in col.get("kind", ())]
    kind = np.ascontiguousarray(np.asarray(kinds, dtype=np.int32).reshape(-1))
    O = kind.size
    obstacle = np.ascontiguousarray(np.asarray(col.get("obstacle", np.zeros((O, 4))), dtype=np.float64).reshape(-1))
    if obstacle.size != 4 * O:
        raise ValueError("collision: obstacle must be [O, 4] for the O entries of kind")
    cc = _lib.RbCollisionCost()
    cc.n_spheres, cc.n_obstacles = S, O
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    cc.link, cc.center, cc.radius, cc.kind, cc.obstacle = ip(link), dp(center), dp(radius), ip(kind), dp(obstacle)
    cc.margin = float(col.get("margin", 0.0))
    cc.w = float(col.get("w", 0.0))
    cc.w_final = float(col.get("w_final", 0.0))
    return cc, [link, center, radius, kind, obstacle]


_ROLLOUT_FN = None
_ROLLOUT_COST_FN = None


def _rollout_function():
    """The torch.autograd.Function behind Multibody.rollout_autograd (built on first use: torch stays a lazy import)."""
    global _ROLLOUT_FN
    if _ROLLOUT_FN is None:
        import torch

        class RolloutFunction(torch.autograd.Function):
            @staticmethod
            def forward(ctx, mb, q0, dq0, tau, dt):
                for name, t in (("q0", q0), ("dq0", dq0), ("tau", tau)):
                    if not (_is_torch(t) and t.is_cuda and t.dtype == torch.float64):
                        raise TypeError(f"rollout_autograd: {name} must be a CUDA float64 tensor")
                q0, dq0, tau = q0.contiguous(), dq0.contiguous(), tau.contiguous()
                qt, dqt = mb.rollout(q0, dq0, tau, dt)
                ctx.mb, ctx.dt = mb, dt
                ctx.save_for_backward(q0, dq0, tau, qt, dqt)
                return qt, dqt

            @staticmethod
            def backward(ctx, g_qt, g_dqt):
                q0, dq0, tau, qt, dqt = ctx.saved_tensors
                c = lambda g: None if g is None else g.contiguous()
                gt, gq, gdq = ctx.mb.rollout_vjp(q0, dq0, tau, ctx.dt, qt, dqt, c(g_qt), c(g_dqt))
                return None, gq, gdq, gt, None

        _ROLLOUT_FN = RolloutFunction
    return _ROLLOUT_FN


def _rollout_cost_function():
    """The torch.autograd.Function behind Multibody.rollout_cost_autograd (built on first use: torch stays a lazy import)."""
    global _ROLLOUT_COST_FN
    if _ROLLOUT_COST_FN is None:
        import torch

        class RolloutCostFunction(torch.autograd.Function):
            @staticmethod
            def forward(ctx, mb, q0, dq0, tau, dt, tip, collision, weights):
                for name, t in (("q0", q0), ("dq0", dq0), ("tau", tau)):
                    if not (_is_torch(t) and t.is_cuda and t.dtype == torch.float64):
                        raise TypeError(f"rollout_cost_autograd: {name} must be a CUDA float64 tensor")
                q0, dq0, tau = q0.contiguous(), dq0.contiguous(), tau.contiguous()
                if any(ctx.needs_input_grad[1:4]):
                    cost, gt, gq, gdq = mb.rollout_cost_grad(q0, dq0, tau, dt, tip=tip, collision=collision, **weights)
                    ctx.save_for_backward(gq, gdq, gt)
                else:
                    cost = mb.rollout_cost(q0, dq0, tau, dt, tip=tip, collision=collision, **weights)
                return cost

            @staticmethod
            def backward(ctx, g_cost):
                gq, gdq, gt = ctx.saved_tensors
                g = g_cost.contiguous()
                return None, gq * g[None, :], gdq * g[None, :], gt * g[None, None, :], None, None, None, None

        _ROLLOUT_COST_FN = RolloutCostFunction
    return _ROLLOUT_COST_FN
