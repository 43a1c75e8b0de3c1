"""Loads librigidbody_b200.so (the C ABI of include/rigidbody.h) and declares its prototypes.

There is no Python or CPU implementation of the dynamics behind this module: if the library is missing
or cannot be loaded, importing fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# RIGIDBODY_B200_LIB lets tools/kbench.py time alternative builds of the same library (tuning experiments).
LIB_PATH = os.environ.get("RIGIDBODY_B200_LIB") or os.path.join(_HERE, "librigidbody_b200.so")

RB_OK = 0
RB_ERR_NULL, RB_ERR_ARG, RB_ERR_URDF, RB_ERR_CUDA, RB_ERR_NOT_SPD, RB_ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6
RB_LAYOUT_SOA, RB_LAYOUT_AOS = 0, 1
RB_MEM_HOST, RB_MEM_DEVICE = 0, 1
RB_MAX_JOINTS = 64

_dp = C.POINTER(C.c_double)


class RbChainDesc(C.Structure):
    _fields_ = [("n_joints", C.c_int32), ("parent", C.POINTER(C.c_int32)), ("axis", _dp), ("parent_rot", _dp),
                ("parent_trans", _dp), ("mass", _dp), ("com", _dp), ("inertia_com", _dp), ("gravity", C.c_double * 3)]


class RbQuadCost(C.Structure):
    _fields_ = [(k, _dp) for k in ("q_ref", "w_q", "w_dq", "w_tau", "w_q_final", "w_dq_final")]


class RbTipCost(C.Structure):
    _fields_ = [(k, _dp) for k in ("offset", "p_ref", "w_p", "w_p_final", "R_ref")] + [("w_R", C.c_double), ("w_R_final", C.c_double)]


class RbIkOptions(C.Structure):
    _fields_ = [("offset", _dp), ("w_p", _dp), ("w_R", C.c_double), ("lower", _dp), ("upper", _dp), ("max_iters", C.c_int),
                ("tol_p", C.c_double), ("tol_R", C.c_double), ("damping", C.c_double)]


class RbJointLimits(C.Structure):
    _fields_ = [(k, C.c_double * RB_MAX_JOINTS) for k in ("lower", "upper", "velocity", "effort")]


# every symbol include/rigidbody.h declares: name -> (restype, argtypes)
_vp, _sz, _i, _u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64
PROTOTYPES = {
    "multibody_new": (_vp, []),
    "multibody_new_from_urdf": (_vp, [C.c_char_p]),
    "multibody_fwd_kin": (_dp, [_vp, _dp]),
    "multibody_jac": (_dp, [_vp, _dp]),
    "multibody_rnea": (_dp, [_vp, _dp, _dp, _dp]),
    "multibody_crba": (_dp, [_vp, _dp]),
    "multibody_free": (None, [_vp]),
    "multibody_free_result": (None, [_dp]),
    "multibody_n_joints": (_i, [_vp]),
    "multibody_get_model": (_i, [_vp, _dp, _dp, _dp, _dp, _dp]),
    "multibody_get_chain": (_i, [_vp, C.POINTER(C.c_int32), _dp, _dp, _dp, _dp, _dp, _dp]),
    "multibody_gpu_new": (_i, [C.POINTER(RbChainDesc), _i, C.POINTER(_vp)]),
    "multibody_gpu_new_from_urdf": (_i, [C.c_char_p, _i, C.POINTER(_vp)]),
    "multibody_gpu_from_multibody": (_i, [_vp, _i, C.POINTER(_vp)]),
    "multibody_gpu_free": (None, [_vp]),
    "multibody_gpu_n_joints": (_i, [_vp]),
    "multibody_gpu_device": (_i, [_vp]),
    "multibody_gpu_kernel_variant": (C.c_char_p, [_vp]),
    "multibody_gpu_family_note": (C.c_char_p, [_vp]),
    "multibody_jit_precompile": (_i, [C.POINTER(RbChainDesc), C.c_char_p, C.c_char_p, _sz]),
    "multibody_gpu_get_model": (_i, [_vp, _dp, _dp, _dp, _dp, _dp]),
    "multibody_gpu_get_limits": (_i, [_vp, C.POINTER(RbJointLimits)]),
    "multibody_last_error": (C.c_char_p, []),
    "multibody_rnea_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_forward_dynamics_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rnea_batch_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _sz, _vp]),
    "multibody_forward_dynamics_batch_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _sz, _vp]),
    "multibody_rnea_fd_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rnea_derivatives_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_fd_derivatives_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_crba_batch": (_i, [_vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_fwd_kin_batch": (_i, [_vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_jac_batch": (_i, [_vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rollout": (_i, [_vp, _vp, _vp, _vp, C.c_double, _i, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rollout_cost": (_i, [_vp, _vp, _vp, _vp, C.c_double, _i, C.POINTER(RbQuadCost), _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rollout_vjp": (_i, [_vp, _vp, _vp, _vp, C.c_double, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rollout_cost_grad": (_i, [_vp, _vp, _vp, _vp, C.c_double, _i, C.POINTER(RbQuadCost), _vp, _vp, _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_rollout_tip_cost": (_i, [_vp, _vp, _vp, _vp, C.c_double, _i, C.POINTER(RbQuadCost), C.POINTER(RbTipCost), _vp, _vp, _vp,
                                        _sz, _sz, _i, _i, _vp]),
    "multibody_rollout_tip_cost_grad": (_i, [_vp, _vp, _vp, _vp, C.c_double, _i, C.POINTER(RbQuadCost), C.POINTER(RbTipCost), _vp, _vp,
                                             _vp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_tip_pose_batch": (_i, [_vp, _vp, _dp, _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_ik_batch": (_i, [_vp, _vp, _vp, _vp, C.POINTER(RbIkOptions), _vp, _sz, _sz, _i, _i, _vp]),
    "multibody_gpu_fill": (_i, [_vp, _vp, _u64, C.c_uint32, _dp, _dp, _sz, _sz, _sz, _vp]),
    "multibody_gpu_sync": (_i, [_vp]),
    "multibody_gpu_status": (_i, [_vp]),
    "multibody_gpu_launch_count": (_u64, [_vp]),
    "multibody_host_alloc": (_i, [C.POINTER(_vp), _sz]),
    "multibody_host_free": (None, [_vp]),
    "multibody_gpu_measure_fp64_peak": (_i, [_vp, _i, _dp]),
    "multibody_gpu_new_multi": (_i, [C.POINTER(RbChainDesc), C.POINTER(C.c_int), _i, C.POINTER(_vp)]),
    "multibody_gpu_new_multi_from_urdf": (_i, [C.c_char_p, C.POINTER(C.c_int), _i, C.POINTER(_vp)]),
    "multibody_gpu_n_devices": (_i, [_vp]),
    "multibody_gpu_peer": (_vp, [_vp, _i]),
    "multibody_gpu_measure_copy_peak": (_i, [_vp, _sz, _sz, _i, _dp, _dp]),
}


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
            f"`make -C rigidbody_rs_b200/csrc`.  rigidbody_rs_b200 has no CPU or pure-Python fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)      # AttributeError here = the library does not match the header
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()


class RigidBodyError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{code}] {msg}")
        self.code = code


class NotPositiveDefinite(RigidBodyError):
    pass


def check(rc):
    if rc == RB_OK:
        return
    msg = (lib.multibody_last_error() or b"").decode()
    raise (NotPositiveDefinite if rc == RB_ERR_NOT_SPD else RigidBodyError)(rc, msg)
