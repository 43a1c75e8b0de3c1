//! Rust host side of the B200 batched engine: flattens a `rigidbody::multibody::Multibody` into the
//! `RbChainDesc` of include/rigidbody.h, uploads it once, and exposes safe batched calls.
//!
//! Written against the reference at khaninger/rigidbody-rs:
//!   * `Multibody::iter()`                      rigidbody/src/multibody.rs:79-81
//!   * `RevoluteJoint { axis, parent, body }`   rigidbody/src/joint.rs:26-31   (all `pub`)
//!   * `Inertia { mass, com, inertia_com, .. }` rigidbody/src/inertia.rs:12-17 (`inertia` about the origin is
//!     private, so the C side recomputes it from mass/com/inertia_com exactly as `from_com` does, :31-32)
//!
//! NOT COMPILED in the build container of the CUDA repository (no cargo/rustc there); what stands in for the compiler
//! there: a test that compares the `extern "C"` block below with include/rigidbody.h symbol by symbol, and
//! examples/rust_crate_double.c, a C program that performs this crate's call sequence statement for statement and is
//! run by the GPU test-suite.  Requires
//! `pub use inertia::Inertia;` (or `pub mod inertia`) in rigidbody/src/lib.rs so the field types are nameable;
//! the fields themselves are already public.
use std::ffi::{c_char, c_int, c_void, CStr};
use std::ptr;

use rigidbody::multibody::Multibody;

// ------------------------------------------------------------------ raw C ABI (include/rigidbody.h, Part 2)
#[repr(C)]
pub struct RbChainDesc {
    pub n_joints: i32,
    pub parent: *const i32,
    pub axis: *const f64,
    pub parent_rot: *const f64,
    pub parent_trans: *const f64,
    pub mass: *const f64,
    pub com: *const f64,
    pub inertia_com: *const f64,
    pub gravity: [f64; 3],
}

#[repr(C)]
pub struct RbGpu {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy, PartialEq, Eq)]
pub enum RbLayout {
    Soa = 0,
    Aos = 1,
}

#[repr(C)]
#[derive(Clone, Copy, PartialEq, Eq)]
pub enum RbMem {
    Host = 0,
    Device = 1,
}

/// Per-joint limits read from the URDF (include/rigidbody.h RbJointLimits; RB_MAX_JOINTS = 64).
#[repr(C)]
pub struct RbJointLimits {
    pub lower: [f64; 64],
    pub upper: [f64; 64],
    pub velocity: [f64; 64],
    pub effort: [f64; 64],
}

// Every Part-2 symbol of include/rigidbody.h (tests/test_host.py::test_rust_crate_binds_the_whole_header compares this
// block with the header, name by name and argument count by argument count, since the crate cannot be compiled where
// the CUDA library is built).
extern "C" {
    // ---- construction / teardown
    pub fn multibody_gpu_new(desc: *const RbChainDesc, device: c_int, out: *mut *mut RbGpu) -> c_int;
    pub fn multibody_gpu_new_from_urdf(urdf_path: *const c_char, device: c_int, out: *mut *mut RbGpu) -> c_int;
    pub fn multibody_gpu_from_multibody(mb: *const c_void, device: c_int, out: *mut *mut RbGpu) -> c_int;
    pub fn multibody_gpu_new_multi(desc: *const RbChainDesc, devices: *const c_int, n_dev: c_int, out: *mut *mut RbGpu) -> c_int;
    pub fn multibody_gpu_new_multi_from_urdf(urdf_path: *const c_char, devices: *const c_int, n_dev: c_int, out: *mut *mut RbGpu) -> c_int;
    pub fn multibody_gpu_n_devices(g: *const RbGpu) -> c_int;
    pub fn multibody_gpu_peer(g: *mut RbGpu, index: c_int) -> *mut RbGpu;
    pub fn multibody_gpu_free(g: *mut RbGpu);
    // ---- introspection
    pub fn multibody_gpu_n_joints(g: *const RbGpu) -> c_int;
    pub fn multibody_gpu_device(g: *const RbGpu) -> c_int;
    pub fn multibody_gpu_kernel_variant(g: *const RbGpu) -> *const c_char;
    pub fn multibody_gpu_family_note(g: *const RbGpu) -> *const c_char;
    pub fn multibody_jit_precompile(desc: *const RbChainDesc, urdf_path: *const c_char, log: *mut c_char, log_len: usize) -> c_int;
    pub fn multibody_gpu_get_model(g: *const RbGpu, parent_rot: *mut f64, parent_trans: *mut f64, mass: *mut f64, h: *mut f64,
                                   inertia_origin: *mut f64) -> c_int;
    pub fn multibody_gpu_get_limits(g: *const RbGpu, out: *mut RbJointLimits) -> c_int;
    pub fn multibody_last_error() -> *const c_char;
    // ---- the batched hot path
    pub fn multibody_rnea_batch(g: *mut RbGpu, q: *const f64, dq: *const f64, ddq: *const f64, tau: *mut f64,
                                n_states: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_forward_dynamics_batch(g: *mut RbGpu, q: *const f64, dq: *const f64, tau: *const f64, qdd: *mut f64,
                                            n_states: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rnea_batch_f32(g: *mut RbGpu, q: *const f32, dq: *const f32, ddq: *const f32, tau: *mut f32,
                                    n_states: usize, ld: usize, stream: *mut c_void) -> c_int;
    pub fn multibody_forward_dynamics_batch_f32(g: *mut RbGpu, q: *const f32, dq: *const f32, tau: *const f32, qdd: *mut f32,
                                                n_states: usize, ld: usize, stream: *mut c_void) -> c_int;
    pub fn multibody_rnea_fd_batch(g: *mut RbGpu, q: *const f64, dq: *const f64, ddq: *const f64, tau_in: *const f64, out: *mut f64,
                                   n_states: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_crba_batch(g: *mut RbGpu, q: *const f64, h: *mut f64, n_states: usize, ld: usize, layout: RbLayout,
                                mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rnea_derivatives_batch(g: *mut RbGpu, q: *const f64, dq: *const f64, ddq: *const f64, out: *mut f64,
                                            n_states: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_fd_derivatives_batch(g: *mut RbGpu, q: *const f64, dq: *const f64, tau: *const f64, out: *mut f64,
                                          n_states: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_fwd_kin_batch(g: *mut RbGpu, q: *const f64, xyz: *mut f64, n_states: usize, ld: usize, layout: RbLayout,
                                   mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_jac_batch(g: *mut RbGpu, q: *const f64, j: *mut f64, n_states: usize, ld: usize, layout: RbLayout,
                               mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rollout(g: *mut RbGpu, q0: *const f64, dq0: *const f64, tau: *const f64, dt: f64, horizon: c_int,
                             q_traj: *mut f64, dq_traj: *mut f64, q_final: *mut f64, dq_final: *mut f64,
                             n_traj: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rollout_cost(g: *mut RbGpu, q0: *const f64, dq0: *const f64, tau: *const f64, dt: f64, horizon: c_int,
                                  w: *const RbQuadCost, cost: *mut f64, q_final: *mut f64, dq_final: *mut f64,
                                  n_traj: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rollout_vjp(g: *mut RbGpu, q0: *const f64, dq0: *const f64, tau: *const f64, dt: f64, horizon: c_int,
                                 q_traj: *const f64, dq_traj: *const f64,
                                 g_q_traj: *const f64, g_dq_traj: *const f64, g_q_final: *const f64, g_dq_final: *const f64,
                                 grad_tau: *mut f64, grad_q0: *mut f64, grad_dq0: *mut f64,
                                 n_traj: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rollout_cost_grad(g: *mut RbGpu, q0: *const f64, dq0: *const f64, tau: *const f64, dt: f64, horizon: c_int,
                                       w: *const RbQuadCost, cost: *mut f64, grad_tau: *mut f64, grad_q0: *mut f64, grad_dq0: *mut f64,
                                       n_traj: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rollout_tip_cost(g: *mut RbGpu, q0: *const f64, dq0: *const f64, tau: *const f64, dt: f64, horizon: c_int,
                                      w: *const RbQuadCost, tip: *const RbTipCost, cost: *mut f64, q_final: *mut f64, dq_final: *mut f64,
                                      n_traj: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_rollout_tip_cost_grad(g: *mut RbGpu, q0: *const f64, dq0: *const f64, tau: *const f64, dt: f64, horizon: c_int,
                                           w: *const RbQuadCost, tip: *const RbTipCost, cost: *mut f64, grad_tau: *mut f64,
                                           grad_q0: *mut f64, grad_dq0: *mut f64, n_traj: usize, ld: usize, layout: RbLayout, mem: RbMem,
                                           stream: *mut c_void) -> c_int;
    pub fn multibody_tip_pose_batch(g: *mut RbGpu, q: *const f64, offset: *const f64, pose: *mut f64,
                                    n_states: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    pub fn multibody_ik_batch(g: *mut RbGpu, q_init: *const f64, p_target: *const f64, r_target: *const f64, opt: *const RbIkOptions,
                              out: *mut f64, n_problems: usize, ld: usize, layout: RbLayout, mem: RbMem, stream: *mut c_void) -> c_int;
    // ---- device-side helpers
    pub fn multibody_gpu_fill(g: *mut RbGpu, dev_out: *mut f64, seed: u64, field: u32, lo: *const f64, hi: *const f64,
                              first_index: usize, count: usize, ld: usize, stream: *mut c_void) -> c_int;
    pub fn multibody_gpu_sync(g: *mut RbGpu) -> c_int;
    pub fn multibody_gpu_status(g: *mut RbGpu) -> c_int;
    pub fn multibody_gpu_launch_count(g: *const RbGpu) -> u64;
    pub fn multibody_host_alloc(out: *mut *mut c_void, bytes: usize) -> c_int;
    pub fn multibody_host_free(p: *mut c_void);
    pub fn multibody_gpu_measure_copy_peak(g: *mut RbGpu, h2d_bytes: usize, d2h_bytes: usize, reps: c_int, h2d_gbs: *mut f64,
                                           d2h_gbs: *mut f64) -> c_int;
    pub fn multibody_gpu_measure_fp64_peak(g: *mut RbGpu, millis: c_int, tflops: *mut f64) -> c_int;
}

/// Quadratic running / terminal cost of `multibody_rollout_cost` (include/rigidbody.h RbQuadCost): six host arrays of
/// n per-joint values each; a null pointer means zeros.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RbQuadCost {
    pub q_ref: *const f64,
    pub w_q: *const f64,
    pub w_dq: *const f64,
    pub w_tau: *const f64,
    pub w_q_final: *const f64,
    pub w_dq_final: *const f64,
}

/// Tip-pose tracking terms of `multibody_rollout_tip_cost` (include/rigidbody.h RbTipCost): host arrays of 3 values
/// (`r_ref`: 9, row-major) and two scalar weights; a null pointer means the header's default (zeros, identity `r_ref`).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RbTipCost {
    pub offset: *const f64,
    pub p_ref: *const f64,
    pub w_p: *const f64,
    pub w_p_final: *const f64,
    pub r_ref: *const f64,
    pub w_r: f64,
    pub w_r_final: f64,
}

/// Options of `multibody_ik_batch` (include/rigidbody.h RbIkOptions, where the algorithm is stated): host arrays of 3
/// (`offset`, `w_p`) or n (`lower`, `upper`) values, a null pointer meaning the header's default (tip origin, unit weights,
/// unbounded joints).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RbIkOptions {
    pub offset: *const f64,
    pub w_p: *const f64,
    pub w_r: f64,
    pub lower: *const f64,
    pub upper: *const f64,
    pub max_iters: c_int,
    pub tol_p: f64,
    pub tol_r: f64,
    pub damping: f64,
}

#[derive(Debug)]
pub struct RbError {
    pub code: i32,
    pub message: String,
}

fn check(rc: c_int) -> Result<(), RbError> {
    if rc == 0 {
        return Ok(());
    }
    let message = unsafe { CStr::from_ptr(multibody_last_error()) }.to_string_lossy().into_owned();
    Err(RbError { code: rc, message })
}

// ------------------------------------------------------------------ Multibody -> flattened descriptor
/// Owned arrays behind an `RbChainDesc`; joint i's parent is joint i-1 (the reference is a serial chain; the C side
/// also accepts a `parent` index array for kinematic trees, which `Multibody` cannot express).  Axes other than +z
/// are honoured by the engine (the reference's rnea / crba ignore them, multibody.rs:29,130).
pub struct ChainArrays {
    pub axis: Vec<f64>,
    pub parent_rot: Vec<f64>,
    pub parent_trans: Vec<f64>,
    pub mass: Vec<f64>,
    pub com: Vec<f64>,
    pub inertia_com: Vec<f64>,
}

impl ChainArrays {
    pub fn from_multibody(mb: &Multibody) -> Self {
        let mut a = ChainArrays { axis: vec![], parent_rot: vec![], parent_trans: vec![], mass: vec![], com: vec![], inertia_com: vec![] };
        for jt in mb.iter() {
            a.axis.extend_from_slice(&[jt.axis[0], jt.axis[1], jt.axis[2]]);
            let r = jt.parent.rotation.to_rotation_matrix();
            for row in 0..3 {
                for col in 0..3 {
                    a.parent_rot.push(r[(row, col)]); // row-major
                }
            }
            let t = jt.parent.translation.vector;
            a.parent_trans.extend_from_slice(&[t[0], t[1], t[2]]);
            a.mass.push(jt.body.mass);
            a.com.extend_from_slice(&[jt.body.com[0], jt.body.com[1], jt.body.com[2]]);
            for row in 0..3 {
                for col in 0..3 {
                    a.inertia_com.push(jt.body.inertia_com[(row, col)]);
                }
            }
        }
        a
    }

    pub fn desc(&self) -> RbChainDesc {
        RbChainDesc {
            n_joints: self.mass.len() as i32,
            parent: ptr::null(), // serial chain
            axis: self.axis.as_ptr(),
            parent_rot: self.parent_rot.as_ptr(),
            parent_trans: self.parent_trans.as_ptr(),
            mass: self.mass.as_ptr(),
            com: self.com.as_ptr(),
            inertia_com: self.inertia_com.as_ptr(),
            gravity: [0.0, 0.0, 9.81], // rigidbody/src/multibody.rs:118
        }
    }
}

// ------------------------------------------------------------------ safe wrapper
/// One chain resident on one GPU.  `Send` but not `Sync`: host-batch calls share staging buffers.
pub struct GpuMultibody {
    raw: *mut RbGpu,
    n: usize,
}
unsafe impl Send for GpuMultibody {}

impl GpuMultibody {
    pub fn new(mb: &Multibody, device: i32) -> Result<Self, RbError> {
        let arrays = ChainArrays::from_multibody(mb);
        let desc = arrays.desc();
        let mut raw = ptr::null_mut();
        check(unsafe { multibody_gpu_new(&desc, device, &mut raw) })?;
        Ok(GpuMultibody { raw, n: arrays.mass.len() })
    }

    /// One engine over several GPUs of the box (multibody_gpu_new_multi): every host batch is cut into `devices.len()`
    /// contiguous slices, one per device; results equal a single-device engine's bit for bit.
    pub fn new_multi(mb: &Multibody, devices: &[i32]) -> Result<Self, RbError> {
        let arrays = ChainArrays::from_multibody(mb);
        let desc = arrays.desc();
        let mut raw = ptr::null_mut();
        check(unsafe { multibody_gpu_new_multi(&desc, devices.as_ptr(), devices.len() as c_int, &mut raw) })?;
        Ok(GpuMultibody { raw, n: arrays.mass.len() })
    }

    /// Kernel family serving this chain ("fr3-specialised", "jit-specialised", ...).
    pub fn kernel_variant(&self) -> String {
        unsafe { CStr::from_ptr(multibody_gpu_kernel_variant(self.raw)) }.to_string_lossy().into_owned()
    }

    pub fn n_devices(&self) -> usize {
        unsafe { multibody_gpu_n_devices(self.raw) as usize }
    }

    fn check_len(&self, what: &str, len: usize, per_state: usize, n_states: usize) -> Result<(), RbError> {
        if len != per_state * n_states {
            return Err(RbError { code: -2, message: format!("{what}: expected {} doubles, got {len}", per_state * n_states) });
        }
        Ok(())
    }

    /// Batched superset of `multibody_rnea` (rigidbody_bindings/src/lib.rs:15-30); host slices.
    pub fn rnea_batch(&mut self, q: &[f64], dq: &[f64], ddq: &[f64], tau: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        for (w, s) in [("q", q.len()), ("dq", dq.len()), ("ddq", ddq.len()), ("tau", tau.len())] {
            self.check_len(w, s, self.n, n_states)?;
        }
        check(unsafe { multibody_rnea_batch(self.raw, q.as_ptr(), dq.as_ptr(), ddq.as_ptr(), tau.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// qdd = solve(sym(crba(q)), tau - rnea(q, dq, 0)); host slices.
    pub fn forward_dynamics_batch(&mut self, q: &[f64], dq: &[f64], tau: &[f64], qdd: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        for (w, s) in [("q", q.len()), ("dq", dq.len()), ("tau", tau.len()), ("qdd", qdd.len())] {
            self.check_len(w, s, self.n, n_states)?;
        }
        check(unsafe { multibody_forward_dynamics_batch(self.raw, q.as_ptr(), dq.as_ptr(), tau.as_ptr(), qdd.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// Inverse AND forward dynamics of the same states in one call: `out` holds 2n doubles per state, tau then qdd
    /// (SoA: rows 0..n-1 tau, n..2n-1 qdd).  q and dq cross the bus once and one fused kernel serves both results; this
    /// is the call the end-to-end benchmark figure is measured through.
    #[allow(clippy::too_many_arguments)]
    pub fn rnea_fd_batch(&mut self, q: &[f64], dq: &[f64], ddq: &[f64], tau_in: &[f64], out: &mut [f64], n_states: usize,
                         layout: RbLayout) -> Result<(), RbError> {
        for (w, s) in [("q", q.len()), ("dq", dq.len()), ("ddq", ddq.len()), ("tau_in", tau_in.len())] {
            self.check_len(w, s, self.n, n_states)?;
        }
        self.check_len("out", out.len(), 2 * self.n, n_states)?;
        check(unsafe { multibody_rnea_fd_batch(self.raw, q.as_ptr(), dq.as_ptr(), ddq.as_ptr(), tau_in.as_ptr(), out.as_mut_ptr(), n_states, 0, layout,
                                               RbMem::Host, ptr::null_mut()) })
    }

    /// Batched superset of `multibody_crba` (lib.rs:32-43): n*n entries per state, entry r + n*c.
    pub fn crba_batch(&mut self, q: &[f64], h: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q", q.len(), self.n, n_states)?;
        self.check_len("h", h.len(), self.n * self.n, n_states)?;
        check(unsafe { multibody_crba_batch(self.raw, q.as_ptr(), h.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// Semi-implicit Euler rollout; `tau` is `horizon` consecutive state arrays; returns the full trajectory.
    #[allow(clippy::too_many_arguments)]
    pub fn rollout(&mut self, q0: &[f64], dq0: &[f64], tau: &[f64], dt: f64, horizon: usize, q_traj: &mut [f64], dq_traj: &mut [f64],
                   n_traj: usize, layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q0", q0.len(), self.n, n_traj)?;
        self.check_len("dq0", dq0.len(), self.n, n_traj)?;
        for (w, s) in [("tau", tau.len()), ("q_traj", q_traj.len()), ("dq_traj", dq_traj.len())] {
            self.check_len(w, s, self.n * horizon, n_traj)?;
        }
        check(unsafe { multibody_rollout(self.raw, q0.as_ptr(), dq0.as_ptr(), tau.as_ptr(), dt, horizon as c_int, q_traj.as_mut_ptr(), dq_traj.as_mut_ptr(),
                                         ptr::null_mut(), ptr::null_mut(), n_traj, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// Tip translations (lib.rs:46-57) and tip-frame Jacobians (lib.rs:60-70), batched; host slices.
    pub fn fwd_kin_batch(&mut self, q: &[f64], xyz: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q", q.len(), self.n, n_states)?;
        self.check_len("xyz", xyz.len(), 3, n_states)?;
        check(unsafe { multibody_fwd_kin_batch(self.raw, q.as_ptr(), xyz.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    pub fn jac_batch(&mut self, q: &[f64], jac: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q", q.len(), self.n, n_states)?;
        self.check_len("jac", jac.len(), 6 * self.n, n_states)?;
        check(unsafe { multibody_jac_batch(self.raw, q.as_ptr(), jac.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// Rollout fused with a quadratic cost: one scalar per trajectory (sampling-based MPC); nothing but `tau` is read
    /// per step and no trajectory is written.
    #[allow(clippy::too_many_arguments)]
    pub fn rollout_cost(&mut self, q0: &[f64], dq0: &[f64], tau: &[f64], dt: f64, horizon: usize, w: &RbQuadCost, cost: &mut [f64],
                        n_traj: usize, layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q0", q0.len(), self.n, n_traj)?;
        self.check_len("dq0", dq0.len(), self.n, n_traj)?;
        self.check_len("tau", tau.len(), self.n * horizon, n_traj)?;
        self.check_len("cost", cost.len(), 1, n_traj)?;
        check(unsafe { multibody_rollout_cost(self.raw, q0.as_ptr(), dq0.as_ptr(), tau.as_ptr(), dt, horizon as c_int, w, cost.as_mut_ptr(),
                                              ptr::null_mut(), ptr::null_mut(), n_traj, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// `rollout_cost` plus its gradient (multibody_rollout_cost_grad): the same cost, bit for bit, and d cost / d tau
    /// (shaped like `tau`), d cost / d q0 and d cost / d dq0 (shaped like `q0`); serial chains of at most 12 joints.
    #[allow(clippy::too_many_arguments)]
    pub fn rollout_cost_grad(&mut self, q0: &[f64], dq0: &[f64], tau: &[f64], dt: f64, horizon: usize, w: &RbQuadCost, cost: &mut [f64],
                             grad_tau: &mut [f64], grad_q0: &mut [f64], grad_dq0: &mut [f64], n_traj: usize, layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q0", q0.len(), self.n, n_traj)?;
        self.check_len("dq0", dq0.len(), self.n, n_traj)?;
        self.check_len("tau", tau.len(), self.n * horizon, n_traj)?;
        self.check_len("cost", cost.len(), 1, n_traj)?;
        self.check_len("grad_tau", grad_tau.len(), self.n * horizon, n_traj)?;
        self.check_len("grad_q0", grad_q0.len(), self.n, n_traj)?;
        self.check_len("grad_dq0", grad_dq0.len(), self.n, n_traj)?;
        check(unsafe { multibody_rollout_cost_grad(self.raw, q0.as_ptr(), dq0.as_ptr(), tau.as_ptr(), dt, horizon as c_int, w, cost.as_mut_ptr(),
                                                   grad_tau.as_mut_ptr(), grad_q0.as_mut_ptr(), grad_dq0.as_mut_ptr(), n_traj, 0, layout,
                                                   RbMem::Host, ptr::null_mut()) })
    }

    /// `rollout_cost_grad` with the tip-pose terms of `tip` added (multibody_rollout_tip_cost_grad); host slices, shapes as
    /// `rollout_cost_grad`.  Serial chains of at most 12 joints.
    #[allow(clippy::too_many_arguments)]
    pub fn rollout_tip_cost_grad(&mut self, q0: &[f64], dq0: &[f64], tau: &[f64], dt: f64, horizon: usize, w: &RbQuadCost, tip: &RbTipCost,
                                 cost: &mut [f64], grad_tau: &mut [f64], grad_q0: &mut [f64], grad_dq0: &mut [f64], n_traj: usize,
                                 layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q0", q0.len(), self.n, n_traj)?;
        self.check_len("dq0", dq0.len(), self.n, n_traj)?;
        self.check_len("tau", tau.len(), self.n * horizon, n_traj)?;
        self.check_len("cost", cost.len(), 1, n_traj)?;
        self.check_len("grad_tau", grad_tau.len(), self.n * horizon, n_traj)?;
        self.check_len("grad_q0", grad_q0.len(), self.n, n_traj)?;
        self.check_len("grad_dq0", grad_dq0.len(), self.n, n_traj)?;
        check(unsafe { multibody_rollout_tip_cost_grad(self.raw, q0.as_ptr(), dq0.as_ptr(), tau.as_ptr(), dt, horizon as c_int, w, tip,
                                                       cost.as_mut_ptr(), grad_tau.as_mut_ptr(), grad_q0.as_mut_ptr(), grad_dq0.as_mut_ptr(),
                                                       n_traj, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// Inverse kinematics of the tip frame (multibody_ik_batch): one damped least-squares problem per entry, host slices.
    /// `q_init` n values per problem, `p_target` 3, `r_target` 9 (row-major; may be empty when `opt.w_r == 0`), `out` n + 3:
    /// q, position error, rotation angle error, iterations (-1 = not converged).
    #[allow(clippy::too_many_arguments)]
    pub fn ik(&mut self, q_init: &[f64], p_target: &[f64], r_target: &[f64], opt: &RbIkOptions, out: &mut [f64], n_problems: usize,
              layout: RbLayout) -> Result<(), RbError> {
        self.check_len("q_init", q_init.len(), self.n, n_problems)?;
        self.check_len("p_target", p_target.len(), 3, n_problems)?;
        if opt.w_r != 0.0 {
            self.check_len("r_target", r_target.len(), 9, n_problems)?;
        }
        self.check_len("out", out.len(), self.n + 3, n_problems)?;
        let r = if opt.w_r != 0.0 { r_target.as_ptr() } else { ptr::null() };
        check(unsafe { multibody_ik_batch(self.raw, q_init.as_ptr(), p_target.as_ptr(), r, opt, out.as_mut_ptr(), n_problems, 0, layout,
                                          RbMem::Host, ptr::null_mut()) })
    }

    /// d tau / d q and d tau / d dq (2 n*n doubles per state, block b entry r + n*c); serial chains of at most 32 joints.
    pub fn rnea_derivatives_batch(&mut self, q: &[f64], dq: &[f64], ddq: &[f64], out: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        for (w, s) in [("q", q.len()), ("dq", dq.len()), ("ddq", ddq.len())] {
            self.check_len(w, s, self.n, n_states)?;
        }
        self.check_len("out", out.len(), 2 * self.n * self.n, n_states)?;
        check(unsafe { multibody_rnea_derivatives_batch(self.raw, q.as_ptr(), dq.as_ptr(), ddq.as_ptr(), out.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// d qdd / d q, d qdd / d dq and H^-1 (3 n*n doubles per state) of qdd = forward_dynamics(q, dq, tau); serial chains
    /// of at most 12 joints.
    pub fn fd_derivatives_batch(&mut self, q: &[f64], dq: &[f64], tau: &[f64], out: &mut [f64], n_states: usize, layout: RbLayout) -> Result<(), RbError> {
        for (w, s) in [("q", q.len()), ("dq", dq.len()), ("tau", tau.len())] {
            self.check_len(w, s, self.n, n_states)?;
        }
        self.check_len("out", out.len(), 3 * self.n * self.n, n_states)?;
        check(unsafe { multibody_fd_derivatives_batch(self.raw, q.as_ptr(), dq.as_ptr(), tau.as_ptr(), out.as_mut_ptr(), n_states, 0, layout, RbMem::Host, ptr::null_mut()) })
    }

    /// Raw handle for device-pointer calls (RbMem::Device) from CUDA-aware callers.
    pub fn raw(&mut self) -> *mut RbGpu {
        self.raw
    }

    pub fn sync(&mut self) -> Result<(), RbError> {
        check(unsafe { multibody_gpu_sync(self.raw) })
    }

    /// Waits for the device, then reports (and clears) the status device-pointer calls accumulated: Err(code -5) if a
    /// forward-dynamics state met a mass matrix that is not positive definite.
    pub fn status(&mut self) -> Result<(), RbError> {
        check(unsafe { multibody_gpu_status(self.raw) })
    }

    /// Optional fp32 mode on DEVICE-resident SoA batches (1e-4 tolerance, include/rigidbody.h); raw pointers because
    /// device memory is the caller's (cust / cudarc / raw CUDA).
    ///
    /// # Safety
    /// All four pointers must be device pointers on this engine's GPU to `n * ld` floats each.
    pub unsafe fn rnea_batch_f32_device(&mut self, q: *const f32, dq: *const f32, ddq: *const f32, tau: *mut f32, n_states: usize, ld: usize,
                                        stream: *mut c_void) -> Result<(), RbError> {
        check(multibody_rnea_batch_f32(self.raw, q, dq, ddq, tau, n_states, ld, stream))
    }

    /// # Safety
    /// As `rnea_batch_f32_device`.
    pub unsafe fn forward_dynamics_batch_f32_device(&mut self, q: *const f32, dq: *const f32, tau: *const f32, qdd: *mut f32, n_states: usize,
                                                    ld: usize, stream: *mut c_void) -> Result<(), RbError> {
        check(multibody_forward_dynamics_batch_f32(self.raw, q, dq, tau, qdd, n_states, ld, stream))
    }
}

/// Pinned (page-locked) host memory from `multibody_host_alloc`: host batches in such buffers are copied at full PCIe
/// rate, overlapped with compute; pageable slices work too but at a fraction of the rate (INTEGRATION.md).
pub struct PinnedBuffer {
    ptr: *mut f64,
    len: usize,
}
unsafe impl Send for PinnedBuffer {}

impl PinnedBuffer {
    pub fn new(len: usize) -> Result<Self, RbError> {
        let mut p: *mut c_void = ptr::null_mut();
        check(unsafe { multibody_host_alloc(&mut p, len * std::mem::size_of::<f64>()) })?;
        unsafe { ptr::write_bytes(p as *mut f64, 0, len) };
        Ok(PinnedBuffer { ptr: p as *mut f64, len })
    }
    pub fn as_slice(&self) -> &[f64] {
        unsafe { std::slice::from_raw_parts(self.ptr, self.len) }
    }
    pub fn as_mut_slice(&mut self) -> &mut [f64] {
        unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) }
    }
}

impl Drop for PinnedBuffer {
    fn drop(&mut self) {
        unsafe { multibody_host_free(self.ptr as *mut c_void) }
    }
}

impl Drop for GpuMultibody {
    fn drop(&mut self) {
        unsafe { multibody_gpu_free(self.raw) }
    }
}

// ------------------------------------------------------------------ the one new exported C symbol
/// `int multibody_gpu_from_rust(const Multibody* mb, int device, RbGpu** out)`: lets a C/C++ program that holds
/// the Rust `Multibody*` from `multibody_new()` (rigidbody_bindings/src/lib.rs:8-12) obtain an engine handle.
/// Unlike the reference's exports it never unwinds across the boundary.
#[no_mangle]
pub unsafe extern "C" fn multibody_gpu_from_rust(mb: *const Multibody, device: c_int, out: *mut *mut RbGpu) -> c_int {
    let result = std::panic::catch_unwind(|| {
        let Some(mb) = mb.as_ref() else { return -1 };
        if out.is_null() {
            return -1;
        }
        let arrays = ChainArrays::from_multibody(mb);
        let desc = arrays.desc();
        multibody_gpu_new(&desc, device, out)
    });
    result.unwrap_or(-2)
}
