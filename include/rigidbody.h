/*
 * rigidbody.h -- C ABI of the B200 batched rigid-body dynamics engine.
 *
 * A superset of the reference's rigidbody_bindings/rigidbody.h:11-16.  Part 1 keeps the six
 * single-state symbols with the reference's signatures (so rigidbody_bindings/main.cpp:66-98 links
 * unchanged).  Part 2 adds the batched, caller-allocated, status-returning entry points that the
 * reference's FFI crate (rigidbody_bindings/src/lib.rs) would bind for the batched hot path.
 *
 * Valid as C and as C++ (the reference header is only valid C++: bare `Multibody*` after
 * `struct Multibody;`, rigidbody.h:8,11).  Nothing here mentions torch, CUDA types or C++ types:
 * plain pointers, sizes and enums only.  No call throws or aborts across the boundary; every
 * fallible call returns an RbStatus and records a message readable with multibody_last_error().
 * There is no CPU fallback: without a usable sm_100 device the constructors fail with RB_ERR_CUDA.
 */
#ifndef MULTIBODY_INTERFACE_H
#define MULTIBODY_INTERFACE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ===================================================================== Part 1: reference symbols */
/* Opaque single-model handle; replaces the Rust `Multibody` (rigidbody/src/multibody.rs:32). */
typedef struct Multibody Multibody;

/* rigidbody_bindings/src/lib.rs:8-12.  The reference hard-codes an absolute URDF path (:10); here the
 * path comes from $RIGIDBODY_URDF, else "assets/fr3.urdf" relative to the working directory.
 * Returns NULL on failure (the reference panics). */
Multibody* multibody_new(void);
/* Explicit-path variant of the above (new). */
Multibody* multibody_new_from_urdf(const char* urdf_path);
/* lib.rs:46-57 -> 3 doubles (tip translation).  Result is malloc'ed; release with multibody_free_result
 * (the reference leaks it, lib.rs:55). */
double* multibody_fwd_kin(const Multibody* mb, const double q[7]);
/* lib.rs:60-70 -> 6 x n doubles column-major, rows lin(0-2) then rot(3-5), tip frame. */
double* multibody_jac(const Multibody* mb, const double q[7]);
/* lib.rs:15-30 -> n doubles. */
double* multibody_rnea(const Multibody* mb, const double q[7], const double dq[7], const double ddq[7]);
/* lib.rs:32-43 -> n x n doubles column-major; diagonal + strict upper triangle, lower = 0, as
 * multibody.rs:155-174 leaves it. */
double* multibody_crba(const Multibody* mb, const double q[7]);
/* lib.rs:73-78, null-safe. */
void multibody_free(Multibody* mb);
/* New: frees an array returned by the four calls above (null-safe). */
void multibody_free_result(double* p);
/* New: number of movable joints kept by from_urdf (7 for the FR3; the reference panics otherwise, multibody.rs:76). */
int multibody_n_joints(const Multibody* mb);
/* New: the flattened model as loaded on the host (no GPU needed): parent_rot [9n], parent_trans [3n], mass [n],
 * h = m*com [3n], inertia_origin [6n] (xx xy xz yy yz zz), in the engine's joint frames (equal to the URDF's when
 * every axis is +z, re-based so that the axis is z otherwise).  Any output may be NULL. */
int multibody_get_model(const Multibody* mb, double* parent_rot, double* parent_trans, double* mass,
                        double* h, double* inertia_origin);

/* New: the chain exactly as the reference's Multibody holds it after from_urdf, field for field what
 * `for jt in mb.iter()` (multibody.rs:79-81) exposes: jt.axis (joint.rs:27), jt.parent rotation (row-major 3x3) and
 * translation (joint.rs:29), jt.body.mass / com / inertia_com (inertia.rs:13-15, row-major 3x3), plus the parent
 * index (i-1 for the reference's serial chains).  These are the arrays of an RbChainDesc: a C caller (or the C test
 * double of the Rust crate, examples/rust_crate_double.c) flattens a Multibody with this one call.  Arrays sized as
 * in RbChainDesc; any output may be NULL. */
int multibody_get_chain(const Multibody* mb, int32_t* parent, double* axis, double* parent_rot, double* parent_trans,
                        double* mass, double* com, double* inertia_com);

/* ===================================================================== Part 2: batched engine */
typedef enum RbStatus {
    RB_OK = 0,
    RB_ERR_NULL = -1,          /* a required pointer was NULL */
    RB_ERR_ARG = -2,           /* bad size / layout / enum / chain */
    RB_ERR_URDF = -3,          /* URDF could not be read or holds no movable joint */
    RB_ERR_CUDA = -4,          /* CUDA runtime error or no usable device (no CPU fallback exists) */
    RB_ERR_NOT_SPD = -5,       /* forward dynamics met a mass matrix that is not positive definite */
    RB_ERR_UNSUPPORTED = -6    /* valid request this build cannot serve (e.g. n_joints > RB_MAX_JOINTS) */
} RbStatus;

/* Batch layout of every state array. */
typedef enum RbLayout {
    RB_LAYOUT_SOA = 0,   /* joint-major [n_joints][ld]: element (joint i, state s) at i*ld + s.  Native, coalesced. */
    RB_LAYOUT_AOS = 1    /* state-major [n_states][n_joints]: the reference's per-state double[7], repeated. */
} RbLayout;

/* Where the pointers passed to a batched call live. */
typedef enum RbMem {
    RB_MEM_HOST = 0,     /* host memory (pinned or pageable); the call copies in, computes, copies out */
    RB_MEM_DEVICE = 1    /* device memory on the engine's GPU; nothing is copied */
} RbMem;

#define RB_MAX_JOINTS 64

/*
 * Flattened, topologically ordered chain descriptor: what the Rust side extracts from
 * `Multibody::iter()` (multibody.rs:79-81) and the pub fields of RevoluteJoint / Inertia
 * (joint.rs:26-31, inertia.rs:12-17).  All arrays are borrowed for the duration of the call.
 */
typedef struct RbChainDesc {
    int32_t n_joints;             /* 1..RB_MAX_JOINTS */
    const int32_t* parent;        /* [n] parent link index, -1 = base, parent[i] < i (topological order).  NULL = serial
                                     chain (i-1), the reference's only case (multibody.rs:148,165) and the one the
                                     ahead-of-time kernel families serve; a branching tree gets run-time specialised kernels (<= 18
                                     joints) or the run-time-n family.
                                     The tip of fwd_kin / jac is the last link; H(j, i) = 0 and the Jacobian column
                                     of j is 0 where joint j does not support link i / the tip. */
    const double* axis;           /* [3n] joint axes in the joint frames (joint.rs:27), any non-zero vector (normalised
                                     on load, joint.rs:56).  NULL = all +z.  The reference's rnea/crba hard-code z
                                     (multibody.rs:29,130) and agree with its own kinematics only for +z; here a
                                     non-z axis is used consistently: the loader re-bases the joint frame so that
                                     the axis becomes z, and the kernels stay z-only.  tau, qdd, H, fwd_kin and jac
                                     are those of the chain as described. */
    const double* parent_rot;     /* [9n] row-major rotation of joint frame i in link i-1 (joint.rs:29 .rotation) */
    const double* parent_trans;   /* [3n] translation of joint frame i in link i-1 (joint.rs:29 .translation) */
    const double* mass;           /* [n]  inertia.rs:13 */
    const double* com;            /* [3n] inertia.rs:14, in link coordinates */
    const double* inertia_com;    /* [9n] row-major, about the COM (inertia.rs:15) */
    double gravity[3];            /* base linear acceleration; the reference uses (0,0,+9.81) (multibody.rs:118) */
} RbChainDesc;

/* Per-joint limits read from the URDF (sampling synthetic states; not used by the dynamics). */
typedef struct RbJointLimits {
    double lower[RB_MAX_JOINTS], upper[RB_MAX_JOINTS], velocity[RB_MAX_JOINTS], effort[RB_MAX_JOINTS];
} RbJointLimits;

/* Opaque engine: one chain descriptor resident on one GPU, plus its streams and staging buffers (or, from
 * multibody_gpu_new_multi, one such engine per listed GPU behind a single handle). */
typedef struct RbGpu RbGpu;

/* ---- construction -------------------------------------------------------------------------- */
/* Upload a descriptor to CUDA device `device` (ordinal).  Replaces nothing in the reference: it is the
 * one-time "flatten + upload" step the north star adds next to multibody_new. */
int multibody_gpu_new(const RbChainDesc* desc, int device, RbGpu** out);
/* Load a URDF exactly as Multibody::from_urdf does (multibody.rs:65-77: k-th joint zipped with k-th link in
 * document order, joints whose type contains "fixed" dropped; joint.rs:53-68), then upload. */
int multibody_gpu_new_from_urdf(const char* urdf_path, int device, RbGpu** out);
/* Engine for an existing reference-style handle. */
int multibody_gpu_from_multibody(const Multibody* mb, int device, RbGpu** out);
void multibody_gpu_free(RbGpu* g);
#ifdef RIGIDBODY_HAVE_RUST_BRIDGE
/* Exported by the Rust crate rust/rigidbody_gpu_bindings (not by librigidbody_b200.so), for callers that hold the
 * reference crate's own `Multibody*` (rigidbody_bindings/src/lib.rs:8-12): flattens it with ChainArrays::from_multibody
 * (multibody.rs:79-81, joint.rs:26-31, inertia.rs:12-17) and calls multibody_gpu_new.  See INTEGRATION.md. */
int multibody_gpu_from_rust(const Multibody* mb, int device, RbGpu** out);
#endif

/* ---- one engine over several GPUs of the box ------------------------------------------------- */
/* The one-call shape of the reference (rigidbody_bindings/src/lib.rs:15-30: one host batch in, one result out) over
 * n_dev devices: the chain is uploaded to every device listed, and every RB_MEM_HOST batch call on the returned handle
 * cuts its batch into n_dev contiguous slices (device i owns states [B*i/n_dev, B*(i+1)/n_dev)), each moved and computed
 * by its own host thread, copy streams and staging buffers; the call returns when the last device has written its slice
 * of `out`.  No collective and no peer traffic: results are those of a single-device engine, bit for bit.
 * RB_MEM_DEVICE calls need pointers on ONE device: they return RB_ERR_UNSUPPORTED on this handle; use the per-device
 * engines (multibody_gpu_peer) for device-resident slices.  n_dev = 1 returns an ordinary engine.  devices: distinct
 * CUDA ordinals.  Free with multibody_gpu_free (frees the per-device engines too). */
int multibody_gpu_new_multi(const RbChainDesc* desc, const int* devices, int n_dev, RbGpu** out);
int multibody_gpu_new_multi_from_urdf(const char* urdf_path, const int* devices, int n_dev, RbGpu** out);
/* Devices behind a handle (1 for an ordinary engine) and the single-device engine of device slot `index` (the handle
 * itself for an ordinary engine and index 0); owned by the handle, never freed by the caller. */
int multibody_gpu_n_devices(const RbGpu* g);
RbGpu* multibody_gpu_peer(RbGpu* g, int index);

/* ---- introspection ------------------------------------------------------------------------- */
int multibody_gpu_n_joints(const RbGpu* g);
int multibody_gpu_device(const RbGpu* g);
/* Which kernel family serves this chain: "fr3-specialised" / "chain32-specialised" (compiled in), "jit-specialised"
 * (the same kernels compiled for this chain's constants at load time with NVRTC, cached on disk; <= 18 joints),
 * "jit-long" (19..32 joints: rnea / crba / fwd_kin / jac compiled at load time, the rest run-time-n), "generic-7",
 * "generic-n" (run-time constants).  $RIGIDBODY_B200_VARIANT forces one, $RIGIDBODY_B200_JIT=0 disables the JIT,
 * $RIGIDBODY_B200_CACHE moves the cache directory (default ~/.cache/rigidbody_b200; empty string = no cache). */
const char* multibody_gpu_kernel_variant(const RbGpu* g);
/* Human-readable note on that choice (e.g. why the run-time compiler was not used). */
const char* multibody_gpu_family_note(const RbGpu* g);
/* Compile and cache the specialised kernels of a chain ahead of time (descriptor, or URDF path when desc is NULL).
 * Needs libnvrtc but no GPU; `log` (optional) receives the compiler log. */
int multibody_jit_precompile(const RbChainDesc* desc, const char* urdf_path, char* log, size_t log_len);
/* Copies the flattened descriptor the engine uploaded (tests compare it with the oracle's model):
 * parent_rot [9n], parent_trans [3n], mass [n], h = m*com [3n], inertia_origin [6n] (xx xy xz yy yz zz). */
int multibody_gpu_get_model(const RbGpu* g, double* parent_rot, double* parent_trans, double* mass,
                            double* h, double* inertia_origin);
int multibody_gpu_get_limits(const RbGpu* g, RbJointLimits* out);
/* Thread-local message of the last failing call on this thread ("" if none). */
const char* multibody_last_error(void);

/* ---- the batched hot path ------------------------------------------------------------------ */
/*
 * Common arguments:  n_states states; `ld` = leading dimension in elements for RB_LAYOUT_SOA (>= n_states;
 * 0 means n_states), ignored for AOS; `mem` says where ALL pointers of the call live.
 * RB_MEM_DEVICE calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = the legacy default
 * stream, as in every CUDA library) and return after the launch; sync the stream (or call multibody_gpu_sync)
 * before reading.  `stream` is ignored by RB_MEM_HOST calls.
 * RB_MEM_HOST calls are synchronous: the batch is cut into chunks that flow host -> device staging buffer -> kernel
 * -> device staging buffer -> host on three streams (H2D, compute and D2H of different chunks overlap); copies read and
 * write the CALLER's memory directly, there is no pinned bounce buffer.  Pinned caller memory (multibody_host_alloc, or
 * cudaHostRegister on memory the caller already owns) makes those copies asynchronous DMA at PCIe rate; with pageable
 * memory the CUDA runtime stages every copy itself, the overlap is lost and throughput drops (measured: see
 * profiles/ and bench.py's e2e.pageable).  The call returns when `out` is complete.
 * With n_states = 1, AOS, HOST these are the reference's single-state calls minus the leak.
 */

/* tau = ID(q, dq, ddq): multibody_rnea (lib.rs:15-30) = get_transforms (multibody.rs:83-85) + rnea (:111-153). */
int multibody_rnea_batch(RbGpu* g, const double* q, const double* dq, const double* ddq, double* tau,
                         size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* qdd = FD(q, dq, tau) = chol_solve(sym(crba(q)), tau - rnea(q, dq, 0)) -- composed from multibody.rs:111-153
 * (ddq = 0) and :155-174; the solve is new (SURVEY.md 3.3).  For RB_MEM_HOST calls a non-SPD mass matrix
 * yields RB_ERR_NOT_SPD (qdd of that state is NaN); for device calls query multibody_gpu_status. */
int multibody_forward_dynamics_batch(RbGpu* g, const double* q, const double* dq, const double* tau, double* qdd,
                                     size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Optional fp32 mode of the two calls above (BASELINE.json: "an optional fp32 mode is held to a stated 1e-4
 * tolerance"): the same kernels with float arithmetic and float arrays, for DEVICE-resident SoA batches only
 * (ld as above; asynchronous on `stream`).  Tolerance against the fp64 reference on the same float inputs, per state
 * max_i |x_i - ref_i| <= 1e-4 * max(1, ||ref||_inf) (measured over FR3 states within joint limits: inverse
 * dynamics 3.3e-6, forward dynamics 1.2e-5; cond(H) <= ~1e3).
 * Families without fp32 kernels (run-time-n, 32-joint) return RB_ERR_UNSUPPORTED. */
int multibody_rnea_batch_f32(RbGpu* g, const float* q, const float* dq, const float* ddq, float* tau,
                             size_t n_states, size_t ld, void* stream);
int multibody_forward_dynamics_batch_f32(RbGpu* g, const float* q, const float* dq, const float* tau, float* qdd,
                                         size_t n_states, size_t ld, void* stream);

/* H = crba(q): multibody_crba (lib.rs:32-43).  Output convention of the reference: n*n entries per state,
 * entry k = r + n*c (column-major), diagonal + strict upper triangle filled, strict lower = 0.
 * SOA: H[k*ld + s];  AOS: H[s*n*n + k]. */
int multibody_crba_batch(RbGpu* g, const double* q, double* H,
                         size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* New: inverse AND forward dynamics of the same states in one call -- tau = rnea(q, dq, ddq) and
 * qdd = forward_dynamics(q, dq, tau_in).  Same kernels and results as the two separate calls; q and dq cross the bus
 * (host batches) and are staged once instead of twice.  out holds 2n entries per state: tau then qdd
 * (SOA: out[(blk*n + i)*ld + s];  AOS: out[s*2n + blk*n + i]). */
int multibody_rnea_fd_batch(RbGpu* g, const double* q, const double* dq, const double* ddq, const double* tau_in,
                            double* out, size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* New (README.md:18 lists "Differentiability" as not done): analytical first derivatives of serial chains: inverse
 * dynamics up to 32 joints, forward dynamics up to 12 (RB_ERR_UNSUPPORTED otherwise, and for kinematic trees).
 * multibody_rnea_derivatives_batch: out holds 2 n*n entries per state, block 0 = d tau / d q, block 1 = d tau / d dq of
 *   tau = rnea(q, dq, ddq); within a block entry k = r + n*c is d tau_r / d x_c (column-major, like crba).
 *   (d tau / d ddq is crba(q).)   SOA: out[(blk*n*n + k)*ld + s];  AOS: out[s*2*n*n + blk*n*n + k].
 * multibody_fd_derivatives_batch: out holds 3 n*n entries per state: d qdd / d q, d qdd / d dq and H^-1 = d qdd / d tau
 *   of qdd = forward_dynamics(q, dq, tau); same entry convention.  States with a non-SPD mass matrix get NaN. */
int multibody_rnea_derivatives_batch(RbGpu* g, const double* q, const double* dq, const double* ddq, double* out,
                                     size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);
int multibody_fd_derivatives_batch(RbGpu* g, const double* q, const double* dq, const double* tau, double* out,
                                   size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Tip translation: multibody_fwd_kin (lib.rs:46-57).  3 entries per state (SOA: xyz[k*ld + s]; AOS: xyz[3s + k]). */
int multibody_fwd_kin_batch(RbGpu* g, const double* q, double* xyz,
                            size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Tip-frame Jacobian: multibody_jac (lib.rs:60-70).  6n entries per state, entry k = r + 6*c. */
int multibody_jac_batch(RbGpu* g, const double* q, double* J,
                        size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* MPC rollout (SURVEY.md a14): for t in 0..horizon: qdd = FD(q, dq, tau[t]); dq += dt*qdd; q += dt*dq.
 * q0, dq0: one state array each (layout/ld as above).  tau: `horizon` consecutive state arrays
 * (SOA: [horizon][n][ld]; AOS: [horizon][n_traj][n]).  q_traj/dq_traj: same shape as tau, the state AFTER
 * each step; either may be NULL.  q_final/dq_final (one state array each) may be NULL. */
int multibody_rollout(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                      double* q_traj, double* dq_traj, double* q_final, double* dq_final,
                      size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Fused rollout + running cost for sampling-based MPC (MPPI-style; SURVEY.md 8f.4): the same integration as
 * multibody_rollout, but instead of the trajectory it returns one scalar per trajectory,
 *   cost = sum_t dt * sum_i [ w_q[i] (q_i(t+1) - q_ref[i])^2 + w_dq[i] dq_i(t+1)^2 + w_tau[i] tau_i(t)^2 ]
 *          + sum_i [ w_q_final[i] (q_i(H) - q_ref[i])^2 + w_dq_final[i] dq_i(H)^2 ],
 * so nothing but tau is read and n_traj doubles are written.  Weight arrays are host arrays of n_joints
 * non-negative doubles (NULL = zeros).  cost has n_traj entries (host or device, as `mem` says); a trajectory that
 * met a non-SPD mass matrix gets NaN.  q_final / dq_final (one state array each) may be NULL. */
typedef struct RbQuadCost {
    const double* q_ref;
    const double* w_q;
    const double* w_dq;
    const double* w_tau;
    const double* w_q_final;
    const double* w_dq_final;
} RbQuadCost;
int multibody_rollout_cost(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                           const RbQuadCost* weights, double* cost, double* q_final, double* dq_final,
                           size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Gradients of rollouts, for gradient-based MPC and trajectory optimisation: one adjoint pass backwards through the
 * rollout (one thread per trajectory, O(n) per step), serial chains of at most 12 joints (RB_ERR_UNSUPPORTED otherwise,
 * and for kinematic trees), fp64.  They are the gradients of the exact-arithmetic rollout map evaluated at the computed
 * states, not of its rounded floating-point evaluation.  Layouts, ld, host/device memory, horizon == 0, multi-device
 * handles and status reporting as multibody_rollout; a trajectory that meets a non-SPD mass matrix gets NaN gradients.
 * Reverse-mode (vector-Jacobian) product of multibody_rollout.  q_traj / dq_traj: what multibody_rollout returned for
 * these q0, dq0, tau, dt (the states the pass linearises about; not re-checked).  g_*: upstream gradients shaped like the
 * matching rollout outputs, each may be NULL (= 0).  grad_tau shaped like tau, grad_q0 / grad_dq0 like q0; each may be NULL.
 * With horizon == 0 tau and the trajectory are not read, grad_q0 = g_q_final and grad_dq0 = g_dq_final. */
int multibody_rollout_vjp(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                          const double* q_traj, const double* dq_traj,
                          const double* g_q_traj, const double* g_dq_traj, const double* g_q_final, const double* g_dq_final,
                          double* grad_tau, double* grad_q0, double* grad_dq0,
                          size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream);
/* multibody_rollout_cost plus its gradient: cost bit-identical to multibody_rollout_cost on the same engine, and
 * d cost / d tau, d cost / d q0, d cost / d dq0 (each may be NULL).  Device calls take a workspace of at most 1 GiB per
 * chunk of trajectories in stream order on `stream` (cudaMallocAsync). */
int multibody_rollout_cost_grad(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                const RbQuadCost* weights, double* cost, double* grad_tau, double* grad_q0, double* grad_dq0,
                                size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Tip-pose tracking terms for the fused rollout cost and its gradient: MPC tasks stated at the end effector.
 * The tip frame is the frame of multibody_jac: the reference's last link frame (for a kinematic tree the last link,
 * reached along its supporting branch).  Its origin is what multibody_fwd_kin returns.  With R(q) its orientation in
 * the base frame and x(q) = p(q) + R(q) offset the tracked point,
 *   cost = [every term of multibody_rollout_cost for `weights`]
 *        + sum_{t=0}^{H-1} dt * ( sum_k w_p[k] (x_k(q_{t+1}) - p_ref[k])^2 + w_R ||R(q_{t+1}) - R_ref||_F^2 )
 *        +                      sum_k w_p_final[k] (x_k(q_H) - p_ref[k])^2 + w_R_final ||R(q_H) - R_ref||_F^2.
 * Weights must be finite and non-negative, offset / p_ref / R_ref finite (RB_ERR_ARG otherwise).  The target is shared
 * by all trajectories and steps. */
typedef struct RbTipCost {
    const double* offset;     /* [3] tracked point in the tip frame (tool centre point); NULL = the tip frame's origin */
    const double* p_ref;      /* [3] its target in the base frame; NULL = 0 */
    const double* w_p;        /* [3] running weights per base-frame axis; NULL = 0 */
    const double* w_p_final;  /* [3] terminal weights per base-frame axis; NULL = 0 */
    const double* R_ref;      /* [9] row-major target orientation of the tip frame in the base frame; NULL = identity */
    double w_R;               /* running weight of ||R - R_ref||_F^2 */
    double w_R_final;         /* terminal weight of the same */
} RbTipCost;
/* multibody_rollout_cost with the tip terms of `tip` added.  weights == NULL: no quadratic terms; tip == NULL: exactly
 * multibody_rollout_cost (same results, same launches).  Every chain and kernel family multibody_rollout_cost serves. */
int multibody_rollout_tip_cost(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                               const RbQuadCost* weights, const RbTipCost* tip, double* cost, double* q_final, double* dq_final,
                               size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream);
/* multibody_rollout_cost_grad with the tip terms: cost bit-identical to multibody_rollout_tip_cost on the same engine, and
 * its gradient (the tip terms' part from one world-frame wrench per state projected on the joint screws, O(n) per state).
 * weights == NULL: no quadratic terms; tip == NULL: exactly multibody_rollout_cost_grad.  Serial chains of at most 12
 * joints (RB_ERR_UNSUPPORTED otherwise), everything else as multibody_rollout_cost_grad. */
int multibody_rollout_tip_cost_grad(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                    const RbQuadCost* weights, const RbTipCost* tip, double* cost, double* grad_tau,
                                    double* grad_q0, double* grad_dq0, size_t n_traj, size_t ld, RbLayout layout, RbMem mem,
                                    void* stream);

/* Pose of the tip frame (the frame of multibody_jac) and of a tracked point in it: 12 entries per state,
 * x = p + R offset (3) then R row-major (9).  SOA: pose[k*ld + s];  AOS: pose[12 s + k].  offset: host [3], NULL = 0
 * (finite, RB_ERR_ARG otherwise).  Every chain, tree and kernel family (one model-agnostic kernel: the same bits under
 * every family). */
int multibody_tip_pose_batch(RbGpu* g, const double* q, const double* offset, double* pose,
                             size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* Inverse kinematics of the tip frame: one damped least-squares (Levenberg-Marquardt) problem per entry, minimising the
 * per-state tip term of RbTipCost,
 *   F(q) = sum_k w_p[k] (x_k(q) - p*_k)^2 + w_R ||R(q) - R*||_F^2,   x = p + R offset.
 * With W = diag(sqrt(w_p), sqrt(2 w_R) 1_3), e = (p* - x ; omega), omega = 1/2 sum_k R[:,k] x R*[:,k], and J the base-frame
 * Jacobian of (x, orientation) (column j = (z_j x (x - P_j) ; z_j) for joints that support the tip, 0 otherwise), a step is
 *   delta = J^T W (W J J^T W + lambda I_6)^-1 W e     (a 6x6 LDL^T; a non-positive pivot counts as a rejected trial)
 * and the loop is
 *   q <- clamp(q_init); lambda <- damping; for k = 0, 1, ...:
 *     converged (pos_err <= tol_p and (w_R == 0 or rot_err <= tol_R)): iters = k, stop;   k == max_iters: iters = -1, stop;
 *     q' <- clamp(q + delta); if F(q') < F(q): q <- q', lambda <- max(lambda / 10, 1e-12); else lambda <- min(10 lambda, 1e12).
 * F never increases: the returned q is never worse than clamp(q_init). */
typedef struct RbIkOptions {
    const double* offset;   /* [3] tracked point in the tip frame (as RbTipCost); NULL = tip origin */
    const double* w_p;      /* [3] position weights per base axis; NULL = 1, 1, 1 */
    double w_R;             /* weight of ||R - R_target||_F^2; 0 = position only (R_target is not read, may be NULL) */
    const double* lower;    /* [n] joint bounds, +-inf allowed; NULL = unbounded */
    const double* upper;    /* [n] */
    int max_iters;          /* >= 0 */
    double tol_p;           /* position tolerance (m) */
    double tol_R;           /* rotation-angle tolerance (rad) */
    double damping;         /* initial Levenberg-Marquardt lambda, in [1e-12, 1e12] */
} RbIkOptions;

/* One damped least-squares problem per entry: q_init n per problem, p_target 3, R_target 9 (row-major).
 * out: n + 3 entries per problem: q, then the position error ||x - p*||_2 over the axes with w_p[k] > 0, the rotation angle
 * error 2 asin(min(1, ||R - R*||_F / sqrt 8)) (0 when w_R == 0), and the iterations taken (-1 = not converged).  A problem
 * with a non-finite q_init or target gets NaN in q and both errors and -1, and the call still succeeds.  RB_ERR_ARG for a
 * negative or non-finite weight, a NaN bound or lower > upper, max_iters < 0, a negative tolerance, damping outside
 * [1e-12, 1e12]; RB_ERR_NULL for opt == NULL or R_target == NULL with w_R > 0.  Layouts, ld, mem, stream and multi-device
 * slicing as every batched call.  Every chain, tree and kernel family (the same bits under every family).  Device calls
 * take a workspace of n doubles per thread of the launch in stream order on `stream` (cudaMallocAsync). */
int multibody_ik_batch(RbGpu* g, const double* q_init, const double* p_target, const double* R_target,
                       const RbIkOptions* opt, double* out, size_t n_problems, size_t ld, RbLayout layout,
                       RbMem mem, void* stream);

/* ---- link poses and collision-sphere cost terms (DESIGN.md 4.11) ---------------------------------
 * Link l is the child link of joint l; its frame is the joint frame of the descriptor / URDF (the engine re-bases a
 * joint whose axis is not +z internally; that rotation is undone here).  The tip frame of multibody_jac and
 * multibody_tip_pose_batch is link n-1's frame.
 *
 * Pose of every link: 12 entries per link per state, P_l (3) then R_l row-major (9), in the base frame.
 * SOA: pose[(12 l + m) ld + s];  AOS: pose[12 n s + 12 l + m].  Every chain, tree and kernel family (one model-agnostic
 * kernel: the same bits under every family). */
int multibody_link_poses_batch(RbGpu* g, const double* q, double* pose, size_t n_states, size_t ld, RbLayout layout,
                               RbMem mem, void* stream);

#define RB_MAX_SPHERES 256
#define RB_MAX_OBSTACLES 64
typedef enum RbObstacleKind { RB_OBSTACLE_SPHERE = 0, RB_OBSTACLE_HALFSPACE = 1 } RbObstacleKind;
/* Spheres fixed to the links and obstacles shared by all states.  Sphere k sits on link link[k] with centre c_k (in that
 * link's frame) and radius r_k >= 0; its world centre is x_k = P_l + R_l c_k.  Obstacle o is
 *   RB_OBSTACLE_SPHERE    (obstacle[4o..4o+3] = centre o, radius rho >= 0):  d_ko = ||x_k - o|| - r_k - rho,
 *   RB_OBSTACLE_HALFSPACE (obstacle[4o..4o+3] = normal n, offset h; n is normalised on load, the free side is
 *                          n.x >= h):                                    d_ko = n.x_k - h - r_k.
 * With margin m >= 0 the penalty of a pair is phi(d) = max(0, m - d)^2 (C^1), and Phi(q) = sum_k sum_o phi(d_ko).
 * A rollout cost gains  sum_{t=1}^{H} dt w Phi(q_t) + w_final Phi(q_H).
 * Gradient: dPhi/dq_j = s_j . sum_{l supported by j} w_l, s_j = (z_j ; P_j x z_j) the joint's world screw and
 * w_l = sum_{k on l} (x_k x g_k ; g_k) the link's world wrench, g_k = sum_o -2 max(0, m - d_ko) u_ko, where
 * u_ko = (x_k - o) / ||x_k - o|| (u = 0 when x_k = o exactly) or n for a half-space.
 * RB_ERR_NULL for a NULL array behind a non-zero count; RB_ERR_ARG for a count below 0 or above its cap, link outside
 * [0, n), a non-finite centre / obstacle entry, a negative radius, an unknown kind, a zero half-space normal, or a
 * negative or non-finite margin or weight. */
typedef struct RbCollisionCost {
    int32_t n_spheres;
    const int32_t* link;      /* [S] link of each sphere */
    const double* center;     /* [3S] centre in the link's frame */
    const double* radius;     /* [S] */
    int32_t n_obstacles;
    const int32_t* kind;      /* [O] RbObstacleKind */
    const double* obstacle;   /* [4O] (o, rho) or (n, h) */
    double margin;            /* m */
    double w;                 /* running weight */
    double w_final;           /* terminal weight */
} RbCollisionCost;

/* Per state: min_{k,o} d_ko, then Phi(q) (unweighted; w / w_final are checked but not used).  2 entries per state, SOA
 * out[m ld + s], AOS out[2 s + m].  At least one sphere and one obstacle (RB_ERR_ARG otherwise).  Every chain, tree and
 * kernel family. */
int multibody_sphere_distance_batch(RbGpu* g, const double* q, const RbCollisionCost* col, double* out, size_t n_states,
                                    size_t ld, RbLayout layout, RbMem mem, void* stream);
/* multibody_rollout_tip_cost with the collision terms of `col` added.  col == NULL, or one with no sphere, no obstacle or
 * w = w_final = 0: exactly multibody_rollout_tip_cost (same results, same launches).  Every chain and kernel family
 * multibody_rollout_tip_cost serves. */
int multibody_rollout_collision_cost(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                     const RbQuadCost* weights, const RbTipCost* tip, const RbCollisionCost* col, double* cost,
                                     double* q_final, double* dq_final, size_t n_traj, size_t ld, RbLayout layout, RbMem mem,
                                     void* stream);
/* multibody_rollout_tip_cost_grad with the collision terms: cost bit-identical to multibody_rollout_collision_cost on the
 * same engine, and its gradient (one world wrench per link per state projected on the joint screws, O(n + S O) per state).
 * col NULL or inactive: exactly multibody_rollout_tip_cost_grad.  Serial chains of at most 12 joints (RB_ERR_UNSUPPORTED
 * otherwise). */
int multibody_rollout_collision_cost_grad(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt,
                                          int horizon, const RbQuadCost* weights, const RbTipCost* tip,
                                          const RbCollisionCost* col, double* cost, double* grad_tau, double* grad_q0,
                                          double* grad_dq0, size_t n_traj, size_t ld, RbLayout layout, RbMem mem,
                                          void* stream);

/* ---- one MPPI iteration (DESIGN.md 4.12) ------------------------------------------------------
 * P = n_problems independent problems, each with its own start state (q0, dq0) and nominal torque sequence u_nom, all
 * sharing the cost terms (weights, tip, col: checked and selected as in multibody_rollout_collision_cost; weights == NULL
 * = no quadratic terms, a NULL or inactive tip / col = those terms off).  q0, dq0 are laid out like one state array and
 * u_nom, u_new like tau of a rollout with n_traj = P (layout and ld refer to P).  With K = n_samples, H = horizon:
 *   noise: sample s = p K + k (global over the batch), step t, joint i use the counter c = (s H + t) n + i and
 *     z = splitmix64(seed + 0x9E3779B97F4A7C15 (c + 1))   (the mixer of multibody_gpu_fill),
 *     u1 = ((z >> 32) + 0.5) 2^-32,  u2 = (z & 0xffffffff) 2^-32,  eps = sqrt(-2 ln u1) cospi(2 u2);
 *     sample 0 of every problem has eps = 0 (it is the nominal sequence);
 *   samples: tau_{p,k,t,i} = min(max(fma(sigma_i, eps, u_nom_{p,t,i}), lower_i), upper_i)  (a NaN passes through);
 *   cost: c_{p,k} = what multibody_rollout_collision_cost returns for (q0_p, dq0_p, tau_{p,k}, dt, H) with these terms, bit
 *     for bit on the same engine;
 *   weights: m_p = min over the finite c_{p,k};  w_{p,k} = exp((m_p - c_{p,k}) / lambda) for a finite cost, else 0;
 *     eta_p = sum_k w_{p,k};
 *   update: u_new_{p,t,i} = (sum_k w_{p,k} tau_{p,k,t,i}) / eta_p, the weighted mean of the clamped samples (within the
 *     bounds up to rounding).  A problem with no finite cost gets NaN in u_new and in its weights.
 * Optional outputs (each may be NULL): cost [P K] (sample k of problem p at p K + k), sample_weights [P K] = w / eta, and
 * samples = tau shaped like tau of a rollout with n_traj = P K (SOA dense [H][n][P K], leading dimension P K whatever ld
 * is; AOS [H][P K][n]).  A sample that meets a non-SPD mass matrix sets the status as the rollout cost does (RB_ERR_NOT_SPD
 * from host calls, the status word for device calls); its cost is NaN, its weight 0, and every output is still written.
 * horizon == 0: every sample costs the terminal cost of q0 and the weights are uniform; u_nom is not read and u_new is not
 * written.  RB_ERR_NULL for opt or sigma NULL, q0, dq0, u_nom or u_new NULL when H > 0, or q0 or dq0 NULL when H == 0 and
 * cost or sample_weights is asked for; RB_ERR_ARG for n_samples < 1,
 * a temperature that is not finite and > 0, a negative or non-finite sigma, a NaN bound or lower > upper, and whatever the
 * cost calls reject.  The results depend on the inputs and the seed only: not on layout, memory kind, chunking or a
 * multi-device handle (host calls slice the problems; a problem runs on one device), and every sum runs in an order fixed
 * by (P, K, H, n), without atomics.  Every chain, tree and kernel family multibody_rollout_cost serves.  Every call takes a
 * stream-ordered workspace on its stream of at most 1 GiB per chunk of whole problems, plus, when `samples` is given (the
 * rollout then reads it in place), the broadcast start states: 16 n bytes per sample.  It comes from a pool the engine owns,
 * which keeps up to 1 GiB of it between calls and gives that back when the engine is freed.  Host and AoS calls stage only
 * the arguments passed: without `samples`, nothing of size H n P K is staged. */
typedef struct RbMppiOptions {
    const double* sigma;      /* [n] noise standard deviation per joint, finite, >= 0 (required) */
    const double* lower;      /* [n] torque bounds, +-inf allowed; NULL = unbounded */
    const double* upper;      /* [n] */
    double temperature;       /* lambda > 0, finite */
    int32_t n_samples;        /* K >= 1 samples per problem */
    uint64_t seed;
} RbMppiOptions;
int multibody_mppi_step(RbGpu* g, const double* q0, const double* dq0, const double* u_nom, double dt, int horizon,
                        const RbQuadCost* weights, const RbTipCost* tip, const RbCollisionCost* col,
                        const RbMppiOptions* opt, double* u_new, double* cost, double* sample_weights, double* samples,
                        size_t n_problems, size_t ld, RbLayout layout, RbMem mem, void* stream);

/* ---- device-side helpers (bench / tests) --------------------------------------------------- */
/* Fill a device SOA array [n][ld] with the counter-based sampler of SURVEY.md 8d:
 * value(joint i, state s) = fma(hi[i]-lo[i], u, lo[i]),  u = top 53 bits of
 * splitmix64(seed + GOLDEN*(1 + (field<<58 | i<<50 | first_index+s))).  lo/hi are host arrays [n]. */
int multibody_gpu_fill(RbGpu* g, double* dev_out, uint64_t seed, uint32_t field, const double* lo, const double* hi,
                       size_t first_index, size_t count, size_t ld, void* stream);
/* Wait for all work on the engine's device, then report (and clear) the device-side status word:
 * RB_ERR_NOT_SPD if any forward-dynamics state since the last query met a non-SPD mass matrix. */
int multibody_gpu_sync(RbGpu* g);
int multibody_gpu_status(RbGpu* g);     /* alias of multibody_gpu_sync */
/* Kernel launches issued by this engine since creation (bench.py's `gpu_launches`). */
uint64_t multibody_gpu_launch_count(const RbGpu* g);
/* Pinned host allocations, so RB_MEM_HOST calls copy at full PCIe rate without a staging hop. */
int multibody_host_alloc(void** out, size_t bytes);
void multibody_host_free(void* p);
/* Bare ceiling of the host<->device path RB_MEM_HOST calls use: h2d_bytes from pinned host memory to the device and,
 * concurrently, d2h_bytes back (both split evenly over the devices of a multi-device engine, all devices at once), no
 * kernel in between; mean of `reps` passes by wall clock.  Returns GB/s per direction, summed over devices: what an
 * end-to-end call moving the same bytes cannot beat (bench.py reports e2e as a fraction of it). */
int multibody_gpu_measure_copy_peak(RbGpu* g, size_t h2d_bytes, size_t d2h_bytes, int reps, double* h2d_gbs, double* d2h_gbs);
/* Sustained FP64 FMA throughput of the device in TFLOP/s (2 flops per DFMA), measured with a register-only
 * dependent-chain kernel for `millis` ms: the FP64 roofline denominator bench.py reports against. */
int multibody_gpu_measure_fp64_peak(RbGpu* g, int millis, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* MULTIBODY_INTERFACE_H */
