// rb_model.h -- flattened chain model shared by host code and kernels.
//
// One RbJointK per movable joint, in chain order.  It is what RevoluteJoint{parent, body}
// (reference rigidbody/src/joint.rs:26-31) reduces to once the quaternion isometry is a 3x3 matrix and
// the (mass, com, inertia_com, inertia) quadruple (inertia.rs:12-18) is the 10-parameter spatial inertia
// (m, h = m*com, I_o).  24 doubles = 192 B per joint; FR3 = 1.3 KB, a 32-joint chain = 6.1 KB: the whole
// model travels as a __grid_constant__ kernel parameter and is read from the constant bank.
#pragma once

#define RB_MAX_N 64

struct RbJointK {
    double R[9];   // parent_rot, row-major: child-frame vector -> parent-frame vector (before the joint rotation)
    double t[3];   // parent_trans
    double m;      // mass
    double mc;     // composite mass of the sub-tree rooted at link i (links i..n-1 of a serial chain): a model
                   // constant, CRBA's running mass (multibody.rs:170)
    double h[3];   // m * com
    double I[6];   // inertia about the link origin: xx xy xz yy yz zz   (inertia.rs:31-32)
    double parent; // index of the parent link, -1 = base (i-1 for the reference's serial chains); row = 24 doubles = 192 B
};

template <int N>
struct RbModelK {
    RbJointK jt[N];
    double g[3];   // base linear acceleration (reference: 0,0,+9.81; multibody.rs:118)
    double tip[9]; // row-major orientation of the reference's last link frame in the model's last frame: identity
                   // unless the last joint axis had to be re-based onto z (rb_host_model.cpp); read by jac only
};

#define RB_MODEL_TAIL 12                                   // doubles after the joint rows: g[3] + tip[9]
#define RB_MODEL_DOUBLES(n) ((n) * 24 + RB_MODEL_TAIL)

// Entry-class tags used by compile-time-specialised models to drop multiplications by 0 and +-1.
enum : int { RB_GEN = 0, RB_ZERO = 1, RB_ONE = 2, RB_NEG1 = 3 };

// Tip-pose cost terms of a rollout (RbTipCost in rigidbody.h), packed into one row of the engine's cost-weight block:
// tracked point in the tip frame, its target, running / terminal weights per base axis, target orientation (row-major),
// running / terminal orientation weights.
enum : int { RB_TW_OFFSET = 0, RB_TW_PREF = 3, RB_TW_WP = 6, RB_TW_WPF = 9, RB_TW_RREF = 12, RB_TW_WR = 21, RB_TW_WRF = 22, RB_TW_COUNT = 23 };

// Collision-sphere cost terms (RbCollisionCost in rigidbody.h), packed by the host into the block behind the cost-weight
// rows (doubles): margin, running / terminal weight, the numbers of sphere and half-space obstacles, per link l the first
// sphere index (entry l; entry n = the sphere count), the obstacles (4 each: sphere ones first, then half-spaces with
// unit normals), and the spheres grouped by link (4 each: centre in the link's engine frame, radius).
#define RB_CL_MAX_SPHERES 256    // RB_MAX_SPHERES
#define RB_CL_MAX_OBSTACLES 64   // RB_MAX_OBSTACLES
enum : int { RB_CL_MARGIN = 0, RB_CL_W = 1, RB_CL_WF = 2, RB_CL_NOS = 3, RB_CL_NOH = 4, RB_CL_TAB = 5,
             RB_CL_OBS = RB_CL_TAB + RB_MAX_N + 1, RB_CL_SPH = RB_CL_OBS + 4 * RB_CL_MAX_OBSTACLES,
             RB_CL_COUNT = RB_CL_SPH + 4 * RB_CL_MAX_SPHERES };

// Field selectors for the model policy accessors.
enum : int { RB_F_R = 0, RB_F_T = 1, RB_F_M = 2, RB_F_H = 3, RB_F_I = 4 };
