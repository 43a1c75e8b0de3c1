// rb_host_model.h -- host-side model loading: URDF / RbChainDesc -> flattened RbJointK rows.
//
// Mirrors what the reference does once at load time:
//   Multibody::from_urdf           rigidbody/src/multibody.rs:65-77   (zip k-th joint with k-th link, drop "fixed")
//   RevoluteJoint::from_xurdf_joint rigidbody/src/joint.rs:53-68      (axis, parent isometry, Inertia::from_com)
//   Inertia::from_com              rigidbody/src/inertia.rs:21-35     (I_o = I_c + m [c]x [c]x^T)
#pragma once
#include <string>
#include <vector>
#include "rb_model.h"
#include "../../include/rigidbody.h"

// One movable joint as the sources give it (URDF or RbChainDesc): axis and link inertia in the joint's own (child)
// frame -- field for field what the reference keeps in RevoluteJoint { axis, parent, body } (joint.rs:26-31) and
// Inertia { mass, com, inertia_com } (inertia.rs:12-17).
struct RbRawJoint {
    double axis[3]; double R[9]; double t[3]; double mass; double com[3]; double Ic[9]; int parent;
};

struct RbHostModel {
    int n = 0;
    std::vector<RbRawJoint> raw;             // the chain as loaded, before re-basing / flattening (multibody_get_chain)
    std::vector<RbJointK> jt;
    double g[3] = {0.0, 0.0, 9.81};          // multibody.rs:118
    double tip[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    // n x 9, row-major: link l's descriptor (URDF) frame seen from its re-based engine frame, Q_l^T; tip is link n-1's
    std::vector<double> link_rot;
    bool serial = true;                      // every joint hangs off the previous one (the reference's only case)
    RbJointLimits lim{};
    std::vector<std::string> names;
};

// Returns RB_OK or an RbStatus error with a message in `err`.
int rb_model_from_urdf(const char* path, RbHostModel& out, std::string& err);
int rb_model_from_desc(const RbChainDesc* d, RbHostModel& out, std::string& err);

// Emits a C++ header defining `struct <tab_name> { N, T[N][24], G[3] }` with exact (hex-float) constants:
// the compile-time table CtModel<> specialises the kernels on.
std::string rb_model_emit_header(const RbHostModel& m, const char* tab_name);

// Flattens the model into the layout of RbModelK<n> (n rows of 24 doubles, then g[3] and tip[9]).
std::vector<double> rb_model_flat(const RbHostModel& m);
