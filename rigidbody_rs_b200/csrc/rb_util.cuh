// rb_util.cuh -- utility kernels of the engine (defined in rb_kernels_n.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "rb_model.h"

struct RbFillRange { double lo[RB_MAX_N]; double hi[RB_MAX_N]; };
#define RB_PEAK_INNER 64

cudaError_t rb_launch_fill(double* out, uint64_t seed, uint32_t field, int n, const RbFillRange& rg,
                           size_t first, size_t count, size_t ld, cudaStream_t st);
// `per_state` doubles per state: [B][per_state] <-> [per_state][ld]
cudaError_t rb_launch_aos_to_soa(const double* aos, double* soa, int per_state, size_t B, size_t ld, cudaStream_t st);
cudaError_t rb_launch_soa_to_aos(const double* soa, double* aos, int per_state, size_t B, size_t ld, cudaStream_t st);
cudaError_t rb_launch_fp64_peak(double* out, int blocks, int threads, int iters, cudaStream_t st);
// Batched LDL^T solve in shared-memory tiles (rb_kernels_n.cu): H packed upper [n(n+1)/2][hpk_states], rhs/x in qdd.
cudaError_t rb_launch_ldlt_tiles(int n, const double* hpk, size_t hpk_states, double* qdd, size_t cnt, size_t ld,
                                 int* status, cudaStream_t st);
// Forward dynamics of a chain of n <= 32 joints, one warp per state / one lane per joint (rb_kernels_warp.cu);
// `model` = device rows in the rb_model.h layout (n x 24 doubles, then g[3]).
cudaError_t rb_launch_warp_fd(const double* model, int n, const double* q, const double* dq, const double* tau,
                              double* qdd, size_t B, size_t ld, int* status, cudaStream_t st);
#ifndef RB_WARP_FD
#define RB_WARP_FD 1
#endif
// Analytical derivatives (rb_kernels_deriv.cu) of serial chains of n <= RB_DERIV_MAX_N joints; `flat_model` = HOST rows in
// the rb_model.h layout (passed on as a kernel parameter).  out: [2 n^2][ld] resp. [3 n^2][ld], see include/rigidbody.h.
#define RB_DERIV_MAX_N 12        // forward-dynamics derivatives
#define RB_RNEA_DERIV_MAX_N 32   // inverse-dynamics derivatives
cudaError_t rb_launch_rnea_deriv(int n, const double* flat_model, const double* q, const double* dq, const double* ddq,
                                 double* out, size_t B, size_t ld, cudaStream_t st);
cudaError_t rb_launch_fd_deriv(int n, const double* flat_model, const double* q, const double* dq, const double* tau,
                               double* out, size_t B, size_t ld, int* status, cudaStream_t st);
// Reverse-mode pass through a rollout (rb_kernels_deriv.cu, where the recursion is stated), serial chains of
// n <= RB_DERIV_MAX_N joints.  Device pointers; q0 / dq0 / tau / g_* / grad_* use the leading dimension `ld` of the
// launch, the stored trajectory its own.  cost_w != NULL selects the cost of that weight block, with the terms of
// `terms`, as the upstream gradient, and g_* are ignored; otherwise a NULL g_* is zero.  A NULL grad_* is not written.
struct RbAdjointArgs {
    const double *q0, *dq0, *tau;                        // [n][ld], [n][ld], [horizon][n][ld]
    const double *q_traj, *dq_traj; size_t ld_traj;      // [horizon][n][ld_traj]: the states after each step
    const double *g_q, *g_dq, *g_qf, *g_dqf;             // shaped like q_traj (with ld), q0
    const double* cost_w;
    double *grad_tau, *grad_q0, *grad_dq0;
    double dt; int horizon;
    RbCostTerms terms = RB_COST_QUAD;                    // with cost_w: the terms of the block, as for RbOps::rollout
};
cudaError_t rb_launch_rollout_adjoint(int n, const double* flat_model, const RbAdjointArgs& a, size_t B, size_t ld, int* status,
                                      cudaStream_t st);
// Tip pose and damped least-squares inverse kinematics of the tip frame (rb_kernels_ik.cu), any chain or tree;
// `model` = device rows in the rb_model.h layout.  Pose: [12][ld], x = p + R offset then R row-major.
struct RbIkParam {
    double offset[3];                  // tracked point in the tip frame
    double w_p[3], w_R;                // objective weights
    double sw[6];                      // diagonal of W: sqrt(w_p), sqrt(2 w_R) x 3
    double tol_p, tol_R, damping;
    double lower[RB_MAX_N], upper[RB_MAX_N];
    int max_iters;
    int tree;                          // 1 = some joints do not support the tip
};
cudaError_t rb_launch_tip_pose(const double* model, int n, const double* offset, const double* q, double* pose, size_t B,
                               size_t ld, cudaStream_t st);
// Pose of every link in its descriptor frame (rb_kernels_ik.cu): [12 n][ld], per link P then R row-major; link_rot = device
// [n][9] rotations Q_l^T taking each engine frame to the descriptor one.
cudaError_t rb_launch_link_poses(const double* model, const double* link_rot, int n, const double* q, double* pose, size_t B,
                                 size_t ld, cudaStream_t st);
// min d and Phi (rb_col_link) per state: [2][ld]; col = the device collision block (RB_CL_* entries).
cudaError_t rb_launch_sphere_distance(const double* model, int n, const double* col, const double* q, double* out, size_t B,
                                      size_t ld, cudaStream_t st);
// out: [n + 3][ld] = q, position error, rotation angle error, iterations (-1 = not converged).  Takes a stream-ordered
// workspace of n doubles per thread of the grid (cudaMallocAsync on st).
cudaError_t rb_launch_ik(const double* model, int n, const RbIkParam& P, const double* q_init, const double* p_target,
                         const double* R_target, double* out, size_t B, size_t ld, int sm_count, cudaStream_t st);
// One MPPI step (rb_kernels_mppi.cu, multibody_mppi_step), on a chunk of `cnt` problems of K samples each, device SoA.
struct RbMppiParam {
    double sigma[RB_MAX_N], lower[RB_MAX_N], upper[RB_MAX_N];
    uint64_t seed;
    size_t K;                          // samples per problem
    int n, H;
};
// Sampler: the start states q0s / dq0s [n][ldS] and tau [H][n][ldS] of sample j = p K + k of the chunk (column j), from
// q0 / dq0 [n][ld] and u_nom [H][n][ld] (column p); p_first = the global index of the chunk's first problem.
cudaError_t rb_launch_mppi_sample(const RbMppiParam& P, const double* q0, const double* dq0, const double* u_nom, size_t ld,
                                  size_t p_first, size_t cnt, double* tau, double* q0s, double* dq0s, size_t ldS, cudaStream_t st);
// Weights: from cost [cnt K], the unnormalised weights w [cnt K] and their sums eta [cnt]; sw [cnt K] = w / eta unless NULL.
cudaError_t rb_launch_mppi_weights(const double* cost, size_t K, double lambda, size_t cnt, double* w, double* eta, double* sw,
                                   cudaStream_t st);
// Update, two launches: u_new [rows][ld] (column p) = sum_k w tau / eta over tau [rows][ldS], rows = H n.  `part` holds
// cnt * rb_mppi_tiles(K) * rows doubles.
size_t rb_mppi_tiles(size_t K);
cudaError_t rb_launch_mppi_update(const double* tau, size_t ldS, size_t K, int rows, const double* w, const double* eta, size_t cnt,
                                  double* part, double* u_new, size_t ld, cudaStream_t st);
