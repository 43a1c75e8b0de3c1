// rb_kernels_ik.cu -- batched tip pose and damped least-squares inverse kinematics of the tip frame
// (multibody_tip_pose_batch, multibody_ik_batch), link poses and sphere distances (multibody_link_poses_batch,
// multibody_sphere_distance_batch).  Model-agnostic: the kernels run the run-time-n loop kinematics of rb_dyn_n.cuh
// (rbn_tip_pose, rbn_link_walk) on the model rows in device memory, so every kernel family gives the same bits.
#include "rb_kernels.cuh"
#include "rb_dyn_n.cuh"
#include "rb_util.cuh"

namespace {

// Tracked point x = r + A off and the tip-frame Jacobian column of the joint whose frame (A, r) is expressed in:
// lin = A^T (z x x), rot = A^T z.
RB_DI void ik_column(const double (&A)[3][3], const double (&r)[3], const double* off, double (&c)[6]) {
    double x[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) x[k] = fma(A[k][2], off[2], fma(A[k][1], off[1], fma(A[k][0], off[0], r[k])));
#pragma unroll
    for (int k = 0; k < 3; ++k) { c[k] = fma(A[1][k], x[0], -(A[0][k] * x[1])); c[3 + k] = A[2][k]; }
}

// Packed upper triangle of a symmetric 6x6 matrix: entry (a, b), a <= b.
RB_DI constexpr int ik_sym(int a, int b) { return a <= b ? a * 6 - a * (a - 1) / 2 + (b - a) : b * 6 - b * (b - 1) / 2 + (a - b); }

// One walk of the tip frame at the joint values of `q` (strided view): the tip pose (R, x = p + R off) and
// M = sum_j c_j c_j^T of the tip-frame columns of the joints that support the tip.
RB_DI void ik_walk(const RbJointK* jt, const double* tip, int n, const double* off, const RbScratch& q, double (&M)[21],
                   double (&R)[3][3], double (&x)[3]) {
#pragma unroll
    for (int k = 0; k < 21; ++k) M[k] = 0.0;
    double r[3];
    rbn_tip_pose(jt, tip, n, [&](int i, double* sn, double* cs) { sincos(q[i], sn, cs); },
                 [&](int, const double (&A)[3][3], const double (&rr)[3]) {
                     double c[6];
                     ik_column(A, rr, off, c);
#pragma unroll
                     for (int a = 0; a < 6; ++a)
#pragma unroll
                         for (int b = a; b < 6; ++b) M[ik_sym(a, b)] = fma(c[a], c[b], M[ik_sym(a, b)]);
                 }, R, r);
#pragma unroll
    for (int k = 0; k < 3; ++k) x[k] = fma(R[k][2], off[2], fma(R[k][1], off[1], fma(R[k][0], off[0], r[k])));
}

RB_DI double ik_clamp(const RbIkParam& P, int i, double v) { return fmin(fmax(v, P.lower[i]), P.upper[i]); }

// F = sum_k w_p[k] (x_k - p*_k)^2 + w_R ||R - R*||_F^2;  also the squared position error over the weighted axes and
// ||R - R*||_F^2 (0 when w_R == 0: R* is not read).
RB_DI double ik_objective(const RbIkParam& P, const double (&R)[3][3], const double (&x)[3], const double (&pt)[3],
                          const double (&Rt)[9], double& pos2, double& rot2) {
    double F = 0.0;
    pos2 = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double e = x[k] - pt[k];
        F = fma(P.w_p[k] * e, e, F);
        if (P.w_p[k] > 0.0) pos2 = fma(e, e, pos2);
    }
    rot2 = 0.0;
    if (P.w_R > 0.0) {
#pragma unroll
        for (int k = 0; k < 9; ++k) { const double d = R[k / 3][k % 3] - Rt[k]; rot2 = fma(d, d, rot2); }
        F = fma(P.w_R, rot2, F);
    }
    return F;
}

}  // namespace

__global__ void __launch_bounds__(RB_BLOCK)
rbn_tip_pose_kernel(const double* __restrict__ model, int n, double o0, double o1, double o2, const double* __restrict__ q,
                    double* __restrict__ pose, size_t B, size_t ld) {
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    const double off[3] = {o0, o1, o2};
    double R[3][3], r[3];
    rbn_tip_pose(reinterpret_cast<const RbJointK*>(model), model + (size_t)n * 24 + 3, n,
                 [&](int i, double* sn, double* cs) { sincos(__ldcs(q + (size_t)i * ld + s), sn, cs); },
                 [](int, const double (&)[3][3], const double (&)[3]) {}, R, r);
#pragma unroll
    for (int k = 0; k < 3; ++k)
        __stcs(pose + (size_t)k * ld + s, fma(R[k][2], off[2], fma(R[k][1], off[1], fma(R[k][0], off[0], r[k]))));
#pragma unroll
    for (int k = 0; k < 9; ++k) __stcs(pose + (size_t)(3 + k) * ld + s, R[k / 3][k % 3]);
}

// Link l's descriptor frame: P_l, and R_l = R_engine,l Q_l^T (link_rot row l = Q_l^T, row-major).
__global__ void __launch_bounds__(RB_BLOCK)
rbn_link_poses_kernel(const double* __restrict__ model, const double* __restrict__ link_rot, int n, const double* __restrict__ q,
                      double* __restrict__ pose, size_t B, size_t ld) {
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    rbn_link_walk(reinterpret_cast<const RbJointK*>(model), n,
                  [&](int i, double* sn, double* cs) { sincos(__ldg(q + (size_t)i * ld + s), sn, cs); },
                  [&](int l, const double (&R)[3][3], const double (&P)[3]) {
                      double* o = pose + (size_t)(12 * l) * ld + s;
                      const double* Qt = link_rot + 9 * l;
#pragma unroll
                      for (int k = 0; k < 3; ++k) __stcs(o + (size_t)k * ld, P[k]);
#pragma unroll
                      for (int a = 0; a < 3; ++a)
#pragma unroll
                          for (int k = 0; k < 3; ++k)
                              __stcs(o + (size_t)(3 + 3 * a + k) * ld,
                                     fma(R[a][2], __ldg(Qt + 6 + k), fma(R[a][1], __ldg(Qt + 3 + k), R[a][0] * __ldg(Qt + k))));
                  });
}

// min_{k,o} d_ko and Phi(q) of the collision block col (RB_CL_* entries): every pair's distance, with the penalty formed
// as rb_col_link forms it.
__global__ void __launch_bounds__(RB_BLOCK)
rbn_sphere_distance_kernel(const double* __restrict__ model, int n, const double* __restrict__ col, const double* __restrict__ q,
                           double* __restrict__ out, size_t B, size_t ld) {
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    const int nos = (int)__ldg(col + RB_CL_NOS), noh = (int)__ldg(col + RB_CL_NOH);
    const double m = __ldg(col + RB_CL_MARGIN);
    double dmin = INFINITY, phi = 0.0;
    rbn_link_walk(reinterpret_cast<const RbJointK*>(model), n,
                  [&](int i, double* sn, double* cs) { sincos(__ldg(q + (size_t)i * ld + s), sn, cs); },
                  [&](int l, const double (&R)[3][3], const double (&P)[3]) {
                      const int b = (int)__ldg(col + RB_CL_TAB + l), e = (int)__ldg(col + RB_CL_TAB + l + 1);
                      for (int k = b; k < e; ++k) {
                          const double* sp = col + RB_CL_SPH + 4 * k;
                          const double c0 = __ldg(sp), c1 = __ldg(sp + 1), c2 = __ldg(sp + 2), r = __ldg(sp + 3);
                          double x[3];
#pragma unroll
                          for (int a = 0; a < 3; ++a) x[a] = fma(R[a][2], c2, fma(R[a][1], c1, fma(R[a][0], c0, P[a])));
                          for (int o = 0; o < nos + noh; ++o) {
                              const double* ob = col + RB_CL_OBS + 4 * o;
                              double d, pen;
                              if (o < nos) {
                                  const double d0 = x[0] - __ldg(ob), d1 = x[1] - __ldg(ob + 1), d2 = x[2] - __ldg(ob + 2);
                                  const double nrm = sqrt(fma(d0, d0, fma(d1, d1, d2 * d2)));
                                  d = nrm - r - __ldg(ob + 3);
                                  pen = (r + __ldg(ob + 3) + m) - nrm;
                              } else {
                                  const double h = fma(__ldg(ob), x[0], fma(__ldg(ob + 1), x[1], __ldg(ob + 2) * x[2]));
                                  d = h - __ldg(ob + 3) - r;
                                  pen = (m + __ldg(ob + 3) + r) - h;
                              }
                              dmin = fmin(dmin, d);
                              if (pen > 0.0) phi = fma(pen, pen, phi);
                          }
                      }
                  });
    __stcs(out + s, dmin);
    __stcs(out + ld + s, phi);
}

// One thread per problem, grid-stride.  q lives in the output rows, the trial q' in `ws` (n doubles per thread,
// [slot][thread]); the two views swap when a trial is accepted, so no copy is made until the end.  Per iteration:
//   the 6x6 system  A = W M_b W + lambda I  from M (tip-frame sum of c c^T at q, kept from the walk that reached q),
//   rotated to the base frame once;  rhs W e;  LDL^T;  z = W y, rotated back to the tip frame;
//   walk at q: delta_j = c_j . z, q'_j = clamp(q_j + delta_j) (the columns are not stored: this walk recomputes them);
//   trial walk at q': its pose gives F', and it accumulates M at q', which becomes the next iteration's when accepted.
__global__ void __launch_bounds__(RB_BLOCK)
rbn_ik_kernel(const double* __restrict__ model, int n, const __grid_constant__ RbIkParam P, const double* __restrict__ q_init,
              const double* __restrict__ p_target, const double* __restrict__ R_target, double* __restrict__ out,
              double* __restrict__ ws, size_t B, size_t ld) {
    const size_t tid = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * RB_BLOCK;
    const RbJointK* jt = reinterpret_cast<const RbJointK*>(model);
    const double* tip = model + (size_t)n * 24 + 3;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (size_t s = tid; s < B; s += nthr) {
        double pt[3], Rt[9];
        bool finite = true;
#pragma unroll
        for (int k = 0; k < 3; ++k) { pt[k] = p_target[(size_t)k * ld + s]; finite = finite && isfinite(pt[k]); }
#pragma unroll
        for (int k = 0; k < 9; ++k) { Rt[k] = P.w_R > 0.0 ? R_target[(size_t)k * ld + s] : 0.0; finite = finite && isfinite(Rt[k]); }
        RbScratch qc{out + s, ld}, qt{ws + tid, nthr};
        for (int i = 0; i < n; ++i) {
            const double v = q_init[(size_t)i * ld + s];
            finite = finite && isfinite(v);
            qc[i] = ik_clamp(P, i, v);
        }
        if (!finite) {
            for (int i = 0; i < n; ++i) qc[i] = nan;
            out[(size_t)n * ld + s] = nan; out[(size_t)(n + 1) * ld + s] = nan; out[(size_t)(n + 2) * ld + s] = -1.0;
            continue;
        }
        double M[21], R[3][3], x[3], pos2, rot2;
        ik_walk(jt, tip, n, P.offset, qc, M, R, x);
        double F = ik_objective(P, R, x, pt, Rt, pos2, rot2);
        double lambda = P.damping;
        int iters = -1;
        for (int k = 0;; ++k) {
            if (sqrt(pos2) <= P.tol_p && (P.w_R == 0.0 || 2.0 * asin(fmin(1.0, sqrt(rot2) * 0.35355339059327373)) <= P.tol_R)) { iters = k; break; }
            if (k == P.max_iters) break;
            // W M_b W + lambda I with M_b = blockdiag(R, R) M blockdiag(R, R)^T
            double Ab[21];
#pragma unroll
            for (int bi = 0; bi < 2; ++bi)
#pragma unroll
                for (int bj = bi; bj < 2; ++bj) {
                    double T[3][3];                          // R M_(bi,bj)
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            T[a][c] = fma(R[a][2], M[ik_sym(3 * bi + 2, 3 * bj + c)],
                                          fma(R[a][1], M[ik_sym(3 * bi + 1, 3 * bj + c)], R[a][0] * M[ik_sym(3 * bi, 3 * bj + c)]));
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int c = (bi == bj ? a : 0); c < 3; ++c) {
                            const int ra = 3 * bi + a, rc = 3 * bj + c;
                            const double v = fma(T[a][2], R[c][2], fma(T[a][1], R[c][1], T[a][0] * R[c][0]));
                            Ab[ik_sym(ra, rc)] = fma(P.sw[ra] * v, P.sw[rc], ra == rc ? lambda : 0.0);
                        }
                }
            // rhs W e, e = (p* - x ; omega), omega = 1/2 sum_k R[:,k] x R*[:,k]
            double y[6];
#pragma unroll
            for (int a = 0; a < 3; ++a) y[a] = P.sw[a] * (pt[a] - x[a]);
            double w[3] = {0.0, 0.0, 0.0};
            if (P.w_R > 0.0) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    w[0] = fma(R[1][c], Rt[6 + c], fma(-R[2][c], Rt[3 + c], w[0]));
                    w[1] = fma(R[2][c], Rt[c], fma(-R[0][c], Rt[6 + c], w[1]));
                    w[2] = fma(R[0][c], Rt[3 + c], fma(-R[1][c], Rt[c], w[2]));
                }
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) y[3 + a] = P.sw[3 + a] * (0.5 * w[a]);
            // LDL^T in place (L below the diagonal stored at ik_sym, D on it) and the solve A y = W e
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                double d = Ab[ik_sym(j, j)];
#pragma unroll
                for (int m = 0; m < j; ++m) d = fma(-Ab[ik_sym(j, m)] * Ab[ik_sym(j, m)], Ab[ik_sym(m, m)], d);
                ok = ok && d > 0.0;
                Ab[ik_sym(j, j)] = d;
#pragma unroll
                for (int i = j + 1; i < 6; ++i) {
                    double v = Ab[ik_sym(i, j)];
#pragma unroll
                    for (int m = 0; m < j; ++m) v = fma(-Ab[ik_sym(i, m)] * Ab[ik_sym(j, m)], Ab[ik_sym(m, m)], v);
                    Ab[ik_sym(i, j)] = v / d;
                }
            }
            if (!ok) { lambda = fmin(10.0 * lambda, 1e12); continue; }
#pragma unroll
            for (int i = 1; i < 6; ++i)
#pragma unroll
                for (int m = 0; m < i; ++m) y[i] = fma(-Ab[ik_sym(i, m)], y[m], y[i]);
#pragma unroll
            for (int i = 0; i < 6; ++i) y[i] /= Ab[ik_sym(i, i)];
#pragma unroll
            for (int i = 4; i >= 0; --i)
#pragma unroll
                for (int m = i + 1; m < 6; ++m) y[i] = fma(-Ab[ik_sym(m, i)], y[m], y[i]);
            // z = W y in the base frame, then in the tip frame (R^T per half)
            double z[6];
#pragma unroll
            for (int a = 0; a < 6; ++a) y[a] *= P.sw[a];
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    z[3 * h + c] = fma(R[2][c], y[3 * h + 2], fma(R[1][c], y[3 * h + 1], R[0][c] * y[3 * h]));
            // q' = clamp(q + J^T W y): joints off the tip's branch keep their value
            if (P.tree)
                for (int i = 0; i < n; ++i) qt[i] = qc[i];
            {
                double Rd[3][3], rd[3];
                rbn_tip_pose(jt, tip, n, [&](int i, double* sn, double* cs) { sincos(qc[i], sn, cs); },
                             [&](int i, const double (&A)[3][3], const double (&rr)[3]) {
                                 double c[6];
                                 ik_column(A, rr, P.offset, c);
                                 double d = 0.0;
#pragma unroll
                                 for (int a = 0; a < 6; ++a) d = fma(c[a], z[a], d);
                                 qt[i] = ik_clamp(P, i, qc[i] + d);
                             }, Rd, rd);
            }
            double Mn[21], Rn[3][3], xn[3], pos2n, rot2n;
            ik_walk(jt, tip, n, P.offset, qt, Mn, Rn, xn);
            const double Fn = ik_objective(P, Rn, xn, pt, Rt, pos2n, rot2n);
            if (Fn < F) {
                const RbScratch t = qc; qc = qt; qt = t;
#pragma unroll
                for (int a = 0; a < 21; ++a) M[a] = Mn[a];
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    x[a] = xn[a];
#pragma unroll
                    for (int c = 0; c < 3; ++c) R[a][c] = Rn[a][c];
                }
                F = Fn; pos2 = pos2n; rot2 = rot2n;
                lambda = fmax(0.1 * lambda, 1e-12);
            } else {
                lambda = fmin(10.0 * lambda, 1e12);
            }
        }
        if (qc.base != out + s)
            for (int i = 0; i < n; ++i) out[(size_t)i * ld + s] = qc[i];
        out[(size_t)n * ld + s] = sqrt(pos2);
        out[(size_t)(n + 1) * ld + s] = P.w_R > 0.0 ? 2.0 * asin(fmin(1.0, sqrt(rot2) * 0.35355339059327373)) : 0.0;
        out[(size_t)(n + 2) * ld + s] = (double)iters;
    }
}

cudaError_t rb_launch_tip_pose(const double* model, int n, const double* offset, const double* q, double* pose, size_t B,
                               size_t ld, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    rbn_tip_pose_kernel<<<(unsigned)((B + RB_BLOCK - 1) / RB_BLOCK), RB_BLOCK, 0, st>>>(model, n, offset[0], offset[1], offset[2], q, pose, B, ld);
    return cudaGetLastError();
}

cudaError_t rb_launch_link_poses(const double* model, const double* link_rot, int n, const double* q, double* pose, size_t B,
                                 size_t ld, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    rbn_link_poses_kernel<<<(unsigned)((B + RB_BLOCK - 1) / RB_BLOCK), RB_BLOCK, 0, st>>>(model, link_rot, n, q, pose, B, ld);
    return cudaGetLastError();
}

cudaError_t rb_launch_sphere_distance(const double* model, int n, const double* col, const double* q, double* out, size_t B,
                                      size_t ld, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    rbn_sphere_distance_kernel<<<(unsigned)((B + RB_BLOCK - 1) / RB_BLOCK), RB_BLOCK, 0, st>>>(model, n, col, q, out, B, ld);
    return cudaGetLastError();
}

cudaError_t rb_launch_ik(const double* model, int n, const RbIkParam& P, const double* q_init, const double* p_target,
                         const double* R_target, double* out, size_t B, size_t ld, int sm_count, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    const size_t want = (B + RB_BLOCK - 1) / RB_BLOCK, cap = (size_t)sm_count * 8;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    double* ws = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&ws, (size_t)n * grid * RB_BLOCK * sizeof(double), st);
    if (e != cudaSuccess) return e;
    rbn_ik_kernel<<<grid, RB_BLOCK, 0, st>>>(model, n, P, q_init, p_target, R_target, out, ws, B, ld);
    e = cudaGetLastError();
    const cudaError_t f = cudaFreeAsync(ws, st);
    return e != cudaSuccess ? e : f;
}
