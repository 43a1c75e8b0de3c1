// rb_deriv.cuh -- analytical first derivatives of inverse and forward dynamics (SURVEY.md 8f rank 4; the reference
// lists "Differentiability" as not done, README.md:18).
//
//   rb_rnea_derivatives:  d tau / d q  and  d tau / d dq  of  tau = rnea(q, dq, ddq)   (multibody.rs:111-153)
//   forward dynamics:     d qdd / d x = -H^-1 (d tau / d x at ddq = qdd),  d qdd / d tau = H^-1   (rb_kernels.cuh)
//
// Thread per state like the other kernels, but the algebra is done in the WORLD frame about the world origin, where
// the recursions of rnea / crba become sums along the chain and every partial derivative has a closed form.
// Spatial vectors are (angular ; linear-at-origin), forces (moment-about-origin ; force).  With the joint screws
// s_k = (z_k ; p_k x z_k), body velocities v_k = sum_{l<=k} s_l dq_l, accelerations a_k (base: (0 ; g)), world
// inertias I_k, momenta h_k = I_k v_k, wrenches f_k = I_k a_k + v_k x* h_k and the inertia rates
// Idot_k = v_k x* I_k - I_k v_k x (again a 10-parameter object: mass rate 0, first-moment rate, 6 inertia rates),
// all suffix-summed into composites (^c):
//
//   d/d dq_j:  dv = s_j                 da0 = 2 v_j x s_j
//   d/d  q_j:  dv = v_j x s_j           da0 = a_j x s_j + v_j x (v_j x s_j)
//   for both:  d f_k = [s_j x* f_k] + I_k da0 + Idot_k dv + dv x* h_k     (k >= j; bracket for d/dq only)
//   A_m = I^c_m s_m,  B_m = Idot^c_m s_m - s_m x* h^c_m,  G_j = sum_{k>=j} d f_k
//   d tau_m / d x_j = s_m . G_j             (m <= j)
//                   = da0_j . A_m + dv_j . B_m   (m > j)
//
// (the term from d s_m / d q_j cancels against s_j x* F^c_m).
// tests/ check it against complex-step differentiation of an independent link-frame rnea.
#pragma once
#include "rb_dyn.cuh"

RB_DI void rb_cross3(const double (&a)[3], const double (&b)[3], double (&o)[3]) {
    o[0] = fma(a[1], b[2], -(a[2] * b[1]));
    o[1] = fma(a[2], b[0], -(a[0] * b[2]));
    o[2] = fma(a[0], b[1], -(a[1] * b[0]));
}
RB_DI void rb_cross3_acc(const double (&a)[3], const double (&b)[3], double (&o)[3]) {
    o[0] = fma(a[1], b[2], fma(-a[2], b[1], o[0]));
    o[1] = fma(a[2], b[0], fma(-a[0], b[2], o[1]));
    o[2] = fma(a[0], b[1], fma(-a[1], b[0], o[2]));
}
// o = a x b for motion vectors:  (w1 x w2 ; w1 x v2 + v1 x w2)
RB_DI void rb_mcross(const double (&a)[6], const double (&b)[6], double (&o)[6]) {
    const double aw[3] = {a[0], a[1], a[2]}, av[3] = {a[3], a[4], a[5]};
    const double bw[3] = {b[0], b[1], b[2]}, bv[3] = {b[3], b[4], b[5]};
    double w[3], l[3];
    rb_cross3(aw, bw, w);
    rb_cross3(aw, bv, l);
    rb_cross3_acc(av, bw, l);
    o[0] = w[0]; o[1] = w[1]; o[2] = w[2]; o[3] = l[0]; o[4] = l[1]; o[5] = l[2];
}
// o (+)= a x* f for a motion a and a force f = (n ; f):  (w x n + v x f ; w x f)
template <bool ACC>
RB_DI void rb_fcross(const double (&a)[6], const double (&f)[6], double (&o)[6]) {
    const double aw[3] = {a[0], a[1], a[2]}, av[3] = {a[3], a[4], a[5]};
    const double fn[3] = {f[0], f[1], f[2]}, ff[3] = {f[3], f[4], f[5]};
    double n[3] = {ACC ? o[0] : 0.0, ACC ? o[1] : 0.0, ACC ? o[2] : 0.0};
    double l[3] = {ACC ? o[3] : 0.0, ACC ? o[4] : 0.0, ACC ? o[5] : 0.0};
    rb_cross3_acc(aw, fn, n);
    rb_cross3_acc(av, ff, n);
    rb_cross3_acc(aw, ff, l);
    o[0] = n[0]; o[1] = n[1]; o[2] = n[2]; o[3] = l[0]; o[4] = l[1]; o[5] = l[2];
}
// o (+)= I u for a 10-parameter inertia about the origin (mass m, first moment H, inertia S = xx xy xz yy yz zz):
//   n = S w + H x v,  f = m v - H x w.   The inertia RATE is the same object with m = 0.
template <bool ACC>
RB_DI void rb_wimul(double m, const double (&H)[3], const double (&S)[6], const double (&u)[6], double (&o)[6]) {
    const double w[3] = {u[0], u[1], u[2]}, v[3] = {u[3], u[4], u[5]};
    double n[3] = {ACC ? o[0] : 0.0, ACC ? o[1] : 0.0, ACC ? o[2] : 0.0};
    double f[3] = {ACC ? o[3] : 0.0, ACC ? o[4] : 0.0, ACC ? o[5] : 0.0};
    n[0] = fma(S[0], w[0], fma(S[1], w[1], fma(S[2], w[2], n[0])));
    n[1] = fma(S[1], w[0], fma(S[3], w[1], fma(S[4], w[2], n[1])));
    n[2] = fma(S[2], w[0], fma(S[4], w[1], fma(S[5], w[2], n[2])));
    rb_cross3_acc(H, v, n);
    f[0] = fma(m, v[0], f[0]); f[1] = fma(m, v[1], f[1]); f[2] = fma(m, v[2], f[2]);
    rb_cross3_acc(w, H, f);                                  // -H x w = w x H
    o[0] = n[0]; o[1] = n[1]; o[2] = n[2]; o[3] = f[0]; o[4] = f[1]; o[5] = f[2];
}
RB_DI double rb_dot6(const double (&a)[6], const double (&b)[6]) {
    return fma(a[0], b[0], fma(a[1], b[1], fma(a[2], b[2], fma(a[3], b[3], fma(a[4], b[4], a[5] * b[5])))));
}

// One link back along the chain: (R, P) of link i -> link i-1.  R <- R Rz(q_i)^T R_p^T,  P <- P - R t_i.
RB_DI void rb_pose_back(const RbJointK& J, double sn, double cs, double (&R)[3][3], double (&P)[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const double u0 = fma(cs, R[r][0], -(sn * R[r][1])), u1 = fma(sn, R[r][0], cs * R[r][1]), u2 = R[r][2];
        R[r][0] = fma(J.R[0], u0, fma(J.R[1], u1, J.R[2] * u2));
        R[r][1] = fma(J.R[3], u0, fma(J.R[4], u1, J.R[5] * u2));
        R[r][2] = fma(J.R[6], u0, fma(J.R[7], u1, J.R[8] * u2));
        P[r] = fma(-R[r][0], J.t[0], fma(-R[r][1], J.t[1], fma(-R[r][2], J.t[2], P[r])));
    }
}
// One link out: (R, P) of link i-1 -> link i.  P <- P + R t_i,  R <- R R_p Rz(q_i).
RB_DI void rb_pose_out(const RbJointK& J, double sn, double cs, double (&R)[3][3], double (&P)[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        P[r] = fma(R[r][0], J.t[0], fma(R[r][1], J.t[1], fma(R[r][2], J.t[2], P[r])));
        const double t0 = fma(R[r][0], J.R[0], fma(R[r][1], J.R[3], R[r][2] * J.R[6]));
        const double t1 = fma(R[r][0], J.R[1], fma(R[r][1], J.R[4], R[r][2] * J.R[7]));
        const double t2 = fma(R[r][0], J.R[2], fma(R[r][1], J.R[5], R[r][2] * J.R[8]));
        R[r][0] = fma(cs, t0, sn * t1);
        R[r][1] = fma(cs, t1, -(sn * t0));
        R[r][2] = t2;
    }
}
// Screw of the joint whose frame is (R, P), and the two d/dq column vectors of a body moving with (v, a):
//   s = (z ; P x z),  dv = v x s,  da0 = a x s + v x dv.
RB_DI void rb_screw_cols(const double (&R)[3][3], const double (&P)[3], const double (&v)[6], const double (&a)[6],
                         double (&s)[6], double (&dv)[6], double (&da)[6]) {
    const double z[3] = {R[0][2], R[1][2], R[2][2]};
    double pz[3];
    rb_cross3(P, z, pz);
    s[0] = z[0]; s[1] = z[1]; s[2] = z[2]; s[3] = pz[0]; s[4] = pz[1]; s[5] = pz[2];
    rb_mcross(v, s, dv);
    double t6[6];
    rb_mcross(a, s, da);
    rb_mcross(v, dv, t6);
#pragma unroll
    for (int k = 0; k < 6; ++k) da[k] += t6[k];
}

// ---- the two sweeps both routines below share
// Outward: world pose (R, P), velocity v and acceleration a of the last link; screw(i, s_i) sees every joint's screw.
template <int N, class Screw>
RB_DI void rb_deriv_outward(const RbModelK<N>& p, const double* sn, const double* cs, const double* dq, const double* ddq,
                            double (&R)[3][3], double (&P)[3], double (&v)[6], double (&a)[6], Screw&& screw) {
#pragma unroll 1
    for (int i = 0; i < N; ++i) {
        rb_pose_out(p.jt[i], sn[i], cs[i], R, P);
        const double z[3] = {R[0][2], R[1][2], R[2][2]};
        double pz[3], s6[6], dv[6];
        rb_cross3(P, z, pz);
        s6[0] = z[0]; s6[1] = z[1]; s6[2] = z[2]; s6[3] = pz[0]; s6[4] = pz[1]; s6[5] = pz[2];
        const double dqi = dq[i], ddqi = ddq[i];
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] = fma(s6[k], dqi, v[k]);
        rb_mcross(v, s6, dv);                                // v_i x s_i
#pragma unroll
        for (int k = 0; k < 6; ++k) a[k] = fma(s6[k], ddqi, fma(dv[k], dqi, a[k]));
        screw(i, s6);
    }
}

// Composites of links i..N-1 (^c above): inertia I^c (its mass is the model constant mc), inertia rate Idot^c,
// momentum h^c and wrench F^c, all about the world origin.
struct RbDerivComposites {
    double Hc[3], Ic[6], dHc[3], dIc[6], hc[6], Fc[6];
};

// Inward step at link i (pose R, P, velocity v, acceleration a): adds the link to the composites, then forms the
// per-joint vectors s_i, dv_i, da0_i (rb_screw_cols) and A_i, B_i, G_i, G'_i (the d/d dq counterpart of G_i).
RB_DI void rb_deriv_inward(const RbJointK& Jt, const double (&R)[3][3], const double (&P)[3], const double (&v)[6],
                           const double (&a)[6], RbDerivComposites& C, double (&sI)[6], double (&dvI)[6], double (&daI)[6],
                           double (&A)[6], double (&Bv)[6], double (&G)[6], double (&Gp)[6]) {
    {   // link i about the world origin
        const double m = Jt.m;
        double hw[3], T[3][3], Hm[3], IO[6];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            hw[r] = fma(R[r][0], Jt.h[0], fma(R[r][1], Jt.h[1], R[r][2] * Jt.h[2]));
            T[r][0] = fma(R[r][0], Jt.I[0], fma(R[r][1], Jt.I[1], R[r][2] * Jt.I[2]));
            T[r][1] = fma(R[r][0], Jt.I[1], fma(R[r][1], Jt.I[3], R[r][2] * Jt.I[4]));
            T[r][2] = fma(R[r][0], Jt.I[2], fma(R[r][1], Jt.I[4], R[r][2] * Jt.I[5]));
        }
        double u[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) { Hm[r] = fma(m, P[r], hw[r]); u[r] = fma(0.5 * m, P[r], hw[r]); }
        const double pu2 = 2.0 * fma(P[0], u[0], fma(P[1], u[1], P[2] * u[2]));
        auto rr = [&](int x, int y) { return fma(T[x][0], R[y][0], fma(T[x][1], R[y][1], T[x][2] * R[y][2])); };
        IO[0] = rr(0, 0) - 2.0 * P[0] * u[0] + pu2;
        IO[1] = rr(0, 1) - fma(P[0], u[1], u[0] * P[1]);
        IO[2] = rr(0, 2) - fma(P[0], u[2], u[0] * P[2]);
        IO[3] = rr(1, 1) - 2.0 * P[1] * u[1] + pu2;
        IO[4] = rr(1, 2) - fma(P[1], u[2], u[1] * P[2]);
        IO[5] = rr(2, 2) - 2.0 * P[2] * u[2] + pu2;
        // momentum, wrench, inertia rate of the link; accumulate the composites
        double h6[6], f6[6];
        rb_wimul<false>(m, Hm, IO, v, h6);
        rb_wimul<false>(m, Hm, IO, a, f6);
        rb_fcross<true>(v, h6, f6);
        const double w[3] = {v[0], v[1], v[2]}, vo[3] = {v[3], v[4], v[5]};
        double dH[3] = {m * vo[0], m * vo[1], m * vo[2]};
        rb_cross3_acc(w, Hm, dH);
        // d IO = [w]x IO + ([w]x IO)^T + 2 (H . vo) Id - vo H^T - H vo^T
        const double c0[3] = {IO[0], IO[1], IO[2]}, c1[3] = {IO[1], IO[3], IO[4]}, c2[3] = {IO[2], IO[4], IO[5]};
        double W0[3], W1[3], W2[3];                          // columns of [w]x IO
        rb_cross3(w, c0, W0); rb_cross3(w, c1, W1); rb_cross3(w, c2, W2);
        const double hv2 = 2.0 * fma(Hm[0], vo[0], fma(Hm[1], vo[1], Hm[2] * vo[2]));
        C.dIc[0] += 2.0 * W0[0] + hv2 - 2.0 * vo[0] * Hm[0];
        C.dIc[1] += W1[0] + W0[1] - fma(vo[0], Hm[1], Hm[0] * vo[1]);
        C.dIc[2] += W2[0] + W0[2] - fma(vo[0], Hm[2], Hm[0] * vo[2]);
        C.dIc[3] += 2.0 * W1[1] + hv2 - 2.0 * vo[1] * Hm[1];
        C.dIc[4] += W2[1] + W1[2] - fma(vo[1], Hm[2], Hm[1] * vo[2]);
        C.dIc[5] += 2.0 * W2[2] + hv2 - 2.0 * vo[2] * Hm[2];
#pragma unroll
        for (int k = 0; k < 3; ++k) { C.Hc[k] += Hm[k]; C.dHc[k] += dH[k]; }
#pragma unroll
        for (int k = 0; k < 6; ++k) { C.Ic[k] += IO[k]; C.hc[k] += h6[k]; C.Fc[k] += f6[k]; }
    }
    const double mc = Jt.mc;
    rb_screw_cols(R, P, v, a, sI, dvI, daI);
    double dv2[6], sh[6];
    rb_wimul<false>(mc, C.Hc, C.Ic, sI, A);
    rb_wimul<false>(0.0, C.dHc, C.dIc, sI, Bv);              // Idot^c s
    rb_fcross<false>(sI, C.hc, sh);                          // s x* h^c
#pragma unroll
    for (int k = 0; k < 6; ++k) { Gp[k] = Bv[k] + sh[k]; Bv[k] -= sh[k]; dv2[k] = 2.0 * dvI[k]; }
    rb_wimul<true>(mc, C.Hc, C.Ic, dv2, Gp);
    rb_fcross<false>(sI, C.Fc, G);
    rb_wimul<true>(mc, C.Hc, C.Ic, daI, G);
    rb_wimul<true>(0.0, C.dHc, C.dIc, dvI, G);
    rb_fcross<true>(dvI, C.hc, G);
}

// One link back along the chain for (R, P, v, a), leaving link i whose screw / dv are s / dv:
//   a <- a - s ddq_i - dv dq_i,  v <- v - s dq_i,  pose of link i -> link i-1.
RB_DI void rb_deriv_step_back(const RbJointK& Jt, double sn, double cs, double dqi, double ddqi, const double (&s)[6],
                              const double (&dv)[6], double (&R)[3][3], double (&P)[3], double (&v)[6], double (&a)[6]) {
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        a[k] = fma(-s[k], ddqi, fma(-dv[k], dqi, a[k]));
        v[k] = fma(-s[k], dqi, v[k]);
    }
    rb_pose_back(Jt, sn, cs, R, P);
}

// put(blk, r, c, v): blk 0 = d tau_r / d q_c, blk 1 = d tau_r / d dq_c.
// Real loops over the joints (model rows from the constant bank by index), and no per-joint arrays: a thread cannot
// hold N screws and column vectors next to the composites -- the first, fully unrolled version did and spilled 4 KB
// per thread through L2 to HBM (5x the algorithmic write traffic).  Instead, for every pair (i, j < i) the inward
// sweep walks a copy of (pose, v, a) back from link i to link j and rebuilds s_j, dv_j, da0_j there: ~160 FP64
// instructions per pair, all in registers.  sn, cs, dq, ddq are indexed at run time (thread-local memory, L1).
template <int N, class Put>
RB_DI void rb_rnea_derivatives(const RbModelK<N>& p, const double* sn, const double* cs, const double* dq, const double* ddq,
                               Put&& put) {
    double R[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}}, P[3] = {0.0, 0.0, 0.0};
    double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    double a[6] = {0.0, 0.0, 0.0, p.g[0], p.g[1], p.g[2]};
    rb_deriv_outward<N>(p, sn, cs, dq, ddq, R, P, v, a, [](int, const double (&)[6]) {});
    // ---- inward: composites, the per-joint vectors, and the entries
    RbDerivComposites C = {};
#pragma unroll 1
    for (int i = N - 1; i >= 0; --i) {
        double sI[6], dvI[6], daI[6], A[6], Bv[6], G[6], Gp[6];
        rb_deriv_inward(p.jt[i], R, P, v, a, C, sI, dvI, daI, A, Bv, G, Gp);
        put(0, i, i, rb_dot6(sI, G));
        put(1, i, i, rb_dot6(sI, Gp));
        // walk a copy back to every j < i:  column i above the diagonal, row i below it
        double Rt[3][3], Pt[3], vt[6], at[6];
#pragma unroll
        for (int r = 0; r < 3; ++r) { Pt[r] = P[r]; Rt[r][0] = R[r][0]; Rt[r][1] = R[r][1]; Rt[r][2] = R[r][2]; }
#pragma unroll
        for (int k = 0; k < 6; ++k) { vt[k] = v[k]; at[k] = a[k]; }
#pragma unroll 1
        for (int j = i - 1; j >= 0; --j) {                   // leaving link j+1, whose screw / dv are in sI / dvI
            rb_deriv_step_back(p.jt[j + 1], sn[j + 1], cs[j + 1], dq[j + 1], ddq[j + 1], sI, dvI, Rt, Pt, vt, at);
            rb_screw_cols(Rt, Pt, vt, at, sI, dvI, daI);
            put(0, j, i, rb_dot6(sI, G));
            put(1, j, i, rb_dot6(sI, Gp));
            put(0, i, j, rb_dot6(daI, A) + rb_dot6(dvI, Bv));
            put(1, i, j, fma(2.0, rb_dot6(dvI, A), rb_dot6(sI, Bv)));
            if (j == i - 1) {                                // the first step back is also the main state's
#pragma unroll
                for (int r = 0; r < 3; ++r) { P[r] = Pt[r]; R[r][0] = Rt[r][0]; R[r][1] = Rt[r][1]; R[r][2] = Rt[r][2]; }
#pragma unroll
                for (int k = 0; k < 6; ++k) { v[k] = vt[k]; a[k] = at[k]; }
            }
        }
    }
}

// ---- tip-pose cost terms (RbTipCost) of a state whose last link has the world pose (Rl, P)
// With R = Rl tip (the tip frame), x = P + R offset, e = x - p_ref, the terms a (running) and b (terminal) times
//   sum_k W_k e_k^2 + w ||R - R_ref||_F^2,   W = a w_p + b w_p_final,  w = a w_R + b w_R_final,
// change with joint j's angle at the rate s_j . (n ; f) for the joint's world screw s_j = (z_j ; P_j x z_j) and the world
// wrench (moment about the origin ; force)
//   f = 2 W e,   n = x x f + 2 w sum_k R_ref[:,k] x R[:,k]
// (dx = z_j x (x - P_j) dq_j,  dR = [z_j]x R dq_j,  ||R - R_ref||^2 = 6 - 2 tr(R_ref^T R)).  No Jacobian is formed.
RB_DI void rb_tip_wrench(const double (&Rl)[3][3], const double (&P)[3], const double* tip, const double* __restrict__ tw,
                         double a, double b, double (&w)[6]) {
    auto c = [&](int k) { return __ldg(tw + k); };
    double R[3][3], x[3], f[3], nm[3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k) R[r][k] = fma(Rl[r][2], tip[6 + k], fma(Rl[r][1], tip[3 + k], Rl[r][0] * tip[k]));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x[k] = fma(R[k][2], c(RB_TW_OFFSET + 2), fma(R[k][1], c(RB_TW_OFFSET + 1), fma(R[k][0], c(RB_TW_OFFSET), P[k])));
        const double W = fma(b, c(RB_TW_WPF + k), a * c(RB_TW_WP + k));
        f[k] = 2.0 * (W * (x[k] - c(RB_TW_PREF + k)));
    }
    rb_cross3(x, f, nm);
    const double wr2 = 2.0 * fma(b, c(RB_TW_WRF), a * c(RB_TW_WR));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double rr[3] = {c(RB_TW_RREF + k), c(RB_TW_RREF + 3 + k), c(RB_TW_RREF + 6 + k)}, rk[3] = {R[0][k], R[1][k], R[2][k]};
        double t[3];
        rb_cross3(rr, rk, t);
#pragma unroll
        for (int r = 0; r < 3; ++r) nm[r] = fma(wr2, t[r], nm[r]);
    }
    w[0] = nm[0]; w[1] = nm[1]; w[2] = nm[2]; w[3] = f[0]; w[4] = f[1]; w[5] = f[2];
}

// gq[j] += the derivative of those terms (a running, b terminal) at one state, one sweep out (pose of the last link) and
// one back (the screws).
template <int N>
RB_DI void rb_tip_grad(const RbModelK<N>& p, const double* sn, const double* cs, const double* tw, double a, double b, double* gq) {
    double R[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}}, P[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
    for (int i = 0; i < N; ++i) rb_pose_out(p.jt[i], sn[i], cs[i], R, P);
    double w[6];
    rb_tip_wrench(R, P, p.tip, tw, a, b, w);
#pragma unroll 1
    for (int i = N - 1; i >= 0; --i) {
        const double z[3] = {R[0][2], R[1][2], R[2][2]};
        double pz[3];
        rb_cross3(P, z, pz);
        gq[i] += fma(z[0], w[0], fma(z[1], w[1], fma(z[2], w[2], fma(pz[0], w[3], fma(pz[1], w[4], pz[2] * w[5])))));
        if (i > 0) rb_pose_back(p.jt[i], sn[i], cs[i], R, P);
    }
}

// ---- collision-sphere cost terms (RbCollisionCost) of link l at its world pose (R, P); col = the collision block
// W += a (x_k x g_k ; g_k) summed over the link's spheres, g_k = sum_o -2 max(0, m - d_ko) u_ko the gradient of the
// penalty in the sphere's world centre x_k (u = (x - o) / ||x - o||, 0 when x = o; n for a half-space).  Summed over the
// links a joint supports and dotted with its screw, this is dPhi/dq_j (the same wrench projection as rb_tip_wrench).
RB_DI void rb_col_wrench(const double (&R)[3][3], const double (&P)[3], const double* __restrict__ col, int l, double a,
                         double (&W)[6]) {
    auto c = [&](int k) { return __ldg(col + k); };
    const int b = (int)c(RB_CL_TAB + l), e = (int)c(RB_CL_TAB + l + 1), nos = (int)c(RB_CL_NOS), noh = (int)c(RB_CL_NOH);
    const double m = c(RB_CL_MARGIN);
#pragma unroll 1
    for (int k = b; k < e; ++k) {
        const double* sp = col + RB_CL_SPH + 4 * k;
        const double c0 = __ldg(sp), c1 = __ldg(sp + 1), c2 = __ldg(sp + 2), r = __ldg(sp + 3);
        double x[3], g[3] = {0.0, 0.0, 0.0};
#pragma unroll
        for (int i = 0; i < 3; ++i) x[i] = fma(R[i][2], c2, fma(R[i][1], c1, fma(R[i][0], c0, P[i])));
#pragma unroll 1
        for (int o = 0; o < nos; ++o) {
            const double* ob = col + RB_CL_OBS + 4 * o;
            const double d0 = x[0] - __ldg(ob), d1 = x[1] - __ldg(ob + 1), d2 = x[2] - __ldg(ob + 2);
            const double reach = r + __ldg(ob + 3) + m, dd = fma(d0, d0, fma(d1, d1, d2 * d2));
            if (dd < reach * reach && dd > 0.0) {
                const double nrm = sqrt(dd), f = -2.0 * (reach - nrm) / nrm;
                g[0] = fma(f, d0, g[0]); g[1] = fma(f, d1, g[1]); g[2] = fma(f, d2, g[2]);
            }
        }
#pragma unroll 1
        for (int o = nos; o < nos + noh; ++o) {
            const double* ob = col + RB_CL_OBS + 4 * o;
            const double n0 = __ldg(ob), n1 = __ldg(ob + 1), n2 = __ldg(ob + 2);
            const double pen = (m + __ldg(ob + 3) + r) - fma(n0, x[0], fma(n1, x[1], n2 * x[2]));
            if (pen > 0.0) {
                const double f = -2.0 * pen;
                g[0] = fma(f, n0, g[0]); g[1] = fma(f, n1, g[1]); g[2] = fma(f, n2, g[2]);
            }
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) g[i] *= a;
        double mo[3];
        rb_cross3(x, g, mo);
#pragma unroll
        for (int i = 0; i < 3; ++i) { W[i] += mo[i]; W[3 + i] += g[i]; }
    }
}

// gq[j] += the derivative of the tip-pose terms (rb_tip_grad's) and of a Phi(q) at one state: one sweep out, and one
// back that adds each link's collision wrench to a running wrench and projects it on the joint's screw.
template <int N>
RB_DI void rb_col_grad(const RbModelK<N>& p, const double* sn, const double* cs, const double* tw, const double* col, double a,
                       double b, double* gq) {
    double R[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}}, P[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
    for (int i = 0; i < N; ++i) rb_pose_out(p.jt[i], sn[i], cs[i], R, P);
    double w[6];
    rb_tip_wrench(R, P, p.tip, tw, a, b, w);
    const double wc = fma(b, __ldg(col + RB_CL_WF), a * __ldg(col + RB_CL_W));
#pragma unroll 1
    for (int i = N - 1; i >= 0; --i) {
        rb_col_wrench(R, P, col, i, wc, w);
        const double z[3] = {R[0][2], R[1][2], R[2][2]};
        double pz[3];
        rb_cross3(P, z, pz);
        gq[i] += fma(z[0], w[0], fma(z[1], w[1], fma(z[2], w[2], fma(pz[0], w[3], fma(pz[1], w[4], pz[2] * w[5])))));
        if (i > 0) rb_pose_back(p.jt[i], sn[i], cs[i], R, P);
    }
}

// Vector-Jacobian product of inverse dynamics in O(N), SUBTRACTED from gq and gdq (the adjoints a caller accumulates):
//   gq_j  -= (mu^T d tau / d q )_j = Sbar_j . G_j  +   da0_j . Abar_j + dv_j . Bbar_j
//   gdq_j -= (mu^T d tau / d dq)_j = Sbar_j . G'_j + 2 dv_j . Abar_j +  s_j . Bbar_j
//   Sbar_j = sum_{m <= j} mu_m s_m,   Abar_j = sum_{m > j} mu_m A_m,   Bbar_j = sum_{m > j} mu_m B_m
// (the pair formulas of the header above, summed over m).  The outward sweep adds up Sbar over all joints; the inward
// sweep carries Abar and Bbar and takes each joint's term out of Sbar after using it, so the pair walk-back of
// rb_rnea_derivatives becomes one step back per joint.  Like sn, cs, dq, ddq and mu, gq and gdq are indexed at run
// time (thread-local memory): a caller's adjoints do not occupy registers across the sweeps.
// TIP with tip_a != 0 also ADDS the running tip-pose terms' derivative (rb_tip_wrench, weight tip_a, row tw) at this
// state to gq: the wrench from the outward sweep's last-link pose, projected on each screw the inward sweep forms.
// COL (with TIP) adds the collision terms' derivative as well (weight tip_a times the block's running weight, block col):
// the inward sweep adds each link's collision wrench (rb_col_wrench, from the link pose it holds) to the tip wrench, and
// the running sum is what each screw is projected on.
template <int N, bool TIP = false, bool COL = false>
RB_DI void rb_rnea_vjp(const RbModelK<N>& p, const double* sn, const double* cs, const double* dq, const double* ddq,
                       const double* mu, double* gq, double* gdq, const double* tw = nullptr, double tip_a = 0.0,
                       const double* col = nullptr) {
    double R[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}}, P[3] = {0.0, 0.0, 0.0};
    double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    double a[6] = {0.0, 0.0, 0.0, p.g[0], p.g[1], p.g[2]};
    double Sb[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    rb_deriv_outward<N>(p, sn, cs, dq, ddq, R, P, v, a, [&](int i, const double (&s6)[6]) {
        const double mi = mu[i];
#pragma unroll
        for (int k = 0; k < 6; ++k) Sb[k] = fma(mi, s6[k], Sb[k]);
    });
    double wt[6];
    bool tip = false;
    if constexpr (TIP) {
        tip = tip_a != 0.0;
        if (tip) rb_tip_wrench(R, P, p.tip, tw, tip_a, 0.0, wt);
    }
    double wc = 0.0;
    if constexpr (COL) {
        wc = tip_a * __ldg(col + RB_CL_W);
        if (!tip) {
#pragma unroll
            for (int k = 0; k < 6; ++k) wt[k] = 0.0;
        }
    }
    RbDerivComposites C = {};
    double Ab[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, Bb[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
    for (int i = N - 1; i >= 0; --i) {
        double sI[6], dvI[6], daI[6], A[6], Bv[6], G[6], Gp[6];
        rb_deriv_inward(p.jt[i], R, P, v, a, C, sI, dvI, daI, A, Bv, G, Gp);
        gq[i] -= rb_dot6(Sb, G) + (rb_dot6(daI, Ab) + rb_dot6(dvI, Bb));
        if constexpr (COL) {
            if (wc != 0.0) rb_col_wrench(R, P, col, i, wc, wt);
            gq[i] += rb_dot6(sI, wt);
        } else if constexpr (TIP) { if (tip) gq[i] += rb_dot6(sI, wt); }
        gdq[i] -= rb_dot6(Sb, Gp) + fma(2.0, rb_dot6(dvI, Ab), rb_dot6(sI, Bb));
        const double mi = mu[i];
#pragma unroll
        for (int k = 0; k < 6; ++k) { Ab[k] = fma(mi, A[k], Ab[k]); Bb[k] = fma(mi, Bv[k], Bb[k]); Sb[k] = fma(-mi, sI[k], Sb[k]); }
        if (i > 0) rb_deriv_step_back(p.jt[i], sn[i], cs[i], dq[i], ddq[i], sI, dvI, R, P, v, a);
    }
}

// (the factor-once / solve-many split of the LDL^T, rb_ldlt_factor / rb_ldlt_apply, lives in rb_dyn.cuh)
