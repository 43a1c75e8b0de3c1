// rb_dyn_n.cuh -- run-time-n variant of rb_dyn.cuh: any serial chain of 1..RB_MAX_N joints, and (rbn_tree_*)
// kinematic trees given by parent indices.
//
// Same algebra, same citations, but the joint loop is a real loop and per-link state (f_i, H) lives in a
// per-thread scratch slice of global memory laid out [slot][thread] so every access is coalesced.
// It serves chains the unrolled kernels are not instantiated for (e.g. the synthetic 32-joint chain of
// BASELINE.json configs[4]); the reference itself cannot represent them ([RevoluteJoint; 7],
// multibody.rs:32).
#pragma once
#include "rb_model.h"

#ifndef RB_DI
#define RB_DI __device__ __forceinline__
#endif

struct RbScratch {          // per-thread strided scratch: element k of this thread at base[k * stride]
    double* base;
    size_t stride;
    RB_DI double& operator[](int k) const { return base[(size_t)k * stride]; }
};

RB_DI void rbn_motion(const RbJointK& j, double s, double c, double (&lin)[3], double (&rot)[3]) {
    const double d0 = fma(j.t[2], rot[1], fma(-j.t[1], rot[2], lin[0]));
    const double d1 = fma(j.t[0], rot[2], fma(-j.t[2], rot[0], lin[1]));
    const double d2 = fma(j.t[1], rot[0], fma(-j.t[0], rot[1], lin[2]));
    const double y0 = fma(j.R[6], d2, fma(j.R[3], d1, j.R[0] * d0));
    const double y1 = fma(j.R[7], d2, fma(j.R[4], d1, j.R[1] * d0));
    const double y2 = fma(j.R[8], d2, fma(j.R[5], d1, j.R[2] * d0));
    const double w0 = fma(j.R[6], rot[2], fma(j.R[3], rot[1], j.R[0] * rot[0]));
    const double w1 = fma(j.R[7], rot[2], fma(j.R[4], rot[1], j.R[1] * rot[0]));
    const double w2 = fma(j.R[8], rot[2], fma(j.R[5], rot[1], j.R[2] * rot[0]));
    lin[0] = fma(c, y0, s * y1);  lin[1] = fma(c, y1, -(s * y0));  lin[2] = y2;
    rot[0] = fma(c, w0, s * w1);  rot[1] = fma(c, w1, -(s * w0));  rot[2] = w2;
}

RB_DI void rbn_force(const RbJointK& j, double s, double c, double (&lin)[3], double (&rot)[3]) {
    const double y0 = fma(c, lin[0], -(s * lin[1])), y1 = fma(s, lin[0], c * lin[1]), y2 = lin[2];
    const double w0 = fma(c, rot[0], -(s * rot[1])), w1 = fma(s, rot[0], c * rot[1]), w2 = rot[2];
    const double L0 = fma(j.R[2], y2, fma(j.R[1], y1, j.R[0] * y0));
    const double L1 = fma(j.R[5], y2, fma(j.R[4], y1, j.R[3] * y0));
    const double L2 = fma(j.R[8], y2, fma(j.R[7], y1, j.R[6] * y0));
    double r0 = fma(j.R[2], w2, fma(j.R[1], w1, j.R[0] * w0));
    double r1 = fma(j.R[5], w2, fma(j.R[4], w1, j.R[3] * w0));
    double r2 = fma(j.R[8], w2, fma(j.R[7], w1, j.R[6] * w0));
    r0 = fma(-j.t[2], L1, fma(j.t[1], L2, r0));
    r1 = fma(-j.t[0], L2, fma(j.t[2], L0, r1));
    r2 = fma(-j.t[1], L0, fma(j.t[0], L1, r2));
    lin[0] = L0; lin[1] = L1; lin[2] = L2;
    rot[0] = r0; rot[1] = r1; rot[2] = r2;
}

RB_DI void rbn_inertia_mul(const RbJointK& j, const double (&al)[3], const double (&ar)[3], double (&fl)[3], double (&fr)[3]) {
    fl[0] = fma(j.h[2], ar[1], fma(-j.h[1], ar[2], j.m * al[0]));
    fl[1] = fma(j.h[0], ar[2], fma(-j.h[2], ar[0], j.m * al[1]));
    fl[2] = fma(j.h[1], ar[0], fma(-j.h[0], ar[1], j.m * al[2]));
    fr[0] = fma(-j.h[2], al[1], fma(j.h[1], al[2], fma(j.I[2], ar[2], fma(j.I[1], ar[1], j.I[0] * ar[0]))));
    fr[1] = fma(-j.h[0], al[2], fma(j.h[2], al[0], fma(j.I[4], ar[2], fma(j.I[3], ar[1], j.I[1] * ar[0]))));
    fr[2] = fma(-j.h[1], al[0], fma(j.h[0], al[1], fma(j.I[5], ar[2], fma(j.I[4], ar[1], j.I[2] * ar[0]))));
}

// Scratch use: sc[0..n) sin, sc[n..2n) cos, sc[2n + 6i + k] f_i.   dq/ddq/tau are strided global views
// (element i at x[i*ld]).  ddq == nullptr means ddq = 0.  tau may alias nothing else.
// multibody.rs:111-153
RB_DI void rbn_rnea(const RbJointK* __restrict__ jt, const double* g, int n, const RbScratch& sc,
                    const double* dq, const double* ddq, size_t ld, const RbScratch& tau) {
    double vl[3] = {0.0, 0.0, 0.0}, vr[3] = {0.0, 0.0, 0.0};
    double al[3] = {g[0], g[1], g[2]}, ar[3] = {0.0, 0.0, 0.0};
    for (int i = 0; i < n; ++i) {
        const RbJointK& j = jt[i];
        const double s = sc[i], c = sc[n + i];
        const double dqi = dq[(size_t)i * ld];
        rbn_motion(j, s, c, vl, vr);
        vr[2] += dqi;
        rbn_motion(j, s, c, al, ar);
        if (ddq) ar[2] += ddq[(size_t)i * ld];
        al[0] = fma(vl[1], dqi, al[0]);
        al[1] = fma(-vl[0], dqi, al[1]);
        ar[0] = fma(vr[1], dqi, ar[0]);
        ar[1] = fma(-vr[0], dqi, ar[1]);
        double fl[3], fr[3], Il[3], Ir[3];
        rbn_inertia_mul(j, al, ar, fl, fr);
        rbn_inertia_mul(j, vl, vr, Il, Ir);
        fl[0] = fma(vr[1], Il[2], fma(-vr[2], Il[1], fl[0]));
        fl[1] = fma(vr[2], Il[0], fma(-vr[0], Il[2], fl[1]));
        fl[2] = fma(vr[0], Il[1], fma(-vr[1], Il[0], fl[2]));
        fr[0] = fma(vl[1], Il[2], fma(-vl[2], Il[1], fma(vr[1], Ir[2], fma(-vr[2], Ir[1], fr[0]))));
        fr[1] = fma(vl[2], Il[0], fma(-vl[0], Il[2], fma(vr[2], Ir[0], fma(-vr[0], Ir[2], fr[1]))));
        fr[2] = fma(vl[0], Il[1], fma(-vl[1], Il[0], fma(vr[0], Ir[1], fma(-vr[1], Ir[0], fr[2]))));
        const int o = 2 * n + 6 * i;
        sc[o + 0] = fl[0]; sc[o + 1] = fl[1]; sc[o + 2] = fl[2];
        sc[o + 3] = fr[0]; sc[o + 4] = fr[1]; sc[o + 5] = fr[2];
    }
    double cl[3] = {0.0, 0.0, 0.0}, cr[3] = {0.0, 0.0, 0.0};   // force handed down from link i+1
    for (int i = n - 1; i >= 0; --i) {
        const int o = 2 * n + 6 * i;
        double fl[3] = {sc[o + 0] + cl[0], sc[o + 1] + cl[1], sc[o + 2] + cl[2]};
        double fr[3] = {sc[o + 3] + cr[0], sc[o + 4] + cr[1], sc[o + 5] + cr[2]};
        tau[i] = fr[2];
        if (i > 0) {
            rbn_force(jt[i], sc[i], sc[n + i], fl, fr);
            cl[0] = fl[0]; cl[1] = fl[1]; cl[2] = fl[2];
            cr[0] = fr[0]; cr[1] = fr[1]; cr[2] = fr[2];
        }
    }
}

// multibody.rs:155-174.  H(j, i) for j <= i is written through the functor `put(j, i, value)`.
template <class Put>
RB_DI void rbn_crba(const RbJointK* __restrict__ jt, int n, const RbScratch& sc, Put&& put) {
    double h[3] = {jt[n - 1].h[0], jt[n - 1].h[1], jt[n - 1].h[2]};
    double Ixx = jt[n - 1].I[0], Ixy = jt[n - 1].I[1], Ixz = jt[n - 1].I[2];
    double Iyy = jt[n - 1].I[3], Iyz = jt[n - 1].I[4], Izz = jt[n - 1].I[5];
    for (int i = n - 1; i >= 0; --i) {
        put(i, i, Izz);
        double Fl[3] = {-h[1], h[0], 0.0}, Fr[3] = {Ixz, Iyz, Izz};
        for (int j = i - 1; j >= 0; --j) {
            rbn_force(jt[j + 1], sc[j + 1], sc[n + j + 1], Fl, Fr);
            put(j, i, Fr[2]);
        }
        if (i > 0) {
            const RbJointK& J = jt[i];
            const RbJointK& Pn = jt[i - 1];
            const double si = sc[i], ci = sc[n + i];
            const double g0 = fma(ci, h[0], -(si * h[1])), g1 = fma(si, h[0], ci * h[1]), g2 = h[2];
            const double cs = ci * si, s2 = cs + cs, c2 = fma(ci, ci, -(si * si));
            const double hm = 0.5 * (Ixx - Iyy), hp = 0.5 * (Ixx + Iyy);
            const double u_ = fma(hm, c2, -(Ixy * s2));
            const double A[3][3] = {{hp + u_, fma(hm, s2, Ixy * c2), fma(ci, Ixz, -(si * Iyz))},
                                    {0.0, hp - u_, fma(si, Ixz, ci * Iyz)},
                                    {0.0, 0.0, Izz}};
            auto As = [&](int r, int k) { return r <= k ? A[r][k] : A[k][r]; };
            const double q0 = fma(J.R[2], g2, fma(J.R[1], g1, J.R[0] * g0));
            const double q1 = fma(J.R[5], g2, fma(J.R[4], g1, J.R[3] * g0));
            const double q2 = fma(J.R[8], g2, fma(J.R[7], g1, J.R[6] * g0));
            double P[3][3], Jm[3][3];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    P[r][k] = fma(J.R[3 * r + 2], As(2, k), fma(J.R[3 * r + 1], As(1, k), J.R[3 * r] * As(0, k)));
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int k = r; k < 3; ++k)
                    Jm[r][k] = fma(P[r][2], J.R[3 * k + 2], fma(P[r][1], J.R[3 * k + 1], P[r][0] * J.R[3 * k]));
            const double hmc = 0.5 * J.mc;
            const double u0 = fma(J.t[0], hmc, q0), u1 = fma(J.t[1], hmc, q1), u2 = fma(J.t[2], hmc, q2);
            const double tu0 = J.t[0] * u0, tu1 = J.t[1] * u1, tu2 = J.t[2] * u2;
            Ixx = fma(2.0, tu1 + tu2, Jm[0][0]) + Pn.I[0];
            Iyy = fma(2.0, tu0 + tu2, Jm[1][1]) + Pn.I[3];
            Izz = fma(2.0, tu0 + tu1, Jm[2][2]) + Pn.I[5];
            Ixy = fma(-J.t[1], u0, fma(-J.t[0], u1, Jm[0][1])) + Pn.I[1];
            Ixz = fma(-J.t[2], u0, fma(-J.t[0], u2, Jm[0][2])) + Pn.I[2];
            Iyz = fma(-J.t[2], u1, fma(-J.t[1], u2, Jm[1][2])) + Pn.I[4];
            h[0] = fma(J.t[0], J.mc, q0) + Pn.h[0];
            h[1] = fma(J.t[1], J.mc, q1) + Pn.h[1];
            h[2] = fma(J.t[2], J.mc, q2) + Pn.h[2];
        }
    }
}

// ------------------------------------------------------------------ kinematic trees (parent[i] < i, -1 = base)
// The reference is serial-only (f[i-1], multibody.rs:148; ic[i-1], :170).  With a parent index per joint the same
// recursions run over a tree: motion comes from the parent link instead of link i-1, wrenches and composite
// inertias are accumulated into the parent, and H(j, i) is non-zero only when j supports i.
// Extra scratch: va[12 i + k] = (v.lin, v.rot, a.lin, a.rot) of link i, kept for its children.
RB_DI void rbn_tree_rnea(const RbJointK* __restrict__ jt, const double* g, int n, const RbScratch& sc, const RbScratch& va,
                         const double* dq, const double* ddq, size_t ld, const RbScratch& tau) {
    for (int i = 0; i < n; ++i) {
        const RbJointK& j = jt[i];
        const int p = (int)j.parent;
        double vl[3] = {0.0, 0.0, 0.0}, vr[3] = {0.0, 0.0, 0.0};
        double al[3] = {g[0], g[1], g[2]}, ar[3] = {0.0, 0.0, 0.0};
        if (p >= 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                vl[k] = va[12 * p + k]; vr[k] = va[12 * p + 3 + k]; al[k] = va[12 * p + 6 + k]; ar[k] = va[12 * p + 9 + k];
            }
        }
        const double s = sc[i], c = sc[n + i];
        const double dqi = dq[(size_t)i * ld];
        rbn_motion(j, s, c, vl, vr);
        vr[2] += dqi;
        rbn_motion(j, s, c, al, ar);
        if (ddq) ar[2] += ddq[(size_t)i * ld];
        al[0] = fma(vl[1], dqi, al[0]);
        al[1] = fma(-vl[0], dqi, al[1]);
        ar[0] = fma(vr[1], dqi, ar[0]);
        ar[1] = fma(-vr[0], dqi, ar[1]);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            va[12 * i + k] = vl[k]; va[12 * i + 3 + k] = vr[k]; va[12 * i + 6 + k] = al[k]; va[12 * i + 9 + k] = ar[k];
        }
        double fl[3], fr[3], Il[3], Ir[3];
        rbn_inertia_mul(j, al, ar, fl, fr);
        rbn_inertia_mul(j, vl, vr, Il, Ir);
        fl[0] = fma(vr[1], Il[2], fma(-vr[2], Il[1], fl[0]));
        fl[1] = fma(vr[2], Il[0], fma(-vr[0], Il[2], fl[1]));
        fl[2] = fma(vr[0], Il[1], fma(-vr[1], Il[0], fl[2]));
        fr[0] = fma(vl[1], Il[2], fma(-vl[2], Il[1], fma(vr[1], Ir[2], fma(-vr[2], Ir[1], fr[0]))));
        fr[1] = fma(vl[2], Il[0], fma(-vl[0], Il[2], fma(vr[2], Ir[0], fma(-vr[0], Ir[2], fr[1]))));
        fr[2] = fma(vl[0], Il[1], fma(-vl[1], Il[0], fma(vr[0], Ir[1], fma(-vr[1], Ir[0], fr[2]))));
        const int o = 2 * n + 6 * i;
        sc[o + 0] = fl[0]; sc[o + 1] = fl[1]; sc[o + 2] = fl[2];
        sc[o + 3] = fr[0]; sc[o + 4] = fr[1]; sc[o + 5] = fr[2];
    }
    for (int i = n - 1; i >= 0; --i) {
        const int o = 2 * n + 6 * i;
        double fl[3] = {sc[o + 0], sc[o + 1], sc[o + 2]};
        double fr[3] = {sc[o + 3], sc[o + 4], sc[o + 5]};
        tau[i] = fr[2];
        const int p = (int)jt[i].parent;
        if (p >= 0) {
            rbn_force(jt[i], sc[i], sc[n + i], fl, fr);
            const int op = 2 * n + 6 * p;
#pragma unroll
            for (int k = 0; k < 3; ++k) { sc[op + k] += fl[k]; sc[op + 3 + k] += fr[k]; }
        }
    }
}

// ci[9 i + k]: composite (h[3], Ixx Ixy Ixz Iyy Iyz Izz) of the sub-tree rooted at link i; the composite mass is the
// model constant jt[i].mc.  put(j, i, v) is called for EVERY pair j <= i (zeros where j does not support i).
template <class Put>
RB_DI void rbn_tree_crba(const RbJointK* __restrict__ jt, int n, const RbScratch& sc, const RbScratch& ci, Put&& put) {
    for (int i = 0; i < n; ++i) {
#pragma unroll
        for (int k = 0; k < 3; ++k) ci[9 * i + k] = jt[i].h[k];
#pragma unroll
        for (int k = 0; k < 6; ++k) ci[9 * i + 3 + k] = jt[i].I[k];
    }
    for (int i = n - 1; i >= 0; --i) {
        const double h[3] = {ci[9 * i], ci[9 * i + 1], ci[9 * i + 2]};
        const double Ixx = ci[9 * i + 3], Ixy = ci[9 * i + 4], Ixz = ci[9 * i + 5];
        const double Iyy = ci[9 * i + 6], Iyz = ci[9 * i + 7], Izz = ci[9 * i + 8];
        put(i, i, Izz);
        double Fl[3] = {-h[1], h[0], 0.0}, Fr[3] = {Ixz, Iyz, Izz};
        int cur = i, anc = (int)jt[i].parent;
        for (int j = i - 1; j >= 0; --j) {
            if (j == anc) {
                rbn_force(jt[cur], sc[cur], sc[n + cur], Fl, Fr);
                put(j, i, Fr[2]);
                cur = j; anc = (int)jt[j].parent;
            } else {
                put(j, i, 0.0);
            }
        }
        const int p = (int)jt[i].parent;
        if (p >= 0) {
            const RbJointK& J = jt[i];
            const double si = sc[i], cs_ = sc[n + i];
            const double g0 = fma(cs_, h[0], -(si * h[1])), g1 = fma(si, h[0], cs_ * h[1]), g2 = h[2];
            // A = Rz I Rz^T (full symmetric), then R_p A R_p^T
            const double A[3][3] = {{fma(cs_, fma(cs_, Ixx, -(si * Ixy)), -(si * fma(cs_, Ixy, -(si * Iyy)))),
                                     fma(si, fma(cs_, Ixx, -(si * Ixy)), cs_ * fma(cs_, Ixy, -(si * Iyy))),
                                     fma(cs_, Ixz, -(si * Iyz))},
                                    {0.0, fma(si, fma(si, Ixx, cs_ * Ixy), cs_ * fma(si, Ixy, cs_ * Iyy)), fma(si, Ixz, cs_ * Iyz)},
                                    {0.0, 0.0, Izz}};
            auto As = [&](int r, int k) { return r <= k ? A[r][k] : A[k][r]; };
            const double q0 = fma(J.R[2], g2, fma(J.R[1], g1, J.R[0] * g0));
            const double q1 = fma(J.R[5], g2, fma(J.R[4], g1, J.R[3] * g0));
            const double q2 = fma(J.R[8], g2, fma(J.R[7], g1, J.R[6] * g0));
            double P[3][3], Jm[3][3];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    P[r][k] = fma(J.R[3 * r + 2], As(2, k), fma(J.R[3 * r + 1], As(1, k), J.R[3 * r] * As(0, k)));
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int k = r; k < 3; ++k)
                    Jm[r][k] = fma(P[r][2], J.R[3 * k + 2], fma(P[r][1], J.R[3 * k + 1], P[r][0] * J.R[3 * k]));
            const double hmc = 0.5 * J.mc;
            const double u0 = fma(J.t[0], hmc, q0), u1 = fma(J.t[1], hmc, q1), u2 = fma(J.t[2], hmc, q2);
            const double tu0 = J.t[0] * u0, tu1 = J.t[1] * u1, tu2 = J.t[2] * u2;
            ci[9 * p + 3] += fma(2.0, tu1 + tu2, Jm[0][0]);
            ci[9 * p + 6] += fma(2.0, tu0 + tu2, Jm[1][1]);
            ci[9 * p + 8] += fma(2.0, tu0 + tu1, Jm[2][2]);
            ci[9 * p + 4] += fma(-J.t[1], u0, fma(-J.t[0], u1, Jm[0][1]));
            ci[9 * p + 5] += fma(-J.t[2], u0, fma(-J.t[0], u2, Jm[0][2]));
            ci[9 * p + 7] += fma(-J.t[2], u1, fma(-J.t[1], u2, Jm[1][2]));
            ci[9 * p + 0] += fma(J.t[0], J.mc, q0);
            ci[9 * p + 1] += fma(J.t[1], J.mc, q1);
            ci[9 * p + 2] += fma(J.t[2], J.mc, q2);
        }
    }
}

// In-place LDL^T solve on a strided upper triangle: A(j,i), j <= i, at Hs[j*n + i]; x strided.
RB_DI bool rbn_ldlt_solve(int n, const RbScratch& Hs, const RbScratch& x, const RbScratch& dinv) {
    bool ok = true;
    for (int j = 0; j < n; ++j) {
        const double d = Hs[j * n + j];
        ok = ok && (d > 0.0);
        const double di = 1.0 / d;
        dinv[j] = di;
        for (int i = j + 1; i < n; ++i) {
            const double l = Hs[j * n + i] * di;
            for (int k = i; k < n; ++k) Hs[i * n + k] = fma(-l, Hs[j * n + k], Hs[i * n + k]);
            Hs[j * n + i] = l;
        }
    }
    for (int j = 0; j < n; ++j) {
        const double xj = x[j];
        for (int i = j + 1; i < n; ++i) x[i] = fma(-Hs[j * n + i], xj, x[i]);
    }
    for (int j = 0; j < n; ++j) x[j] = x[j] * dinv[j];
    for (int i = n - 1; i >= 0; --i) {
        double xi = x[i];
        for (int k = i + 1; k < n; ++k) xi = fma(-Hs[i * n + k], x[k], xi);
        x[i] = xi;
    }
    return ok;
}

// Tip frame in the base frame (rb_tip_pose with run-time n): A <- R_p Rz(q_i) A, r <- R_p Rz(q_i) r + t_i from the last
// link down its supporting branch, starting from A = the model's tip rotation `tip` and r = 0.  sincos(i, &s, &c) gives
// joint i's sin/cos; col(i, A, r) sees the pose of the tip in frame i before joint i's step (the Jacobian's column i).
template <class SinCos, class Col>
RB_DI void rbn_tip_pose(const RbJointK* jt, const double* tip, int n, SinCos&& sincos_i, Col&& col, double (&A)[3][3],
                        double (&r)[3]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { A[k][0] = tip[3 * k]; A[k][1] = tip[3 * k + 1]; A[k][2] = tip[3 * k + 2]; r[k] = 0.0; }
    for (int i = n - 1; i >= 0; i = (int)jt[i].parent) {
        const RbJointK& j = jt[i];
        col(i, A, r);
        double sn, cs;
        sincos_i(i, &sn, &cs);
        double Bm[3][3], y[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            Bm[0][k] = fma(cs, A[0][k], -(sn * A[1][k]));
            Bm[1][k] = fma(sn, A[0][k], cs * A[1][k]);
            Bm[2][k] = A[2][k];
        }
        y[0] = fma(cs, r[0], -(sn * r[1])); y[1] = fma(sn, r[0], cs * r[1]); y[2] = r[2];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int k = 0; k < 3; ++k)
                A[a][k] = fma(j.R[3 * a + 2], Bm[2][k], fma(j.R[3 * a + 1], Bm[1][k], j.R[3 * a] * Bm[0][k]));
            r[a] = fma(j.R[3 * a + 2], y[2], fma(j.R[3 * a + 1], y[1], fma(j.R[3 * a], y[0], j.t[a])));
        }
    }
}
