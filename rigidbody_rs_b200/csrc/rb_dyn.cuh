// rb_dyn.cuh -- device-side rigid-body algebra, one thread per state, everything in registers.
//
// What is computed follows the reference line by line (citations relative to the reference checkout);
// how it is computed does not: rotations are 3x3 (R_i = R_p * Rz(q_i)) instead of unit quaternions,
// inertias are the 10-parameter (m, h, I_o) form, the joint loop is unrolled at compile time through a
// model *policy* M so that a model known at compile time (CtModel) drops every multiplication by an
// exact 0 or +-1 of its fixed transforms, while a model known only at run time (RtModel) reads the same
// numbers from the kernel-parameter constant bank.  All arithmetic is fp64 (Real = f64, lib.rs:15).
#pragma once
#include "rb_model.h"

#define RB_DI __device__ __forceinline__
#ifndef RB_BATCHED_SINCOS
#define RB_BATCHED_SINCOS 2      // branch-free, interleavable sin/cos of all joints of a state (rb_sincos_batched): 0 = off, 2 = every kernel
                                 // (RNEA +2.7 %, FD +4 %, rollout +6..14 % against per-joint sincos(): profiles/r2_kbench_rollout.jsonl)
#endif
// Scalar type of the model policy in scope (every function below is templated on a policy M or on a scalar T).
#define RB_R typename M::Real

template <int V> struct RbIC { static constexpr int value = V; };

// f(RbIC<I>) for I = 0..N-1 (ascending) / N-1..0 (descending), fully unrolled.
template <int I, int N, class F> RB_DI void rb_for_up(F&& f) {
    if constexpr (I < N) { f(RbIC<I>{}); rb_for_up<I + 1, N>(f); }
}
template <int I, class F> RB_DI void rb_for_down(F&& f) {
    if constexpr (I >= 0) { f(RbIC<I>{}); rb_for_down<I - 1>(f); }
}

// ------------------------------------------------------------------ class-tagged scalar ops
template <int C, class T> RB_DI T k_mul(T k, T x) {
    if constexpr (C == RB_ZERO) return T(0);
    else if constexpr (C == RB_ONE) return x;
    else if constexpr (C == RB_NEG1) return -x;
    else return k * x;
}
template <int C, class T> RB_DI T k_fma(T k, T x, T acc) {        // acc + k*x
    if constexpr (C == RB_ZERO) return acc;
    else if constexpr (C == RB_ONE) return acc + x;
    else if constexpr (C == RB_NEG1) return acc - x;
    else return fma(k, x, acc);
}
template <int C, class T> RB_DI T k_fnma(T k, T x, T acc) {       // acc - k*x
    if constexpr (C == RB_ZERO) return acc;
    else if constexpr (C == RB_ONE) return acc - x;
    else if constexpr (C == RB_NEG1) return acc + x;
    else return fma(-k, x, acc);
}
template <int C0, int C1, int C2, class T>
RB_DI T k_dot3(T k0, T k1, T k2, T x0, T x1, T x2) {
    if constexpr (C0 != RB_ZERO) return k_fma<C2>(k2, x2, k_fma<C1>(k1, x1, k_mul<C0>(k0, x0)));
    else if constexpr (C1 != RB_ZERO) return k_fma<C2>(k2, x2, k_mul<C1>(k1, x1));
    else return k_mul<C2>(k2, x2);
}
template <int C0, int C1, int C2, class T>
RB_DI T k_dot3_acc(T acc, T k0, T k1, T k2, T x0, T x1, T x2) {
    return k_fma<C2>(k2, x2, k_fma<C1>(k1, x1, k_fma<C0>(k0, x0, acc)));
}

// ------------------------------------------------------------------ model policies
// Run-time model: values from the kernel parameter (constant bank), nothing known at compile time.
// Real is the scalar the kernels compute in (the parameter block always holds doubles).
template <int N_, class Real_ = double>
struct RtModel {
    static constexpr int N = N_;
    static constexpr bool kSpecialised = false;
    using Real = Real_;
    using Param = RbModelK<N_>;
    template <int I, int F, int K> static constexpr int cls() { return RB_GEN; }
    template <int I, int F, int K> static RB_DI Real val(const Param& p) {
        if constexpr (F == RB_F_R) return (Real)p.jt[I].R[K];
        else if constexpr (F == RB_F_T) return (Real)p.jt[I].t[K];
        else if constexpr (F == RB_F_M) return (Real)(K == 0 ? p.jt[I].m : p.jt[I].mc);
        else if constexpr (F == RB_F_H) return (Real)p.jt[I].h[K];
        else return (Real)p.jt[I].I[K];
    }
    template <int K> static constexpr int gcls() { return RB_GEN; }
    template <int K> static RB_DI Real g(const Param& p) { return (Real)p.g[K]; }
    template <int K> static RB_DI Real tip(const Param& p) { return (Real)p.tip[K]; }
    template <int K> static constexpr int tipcls() { return RB_GEN; }
    static constexpr bool kTree = false;     // run-time constants: serial chains only
    template <int I> static constexpr int parent() { return I - 1; }
};

// Compile-time model: Tab supplies `static constexpr int N; static constexpr double T[N][24]; G[3]`
// with each row laid out exactly like RbJointK (R9 t3 m mc h3 I6 + pad).  Real as above: the table is double,
// the constants are rounded to Real at compile time.
struct RbEmptyParam { int unused; };
constexpr int rb_classify(double v) { return v == 0.0 ? RB_ZERO : (v == 1.0 ? RB_ONE : (v == -1.0 ? RB_NEG1 : RB_GEN)); }
template <class Tab, class Real_ = double>
struct CtModel {
    static constexpr int N = Tab::N;
    static constexpr bool kSpecialised = true;
    using Real = Real_;
    using Param = RbEmptyParam;
    template <int F, int K> static constexpr int off() {
        return F == RB_F_R ? K : F == RB_F_T ? 9 + K : F == RB_F_M ? 12 + K : F == RB_F_H ? 14 + K : 17 + K;
    }
    template <int I, int F, int K> static constexpr int cls() { return rb_classify(Tab::T[I][off<F, K>()]); }
    template <int I, int F, int K> static RB_DI Real val(const Param&) {
        constexpr Real v = (Real)Tab::T[I][off<F, K>()];
        return v;
    }
    template <int K> static constexpr int gcls() { return rb_classify(Tab::G[K]); }
    template <int K> static RB_DI Real g(const Param&) { constexpr Real v = (Real)Tab::G[K]; return v; }
    template <int K> static RB_DI Real tip(const Param&) { constexpr Real v = (Real)Tab::TIP[K]; return v; }
    template <int K> static constexpr int tipcls() { return rb_classify(Tab::TIP[K]); }
    // parent link of joint I (slot 23 of the row); a table whose joints do not all hang off their predecessor is a
    // kinematic tree and takes the rb_*_tree forms (rb_dyn_tree.cuh)
    template <int I> static constexpr int parent() { return (int)Tab::T[I][23]; }
    static constexpr bool tree_() {
        for (int i = 0; i < Tab::N; ++i)
            if ((int)Tab::T[i][23] != i - 1) return true;
        return false;
    }
    static constexpr bool kTree = tree_();
};

#define KV(I, F, K) M::template val<I, F, K>(p)
#define KC(I, F, K) M::template cls<I, F, K>()

// ------------------------------------------------------------------ spatial transforms
// Motion vector parent -> child across joint I (spatial.rs:110-116 applied with X_I = parent o Rz(q)):
//   rot' = E rot, lin' = E (lin - t x rot), E = Rz(q)^T R_p^T.
template <class M, int I>
RB_DI void rb_motion(const typename M::Param& p, RB_R s, RB_R c, RB_R (&lin)[3], RB_R (&rot)[3]) {
    const RB_R t0 = KV(I, RB_F_T, 0), t1 = KV(I, RB_F_T, 1), t2 = KV(I, RB_F_T, 2);
    const RB_R d0 = k_fma<KC(I, RB_F_T, 2)>(t2, rot[1], k_fnma<KC(I, RB_F_T, 1)>(t1, rot[2], lin[0]));
    const RB_R d1 = k_fma<KC(I, RB_F_T, 0)>(t0, rot[2], k_fnma<KC(I, RB_F_T, 2)>(t2, rot[0], lin[1]));
    const RB_R d2 = k_fma<KC(I, RB_F_T, 1)>(t1, rot[0], k_fnma<KC(I, RB_F_T, 0)>(t0, rot[1], lin[2]));
    // y = R_p^T x : y_j = sum_k R[k][j] x_k
    const RB_R y0 = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 3), KC(I, RB_F_R, 6)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 3), KV(I, RB_F_R, 6), d0, d1, d2);
    const RB_R y1 = k_dot3<KC(I, RB_F_R, 1), KC(I, RB_F_R, 4), KC(I, RB_F_R, 7)>(KV(I, RB_F_R, 1), KV(I, RB_F_R, 4), KV(I, RB_F_R, 7), d0, d1, d2);
    const RB_R y2 = k_dot3<KC(I, RB_F_R, 2), KC(I, RB_F_R, 5), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 2), KV(I, RB_F_R, 5), KV(I, RB_F_R, 8), d0, d1, d2);
    const RB_R w0 = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 3), KC(I, RB_F_R, 6)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 3), KV(I, RB_F_R, 6), rot[0], rot[1], rot[2]);
    const RB_R w1 = k_dot3<KC(I, RB_F_R, 1), KC(I, RB_F_R, 4), KC(I, RB_F_R, 7)>(KV(I, RB_F_R, 1), KV(I, RB_F_R, 4), KV(I, RB_F_R, 7), rot[0], rot[1], rot[2]);
    const RB_R w2 = k_dot3<KC(I, RB_F_R, 2), KC(I, RB_F_R, 5), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 2), KV(I, RB_F_R, 5), KV(I, RB_F_R, 8), rot[0], rot[1], rot[2]);
    // Rz(q)^T
    lin[0] = fma(c, y0, s * y1);  lin[1] = fma(c, y1, -(s * y0));  lin[2] = y2;
    rot[0] = fma(c, w0, s * w1);  rot[1] = fma(c, w1, -(s * w0));  rot[2] = w2;
}

// Force child -> parent across joint I (spatial.rs:242-248 applied to X_I^-1, as multibody.rs:147,165 do):
//   lin' = R lin, rot' = R rot + t x (R lin), R = R_p Rz(q).   Result written to (ol, orr).
template <class M, int I>
RB_DI void rb_force(const typename M::Param& p, RB_R s, RB_R c, const RB_R (&lin)[3], const RB_R (&rot)[3],
                    RB_R (&ol)[3], RB_R (&orr)[3]) {
    const RB_R y0 = fma(c, lin[0], -(s * lin[1])), y1 = fma(s, lin[0], c * lin[1]), y2 = lin[2];
    const RB_R w0 = fma(c, rot[0], -(s * rot[1])), w1 = fma(s, rot[0], c * rot[1]), w2 = rot[2];
    const RB_R L0 = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), y0, y1, y2);
    const RB_R L1 = k_dot3<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), y0, y1, y2);
    const RB_R L2 = k_dot3<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), y0, y1, y2);
    const RB_R t0 = KV(I, RB_F_T, 0), t1 = KV(I, RB_F_T, 1), t2 = KV(I, RB_F_T, 2);
    RB_R r0 = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), w0, w1, w2);
    RB_R r1 = k_dot3<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), w0, w1, w2);
    RB_R r2 = k_dot3<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), w0, w1, w2);
    r0 = k_fnma<KC(I, RB_F_T, 2)>(t2, L1, k_fma<KC(I, RB_F_T, 1)>(t1, L2, r0));
    r1 = k_fnma<KC(I, RB_F_T, 0)>(t0, L2, k_fma<KC(I, RB_F_T, 2)>(t2, L0, r1));
    r2 = k_fnma<KC(I, RB_F_T, 1)>(t1, L0, k_fma<KC(I, RB_F_T, 0)>(t0, L1, r2));
    ol[0] = L0; ol[1] = L1; ol[2] = L2;
    orr[0] = r0; orr[1] = r1; orr[2] = r2;
}

// f = I_I * a  (inertia.rs:107-117):  lin = m a.lin - h x a.rot ; rot = I_o a.rot + h x a.lin
template <class M, int I>
RB_DI void rb_inertia_mul(const typename M::Param& p, const RB_R (&al)[3], const RB_R (&ar)[3],
                          RB_R (&fl)[3], RB_R (&fr)[3]) {
    const RB_R m = KV(I, RB_F_M, 0);
    const RB_R h0 = KV(I, RB_F_H, 0), h1 = KV(I, RB_F_H, 1), h2 = KV(I, RB_F_H, 2);
    fl[0] = fma(h2, ar[1], fma(-h1, ar[2], m * al[0]));
    fl[1] = fma(h0, ar[2], fma(-h2, ar[0], m * al[1]));
    fl[2] = fma(h1, ar[0], fma(-h0, ar[1], m * al[2]));
    const RB_R Ixx = KV(I, RB_F_I, 0), Ixy = KV(I, RB_F_I, 1), Ixz = KV(I, RB_F_I, 2);
    const RB_R Iyy = KV(I, RB_F_I, 3), Iyz = KV(I, RB_F_I, 4), Izz = KV(I, RB_F_I, 5);
    fr[0] = fma(-h2, al[1], fma(h1, al[2], fma(Ixz, ar[2], fma(Ixy, ar[1], Ixx * ar[0]))));
    fr[1] = fma(-h0, al[2], fma(h2, al[0], fma(Iyz, ar[2], fma(Iyy, ar[1], Ixy * ar[0]))));
    fr[2] = fma(-h1, al[0], fma(h0, al[1], fma(Izz, ar[2], fma(Iyz, ar[1], Ixz * ar[0]))));
}

// sin/cos of every joint angle (joint.rs:48-50 builds the same rotation as a quaternion).
RB_DI void rb_sincos(double x, double* s, double* c) { sincos(x, s, c); }
RB_DI void rb_sincos(float x, float* s, float* c) { sincosf(x, s, c); }
// One angle, |x| < RB_SINCOS_FAST_LIMIT, no branches: three-term Cody-Waite reduction by pi/2 with FMAs (the quotient
// has at most 17 bits, every product is exact inside its FMA), then the fdlibm kernels on [-pi/4, pi/4] (S1..S6,
// C1..C6; < 1 ulp) and the quadrant fix-up with selects.  Same cost as the fast path of CUDA's sincos() (23 FP64
// instructions) but straight-line, so that rb_sincos_all can interleave the joints of a state: CUDA's version carries a
// slow-path branch per call, which serialises them -- 7 dependent ~13-deep FMA chains per state, 38 % of a rollout step
// when a lone warp runs it (profiles/r2_rollout_ws_stalls.txt).  tools/check_sincos.c pins the accuracy on the host.
#define RB_SINCOS_FAST_LIMIT 1.0e5
RB_DI void rb_sincos_fast(double x, double* sn, double* cs) {
    const int k = __double2int_rn(x * 0.6366197723675814);
    const double kd = (double)k;
    double r = fma(-kd, 1.5707963267948966, x);
    r = fma(-kd, 6.123233995736766e-17, r);
    r = fma(-kd, -1.4973849048591698e-33, r);
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(z, ps, 2.75573137070700676789e-06);
    ps = fma(z, ps, -1.98412698298579493134e-04);
    ps = fma(z, ps, 8.33333333332248946124e-03);
    ps = fma(z, ps, -1.66666666666666324348e-01);
    const double s0 = fma(r * z, ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(z, pc, -2.75573143513906633035e-07);
    pc = fma(z, pc, 2.48015872894767294178e-05);
    pc = fma(z, pc, -1.38888888888741095749e-03);
    pc = fma(z, pc, 4.16666666666666019037e-02);
    const double hz = 0.5 * z, w = 1.0 - hz;
    const double c0 = w + ((1.0 - w) - hz + z * (z * pc));
    const double a = (k & 1) ? c0 : s0, b = (k & 1) ? s0 : c0;
    *sn = (k & 2) ? -a : a;
    *cs = ((k + 1) & 2) ? -b : b;
}
// sin/cos of all joints of a state: the branch-free path whenever every angle is in range (one test per state), the
// per-joint library call otherwise (huge angles, NaN, Inf).
template <int N, class T>
RB_DI void rb_sincos_batched(const T (&q)[N], T (&s)[N], T (&c)[N]) {
    if constexpr (sizeof(T) == 8) {
        bool big = false;                         // also true for NaN / Inf
#pragma unroll
        for (int i = 0; i < N; ++i) big = big || !(fabs(q[i]) < RB_SINCOS_FAST_LIMIT);
        if (!big) {
#pragma unroll
            for (int i = 0; i < N; ++i) rb_sincos_fast(q[i], &s[i], &c[i]);
            return;
        }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) rb_sincos(q[i], &s[i], &c[i]);
}
template <int N, class T>
RB_DI void rb_sincos_all(const T (&q)[N], T (&s)[N], T (&c)[N]) {
#if RB_BATCHED_SINCOS >= 2
    rb_sincos_batched<N>(q, s, c);
#else
#pragma unroll
    for (int i = 0; i < N; ++i) rb_sincos(q[i], &s[i], &c[i]);
#endif
}
// ------------------------------------------------------------------ RNEA  (multibody.rs:111-153)
// tau = ID(q, dq, ddq).  HAS_DDQ = false is the bias-force call rnea(q, dq, 0) used by forward dynamics.
//
// Same recursion as the reference, written in the classical Newton-Euler variables instead of spatial ones:
// the reference carries the spatial pair (v, a) and forms f_i = I_i a_i + v_i x* (I_i v_i) (:140); with
// a' = a.lin + w x v.lin (the classical acceleration of the link origin) that wrench is identically
//     F = m a' + alpha x h + w x (w x h),      n = I_o alpha + w x (I_o w) + h x a',
// and a' obeys  a'_i = E_i (a'_{i-1} + alpha_{i-1} x t_i + w_{i-1} x (w_{i-1} x t_i)),  E_i = Rz(q_i)^T R_p^T,
// so the linear velocity never has to be carried (about 20 fewer FP64 instructions per joint).  The outward
// sweep (:122-141) and the inward sweep (:143-150) are otherwise unchanged; gravity is the base's a' (:116-120).
template <class M, int I>
RB_DI void rb_rotate_in(const typename M::Param& p, RB_R s, RB_R c, const RB_R (&x)[3], RB_R (&o)[3]) {
    // o = Rz(q)^T R_p^T x
    const RB_R y0 = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 3), KC(I, RB_F_R, 6)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 3), KV(I, RB_F_R, 6), x[0], x[1], x[2]);
    const RB_R y1 = k_dot3<KC(I, RB_F_R, 1), KC(I, RB_F_R, 4), KC(I, RB_F_R, 7)>(KV(I, RB_F_R, 1), KV(I, RB_F_R, 4), KV(I, RB_F_R, 7), x[0], x[1], x[2]);
    const RB_R y2 = k_dot3<KC(I, RB_F_R, 2), KC(I, RB_F_R, 5), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 2), KV(I, RB_F_R, 5), KV(I, RB_F_R, 8), x[0], x[1], x[2]);
    o[0] = fma(c, y0, s * y1);  o[1] = fma(c, y1, -(s * y0));  o[2] = y2;
}

// kinematic-tree forms (rb_dyn_tree.cuh), taken when M::kTree
template <class M, bool HAS_DDQ>
RB_DI void rb_rnea_tree(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N],
                        const RB_R (&dq)[M::N], const RB_R (&ddq)[M::N], RB_R (&tau)[M::N]);
template <class M, class Put>
RB_DI void rb_crba_put_tree(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N], Put&& put);
template <class M>
RB_DI void rb_fwd_kin_tree(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N], RB_R (&pos)[3]);
template <class M>
RB_DI void rb_jac_tree(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N], RB_R (&J)[M::N][6]);

template <class M, bool HAS_DDQ>
RB_DI void rb_rnea(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N],
                   const RB_R (&dq)[M::N], const RB_R (&ddq)[M::N], RB_R (&tau)[M::N]) {
    constexpr int N = M::N;
    if constexpr (M::kTree) { rb_rnea_tree<M, HAS_DDQ>(p, s, c, dq, ddq, tau); return; }
    RB_R fl[N][3], fr[N][3];
    RB_R w[3], al[3], ac[3];            // omega, alpha, a' of the current link, in its own frame
    rb_for_up<0, N>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        const RB_R dqi = dq[I];
        if constexpr (I == 0) {
            // base: w = alpha = 0, a' = g (:116-120)
            constexpr int G0 = M::template gcls<0>(), G1 = M::template gcls<1>(), G2 = M::template gcls<2>();
            const RB_R g0 = M::template g<0>(p), g1 = M::template g<1>(p), g2 = M::template g<2>(p);
            // y = R_p^T g with both factors model constants
            constexpr bool y0z = (KC(0, RB_F_R, 0) == RB_ZERO || G0 == RB_ZERO) && (KC(0, RB_F_R, 3) == RB_ZERO || G1 == RB_ZERO) && (KC(0, RB_F_R, 6) == RB_ZERO || G2 == RB_ZERO);
            constexpr bool y1z = (KC(0, RB_F_R, 1) == RB_ZERO || G0 == RB_ZERO) && (KC(0, RB_F_R, 4) == RB_ZERO || G1 == RB_ZERO) && (KC(0, RB_F_R, 7) == RB_ZERO || G2 == RB_ZERO);
            const RB_R y0 = k_dot3<KC(0, RB_F_R, 0), KC(0, RB_F_R, 3), KC(0, RB_F_R, 6)>(KV(0, RB_F_R, 0), KV(0, RB_F_R, 3), KV(0, RB_F_R, 6), g0, g1, g2);
            const RB_R y1 = k_dot3<KC(0, RB_F_R, 1), KC(0, RB_F_R, 4), KC(0, RB_F_R, 7)>(KV(0, RB_F_R, 1), KV(0, RB_F_R, 4), KV(0, RB_F_R, 7), g0, g1, g2);
            const RB_R y2 = k_dot3<KC(0, RB_F_R, 2), KC(0, RB_F_R, 5), KC(0, RB_F_R, 8)>(KV(0, RB_F_R, 2), KV(0, RB_F_R, 5), KV(0, RB_F_R, 8), g0, g1, g2);
            w[0] = 0.0; w[1] = 0.0; w[2] = dqi;                                       // :130
            al[0] = 0.0; al[1] = 0.0; al[2] = HAS_DDQ ? ddq[I] : RB_R(0);                 // :133
            RB_R nz;                                                                 // the only entry of f_0 that is ever read (:144)
            if constexpr (y0z && y1z) {
                ac[0] = 0.0; ac[1] = 0.0; ac[2] = y2;
                nz = HAS_DDQ ? KV(0, RB_F_I, 5) * ddq[I] : RB_R(0);
            } else {
                ac[0] = fma(c[0], y0, s[0] * y1);  ac[1] = fma(c[0], y1, -(s[0] * y0));  ac[2] = y2;
                nz = fma(KV(0, RB_F_H, 0), ac[1], -(KV(0, RB_F_H, 1) * ac[0]));
                if constexpr (HAS_DDQ) nz = fma(KV(0, RB_F_I, 5), ddq[I], nz);
            }
            fl[0][0] = 0.0; fl[0][1] = 0.0; fl[0][2] = 0.0;
            fr[0][0] = 0.0; fr[0][1] = 0.0; fr[0][2] = nz;
        } else {
            // a'_i = E (a' + alpha x t + w x (w x t)) with the parent's w, alpha, a'
            const RB_R t0 = KV(I, RB_F_T, 0), t1 = KV(I, RB_F_T, 1), t2 = KV(I, RB_F_T, 2);
            constexpr int T0 = KC(I, RB_F_T, 0), T1 = KC(I, RB_F_T, 1), T2 = KC(I, RB_F_T, 2);
            RB_R b[3];
            if constexpr (T0 == RB_ZERO && T1 == RB_ZERO && T2 == RB_ZERO) {
                b[0] = ac[0]; b[1] = ac[1]; b[2] = ac[2];
            } else {
                // u = w x t
                const RB_R u0 = k_fnma<T1>(t1, w[2], k_mul<T2>(t2, w[1]));
                const RB_R u1 = k_fnma<T2>(t2, w[0], k_mul<T0>(t0, w[2]));
                const RB_R u2 = k_fnma<T0>(t0, w[1], k_mul<T1>(t1, w[0]));
                b[0] = k_fma<T2>(t2, al[1], k_fnma<T1>(t1, al[2], ac[0]));            // + alpha x t
                b[1] = k_fma<T0>(t0, al[2], k_fnma<T2>(t2, al[0], ac[1]));
                b[2] = k_fma<T1>(t1, al[0], k_fnma<T0>(t0, al[1], ac[2]));
                b[0] = fma(w[1], u2, fma(-w[2], u1, b[0]));                            // + w x u
                b[1] = fma(w[2], u0, fma(-w[0], u2, b[1]));
                b[2] = fma(w[0], u1, fma(-w[1], u0, b[2]));
            }
            RB_R wn[3], aln[3];
            rb_rotate_in<M, I>(p, s[I], c[I], b, ac);
            rb_rotate_in<M, I>(p, s[I], c[I], w, wn);                                  // :129
            rb_rotate_in<M, I>(p, s[I], c[I], al, aln);                                // :132
            // alpha_i = E alpha + z ddq + (E w) x z dq   (:133, :137-138);  w_i = E w + z dq (:130)
            al[0] = fma(wn[1], dqi, aln[0]);
            al[1] = fma(-wn[0], dqi, aln[1]);
            al[2] = HAS_DDQ ? aln[2] + ddq[I] : aln[2];
            w[0] = wn[0]; w[1] = wn[1]; w[2] = wn[2] + dqi;
            // wrench of link i about its origin (:140)
            const RB_R m = KV(I, RB_F_M, 0);
            const RB_R h0 = KV(I, RB_F_H, 0), h1 = KV(I, RB_F_H, 1), h2 = KV(I, RB_F_H, 2);
            const RB_R Ixx = KV(I, RB_F_I, 0), Ixy = KV(I, RB_F_I, 1), Ixz = KV(I, RB_F_I, 2);
            const RB_R Iyy = KV(I, RB_F_I, 3), Iyz = KV(I, RB_F_I, 4), Izz = KV(I, RB_F_I, 5);
            const RB_R e0 = fma(w[1], h2, -(w[2] * h1));                             // e = w x h
            const RB_R e1 = fma(w[2], h0, -(w[0] * h2));
            const RB_R e2 = fma(w[0], h1, -(w[1] * h0));
            // F = m a' + alpha x h + w x e
            fl[I][0] = fma(w[1], e2, fma(-w[2], e1, fma(al[1], h2, fma(-al[2], h1, m * ac[0]))));
            fl[I][1] = fma(w[2], e0, fma(-w[0], e2, fma(al[2], h0, fma(-al[0], h2, m * ac[1]))));
            fl[I][2] = fma(w[0], e1, fma(-w[1], e0, fma(al[0], h1, fma(-al[1], h0, m * ac[2]))));
            // L = I_o w ;  n = I_o alpha + w x L + h x a'
            const RB_R L0 = fma(Ixz, w[2], fma(Ixy, w[1], Ixx * w[0]));
            const RB_R L1 = fma(Iyz, w[2], fma(Iyy, w[1], Ixy * w[0]));
            const RB_R L2 = fma(Izz, w[2], fma(Iyz, w[1], Ixz * w[0]));
            fr[I][0] = fma(h1, ac[2], fma(-h2, ac[1], fma(w[1], L2, fma(-w[2], L1, fma(Ixz, al[2], fma(Ixy, al[1], Ixx * al[0]))))));
            fr[I][1] = fma(h2, ac[0], fma(-h0, ac[2], fma(w[2], L0, fma(-w[0], L2, fma(Iyz, al[2], fma(Iyy, al[1], Ixy * al[0]))))));
            fr[I][2] = fma(h0, ac[1], fma(-h1, ac[0], fma(w[0], L1, fma(-w[1], L0, fma(Izz, al[2], fma(Iyz, al[1], Ixz * al[0]))))));
        }
    });
    rb_for_down<N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        tau[I] = fr[I][2];                                                           // :144
        if constexpr (I > 0) {
            RB_R tl[3], tr[3];
            rb_force<M, I>(p, s[I], c[I], fl[I], fr[I], tl, tr);                     // :147
            fl[I - 1][0] += tl[0]; fl[I - 1][1] += tl[1]; fl[I - 1][2] += tl[2];     // :148
            fr[I - 1][0] += tr[0]; fr[I - 1][1] += tr[1]; fr[I - 1][2] += tr[2];
        }
    });
}

// ------------------------------------------------------------------ CRBA  (multibody.rs:155-174)
// H[j][i] for j <= i (row j, column i): diagonal + strict upper triangle, exactly what the reference writes.
// Composite inertia kept as (h, I_o) in the frame of link i; its mass is the model constant mc_i.
// The reference carries (m, com, I_c) and rebuilds I_o with from_com/from_origin (inertia.rs:21-51,81-105);
// the 10-parameter update below is the same map: with R = R_p Rz(q), u = R h + (m/2) t,
//   h' = R h + m t,   I_o' = R I_o R^T - (t u^T + u t^T) + 2 (t.u) Id,   then add link i-1's own (h, I_o).
// `put(RbIC<J>, RbIC<I>, value)` receives every entry H(J, I), J <= I, once.
// s, c: anything indexable by joint (arrays of sin/cos, or a view that reads them from shared memory on demand).
template <class M, class SC, class Put>
RB_DI void rb_crba_put(const typename M::Param& p, const SC& s, const SC& c, Put&& put) {
    constexpr int N = M::N;
    if constexpr (M::kTree) {
        RB_R sa[N], ca[N];
#pragma unroll
        for (int i = 0; i < N; ++i) { sa[i] = s[i]; ca[i] = c[i]; }
        rb_crba_put_tree<M>(p, sa, ca, put);
        return;
    }
    RB_R h[3] = {KV(N - 1, RB_F_H, 0), KV(N - 1, RB_F_H, 1), KV(N - 1, RB_F_H, 2)};            // :157
    RB_R Ixx = KV(N - 1, RB_F_I, 0), Ixy = KV(N - 1, RB_F_I, 1), Ixz = KV(N - 1, RB_F_I, 2);
    RB_R Iyy = KV(N - 1, RB_F_I, 3), Iyz = KV(N - 1, RB_F_I, 4), Izz = KV(N - 1, RB_F_I, 5);
    rb_for_down<N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        put(RbIC<I>{}, RbIC<I>{}, Izz);                                              // :161
        RB_R Fl[3] = {-h[1], h[0], 0.0};                                           // :162  F = I^c * S_z
        RB_R Fr[3] = {Ixz, Iyz, Izz};
        rb_for_down<I - 1>([&](auto jc) {
            constexpr int J = decltype(jc)::value;
            RB_R ol[3], orr[3];
            rb_force<M, J + 1>(p, s[J + 1], c[J + 1], Fl, Fr, ol, orr);              // :165
            Fl[0] = ol[0]; Fl[1] = ol[1]; Fl[2] = ol[2];
            Fr[0] = orr[0]; Fr[1] = orr[1]; Fr[2] = orr[2];
            put(RbIC<J>{}, RbIC<I>{}, Fr[2]);                                        // :166
        });
        if constexpr (I > 0) {                                                       // :169-171
            const RB_R si = s[I], ci = c[I];
            // Rz(q): h, I_o
            const RB_R g0 = fma(ci, h[0], -(si * h[1])), g1 = fma(si, h[0], ci * h[1]), g2 = h[2];
            const RB_R cs = ci * si, s2 = cs + cs, c2 = fma(ci, ci, -(si * si));
            const RB_R hm = RB_R(0.5) * (Ixx - Iyy), hp = RB_R(0.5) * (Ixx + Iyy);
            const RB_R u_ = fma(hm, c2, -(Ixy * s2));
            const RB_R a = hp + u_, e = hp - u_, b = fma(hm, s2, Ixy * c2);
            const RB_R d = fma(ci, Ixz, -(si * Iyz)), f = fma(si, Ixz, ci * Iyz), g = Izz;
            // R_p: h'' = R_p g ; I'' = R_p A R_p^T with A = [[a,b,d],[b,e,f],[d,f,g]]
#define RR(r, k) KV(I, RB_F_R, 3 * (r) + (k))
#define RC(r, k) KC(I, RB_F_R, 3 * (r) + (k))
            const RB_R q0 = k_dot3<RC(0, 0), RC(0, 1), RC(0, 2)>(RR(0, 0), RR(0, 1), RR(0, 2), g0, g1, g2);
            const RB_R q1 = k_dot3<RC(1, 0), RC(1, 1), RC(1, 2)>(RR(1, 0), RR(1, 1), RR(1, 2), g0, g1, g2);
            const RB_R q2 = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), g0, g1, g2);
            // P = R_p A (rows of R_p against columns of symmetric A)
            const RB_R P00 = k_dot3<RC(0, 0), RC(0, 1), RC(0, 2)>(RR(0, 0), RR(0, 1), RR(0, 2), a, b, d);
            const RB_R P01 = k_dot3<RC(0, 0), RC(0, 1), RC(0, 2)>(RR(0, 0), RR(0, 1), RR(0, 2), b, e, f);
            const RB_R P02 = k_dot3<RC(0, 0), RC(0, 1), RC(0, 2)>(RR(0, 0), RR(0, 1), RR(0, 2), d, f, g);
            const RB_R P10 = k_dot3<RC(1, 0), RC(1, 1), RC(1, 2)>(RR(1, 0), RR(1, 1), RR(1, 2), a, b, d);
            const RB_R P11 = k_dot3<RC(1, 0), RC(1, 1), RC(1, 2)>(RR(1, 0), RR(1, 1), RR(1, 2), b, e, f);
            const RB_R P12 = k_dot3<RC(1, 0), RC(1, 1), RC(1, 2)>(RR(1, 0), RR(1, 1), RR(1, 2), d, f, g);
            const RB_R P20 = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), a, b, d);
            const RB_R P21 = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), b, e, f);
            const RB_R P22 = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), d, f, g);
            // I'' = P R_p^T, six unique entries: I''[r][c] = sum_k P[r][k] R_p[c][k]
            RB_R Jxx = k_dot3<RC(0, 0), RC(0, 1), RC(0, 2)>(RR(0, 0), RR(0, 1), RR(0, 2), P00, P01, P02);
            RB_R Jxy = k_dot3<RC(1, 0), RC(1, 1), RC(1, 2)>(RR(1, 0), RR(1, 1), RR(1, 2), P00, P01, P02);
            RB_R Jxz = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), P00, P01, P02);
            RB_R Jyy = k_dot3<RC(1, 0), RC(1, 1), RC(1, 2)>(RR(1, 0), RR(1, 1), RR(1, 2), P10, P11, P12);
            RB_R Jyz = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), P10, P11, P12);
            RB_R Jzz = k_dot3<RC(2, 0), RC(2, 1), RC(2, 2)>(RR(2, 0), RR(2, 1), RR(2, 2), P20, P21, P22);
#undef RR
#undef RC
            // translation by t with composite mass mc_I:  u = h'' + (mc/2) t
            const RB_R mc = KV(I, RB_F_M, 1);
            const RB_R t0 = KV(I, RB_F_T, 0), t1 = KV(I, RB_F_T, 1), t2 = KV(I, RB_F_T, 2);
            constexpr int T0 = KC(I, RB_F_T, 0), T1 = KC(I, RB_F_T, 1), T2 = KC(I, RB_F_T, 2);
            const RB_R hmc = RB_R(0.5) * mc;
            const RB_R u0 = k_fma<T0>(t0, hmc, q0), u1 = k_fma<T1>(t1, hmc, q1), u2 = k_fma<T2>(t2, hmc, q2);
            const RB_R tu0 = k_mul<T0>(t0, u0), tu1 = k_mul<T1>(t1, u1), tu2 = k_mul<T2>(t2, u2);
            // diag: + 2 (t.u - t_k u_k);  off-diag: - (t_r u_c + t_c u_r);  then add link I-1's own inertia
            Ixx = fma(RB_R(2), tu1 + tu2, Jxx) + KV(I - 1, RB_F_I, 0);
            Iyy = fma(RB_R(2), tu0 + tu2, Jyy) + KV(I - 1, RB_F_I, 3);
            Izz = fma(RB_R(2), tu0 + tu1, Jzz) + KV(I - 1, RB_F_I, 5);
            Ixy = k_fnma<T1>(t1, u0, k_fnma<T0>(t0, u1, Jxy)) + KV(I - 1, RB_F_I, 1);
            Ixz = k_fnma<T2>(t2, u0, k_fnma<T0>(t0, u2, Jxz)) + KV(I - 1, RB_F_I, 2);
            Iyz = k_fnma<T2>(t2, u1, k_fnma<T1>(t1, u2, Jyz)) + KV(I - 1, RB_F_I, 4);
            h[0] = k_fma<T0>(t0, mc, q0) + KV(I - 1, RB_F_H, 0);
            h[1] = k_fma<T1>(t1, mc, q1) + KV(I - 1, RB_F_H, 1);
            h[2] = k_fma<T2>(t2, mc, q2) + KV(I - 1, RB_F_H, 2);
        }
    });
}

template <class M, class SC>
RB_DI void rb_crba(const typename M::Param& p, const SC& s, const SC& c, RB_R (&H)[M::N][M::N]) {
    if constexpr (M::kTree) {                        // entries whose row joint does not support the column joint stay 0
#pragma unroll
        for (int r = 0; r < M::N; ++r)
#pragma unroll
            for (int k = 0; k < M::N; ++k) H[r][k] = RB_R(0);
    }
    rb_crba_put<M>(p, s, c, [&](auto jc, auto ic, RB_R v) { H[decltype(jc)::value][decltype(ic)::value] = v; });
}

// 1/d for a pivot d of an SPD matrix (normal, positive): hardware seed (rcp.approx.ftz.f64, ~20 good bits,
// SASS MUFU.RCP64H) + two Newton steps = 5 FP64-pipe instructions against ~12 for the IEEE `1.0 / d` sequence with
// its special-case handling; error <= 1 ulp on normal inputs.  d <= 0 or NaN is reported by the caller (ok flag).
RB_DI double rb_rcp_pos(double d) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
    double e = fma(-d, x, 1.0);
    x = fma(x, e, x);
    e = fma(-d, x, 1.0);
    return fma(x, e, x);
}
RB_DI float rb_rcp_pos(float d) { return __frcp_rn(d); }

// ------------------------------------------------------------------ solve  H x = b, H SPD given by its upper triangle
// In-place right-looking LDL^T (the square-root-free Cholesky; SURVEY.md a13), then the two triangular solves.
// Returns false if a pivot is not positive (H not SPD).
template <int N, class T>
RB_DI bool rb_ldlt_solve(T (&A)[N][N], T (&x)[N]) {
    T dinv[N];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const T d = A[j][j];
        ok = ok && (d > T(0));
        dinv[j] = rb_rcp_pos(d);
#pragma unroll
        for (int i = j + 1; i < N; ++i) {
            const T l = A[j][i] * dinv[j];
#pragma unroll
            for (int k = i; k < N; ++k) A[i][k] = fma(-l, A[j][k], A[i][k]);
            A[j][i] = l;                     // U[j][i] = L[i][j]
        }
    }
#pragma unroll
    for (int j = 0; j < N; ++j) {            // L y = b
#pragma unroll
        for (int i = j + 1; i < N; ++i) x[i] = fma(-A[j][i], x[j], x[i]);
    }
#pragma unroll
    for (int j = 0; j < N; ++j) x[j] *= dinv[j];
#pragma unroll
    for (int i = N - 1; i >= 0; --i) {       // L^T x = z
#pragma unroll
        for (int k = i + 1; k < N; ++k) x[i] = fma(-A[i][k], x[k], x[i]);
    }
    return ok;
}

// The same factorisation with compile-time loop indices (template recursion instead of `#pragma unroll`): beyond
// 7-8 joints nvcc stops unrolling the triple loop of rb_ldlt_solve, indexes H dynamically and so moves the whole
// matrix to local memory (1.2-1.6 KB stack frame at N = 12).  Same operations in the same order.
template <int N, class T>
RB_DI bool rb_ldlt_solve_static(T (&A)[N][N], T (&x)[N]) {
    T dinv[N];
    bool ok = true;
    rb_for_up<0, N>([&](auto jc) {
        constexpr int J = decltype(jc)::value;
        const T d = A[J][J];
        ok = ok && (d > T(0));
        dinv[J] = rb_rcp_pos(d);
        rb_for_up<J + 1, N>([&](auto ic) {
            constexpr int I = decltype(ic)::value;
            const T l = A[J][I] * dinv[J];
            rb_for_up<I, N>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                A[I][K] = fma(-l, A[J][K], A[I][K]);
            });
            A[J][I] = l;
        });
    });
    rb_for_up<0, N>([&](auto jc) {
        constexpr int J = decltype(jc)::value;
        rb_for_up<J + 1, N>([&](auto ic) { constexpr int I = decltype(ic)::value; x[I] = fma(-A[J][I], x[J], x[I]); });
    });
    rb_for_up<0, N>([&](auto jc) { constexpr int J = decltype(jc)::value; x[J] *= dinv[J]; });
    rb_for_down<N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        rb_for_up<I + 1, N>([&](auto kc) { constexpr int K = decltype(kc)::value; x[I] = fma(-A[I][K], x[K], x[I]); });
    });
    return ok;
}

// The same LDL^T in two halves, for callers that factorise and solve in different places (the warp-specialised rollout
// hands L and 1/d from one warp to another).  Operation for operation rb_ldlt_solve / rb_ldlt_solve_static: a
// factorisation here followed by rb_ldlt_apply gives bit-identical results.
template <int N, class T>
RB_DI bool rb_ldlt_factor(T (&A)[N][N], T (&dinv)[N]) {
    bool ok = true;
    rb_for_up<0, N>([&](auto jc) {
        constexpr int J = decltype(jc)::value;
        const T d = A[J][J];
        ok = ok && (d > T(0));
        dinv[J] = rb_rcp_pos(d);
        rb_for_up<J + 1, N>([&](auto ic) {
            constexpr int I = decltype(ic)::value;
            const T l = A[J][I] * dinv[J];
            rb_for_up<I, N>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                A[I][K] = fma(-l, A[J][K], A[I][K]);
            });
            A[J][I] = l;
        });
    });
    return ok;
}
// x <- (L D L^T)^-1 x with L(I, J) = getL(RbIC<J>, RbIC<I>) for J < I (the strict upper triangle rb_ldlt_factor leaves).
template <int N, class T, class GetL>
RB_DI void rb_ldlt_apply_fn(GetL&& getL, const T (&dinv)[N], T (&x)[N]) {
    rb_for_up<0, N>([&](auto jc) {
        constexpr int J = decltype(jc)::value;
        rb_for_up<J + 1, N>([&](auto ic) { constexpr int I = decltype(ic)::value; x[I] = fma(-getL(RbIC<J>{}, RbIC<I>{}), x[J], x[I]); });
    });
    rb_for_up<0, N>([&](auto jc) { constexpr int J = decltype(jc)::value; x[J] *= dinv[J]; });
    rb_for_down<N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        rb_for_up<I + 1, N>([&](auto kc) { constexpr int K = decltype(kc)::value; x[I] = fma(-getL(RbIC<I>{}, RbIC<K>{}), x[K], x[I]); });
    });
}

// ... with L in the array rb_ldlt_factor left it in.
template <int N, class T>
RB_DI void rb_ldlt_apply(const T (&A)[N][N], const T (&dinv)[N], T (&x)[N]) {
    rb_ldlt_apply_fn<N>([&](auto jc, auto ic) { return A[decltype(jc)::value][decltype(ic)::value]; }, dinv, x);
}

// ------------------------------------------------------------------ forward dynamics (SURVEY.md 3.3)
// qdd = solve(sym(crba(q)), tau - rnea(q, dq, 0)); sin/cos computed once and shared by both halves.
template <class M>
RB_DI bool rb_forward_dynamics(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N],
                               const RB_R (&dq)[M::N], const RB_R (&tau)[M::N], RB_R (&qdd)[M::N]) {
    constexpr int N = M::N;
    {
        RB_R bias[N];
        rb_rnea<M, false>(p, s, c, dq, dq /*unused*/, bias);
#pragma unroll
        for (int i = 0; i < N; ++i) qdd[i] = tau[i] - bias[i];
    }
    RB_R H[N][N];
    rb_crba<M>(p, s, c, H);
    if constexpr (N > 7) return rb_ldlt_solve_static<N>(H, qdd);
    else return rb_ldlt_solve<N>(H, qdd);
}

// ------------------------------------------------------------------ inverse + forward dynamics of ONE state, fused
// What multibody_rnea_fd_batch asks for: tau = rnea(q, dq, ddq) (multibody.rs:111-153) and
// qdd = solve(sym(crba(q)), tau_in - rnea(q, dq, 0)) (:155-174 + the solve) of the same (q, dq).  Everything the two
// share is computed once: sin/cos, the bias recursion rnea(q, dq, 0) and the mass matrix.  The inverse-dynamics result
// then comes from the identity the equations of motion are (and tests/test_oracle.py pins):
//     rnea(q, dq, ddq) = sym(crba(q)) ddq + rnea(q, dq, 0),
// accumulated entry by entry while CRBA produces H (49 FMAs for 7 joints instead of a second ~500-instruction
// recursion).  Rounding differs from the recursion by a few ulp of sum_j |H_ij| |ddq_j| (measured <= 2e-14 relative on
// the FR3, tests/test_gpu_parity.py::test_fused_rnea_fd*), far inside the 1e-10 bar.
template <class M>
RB_DI bool rb_rnea_fd_fused(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N],
                            const RB_R (&dq)[M::N], const RB_R (&ddq)[M::N], const RB_R (&tau_in)[M::N],
                            RB_R (&tau)[M::N], RB_R (&qdd)[M::N]) {
    constexpr int N = M::N;
    rb_rnea<M, false>(p, s, c, dq, dq /*unused*/, tau);            // bias
#pragma unroll
    for (int i = 0; i < N; ++i) qdd[i] = tau_in[i] - tau[i];
    RB_R H[N][N];
    if constexpr (M::kTree) {
#pragma unroll
        for (int r = 0; r < N; ++r)
#pragma unroll
            for (int k = 0; k < N; ++k) H[r][k] = RB_R(0);
    }
    rb_crba_put<M>(p, s, c, [&](auto jc, auto ic, RB_R v) {
        constexpr int J = decltype(jc)::value, I = decltype(ic)::value;
        H[J][I] = v;
        tau[J] = fma(v, ddq[I], tau[J]);
        if constexpr (J != I) tau[I] = fma(v, ddq[J], tau[I]);
    });
    if constexpr (N > 7) return rb_ldlt_solve_static<N>(H, qdd);
    else return rb_ldlt_solve<N>(H, qdd);
}

// ------------------------------------------------------------------ forward kinematics / Jacobian
// Tip pose in the base frame, composed tip -> base as multibody.rs:87-93 does: p <- R_i p + t_i.
template <class M>
RB_DI void rb_fwd_kin(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N], RB_R (&pos)[3]) {
    constexpr int N = M::N;
    if constexpr (M::kTree) { rb_fwd_kin_tree<M>(p, s, c, pos); return; }
    pos[0] = 0.0; pos[1] = 0.0; pos[2] = 0.0;
    rb_for_down<N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        const RB_R y0 = fma(c[I], pos[0], -(s[I] * pos[1])), y1 = fma(s[I], pos[0], c[I] * pos[1]), y2 = pos[2];
        pos[0] = k_dot3_acc<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_T, 0), KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), y0, y1, y2);
        pos[1] = k_dot3_acc<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_T, 1), KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), y0, y1, y2);
        pos[2] = k_dot3_acc<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_T, 2), KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), y0, y1, y2);
    });
}

// Tip-frame Jacobian (multibody.rs:95-108): column i = S_z carried from frame i to the tip frame by the
// motion transform of the accumulated pose (A, r) of the tip in frame i:  rot = A^T z, lin = A^T (-(r x z)).
// J is [N][6]: J[i][0..2] lin, J[i][3..5] rot.
template <class M>
RB_DI void rb_jac(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N], RB_R (&J)[M::N][6]) {
    constexpr int N = M::N;
    if constexpr (M::kTree) { rb_jac_tree<M>(p, s, c, J); return; }
    // orientation of the reference's tip frame in the model's last frame (identity unless the last axis was re-based)
    RB_R A[3][3] = {{M::template tip<0>(p), M::template tip<1>(p), M::template tip<2>(p)},
                    {M::template tip<3>(p), M::template tip<4>(p), M::template tip<5>(p)},
                    {M::template tip<6>(p), M::template tip<7>(p), M::template tip<8>(p)}};
    RB_R r[3] = {0.0, 0.0, 0.0};
    rb_for_down<N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        // -(r x z) = (-r1, r0, 0)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            J[I][k] = fma(A[1][k], r[0], -(A[0][k] * r[1]));
            J[I][3 + k] = A[2][k];
        }
        if constexpr (I > 0) {
            // (A, r) <- X_I o (A, r):  A <- R_p Rz A,  r <- R_p Rz r + t
            RB_R B[3][3], y[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                B[0][k] = fma(c[I], A[0][k], -(s[I] * A[1][k]));
                B[1][k] = fma(s[I], A[0][k], c[I] * A[1][k]);
                B[2][k] = A[2][k];
            }
            y[0] = fma(c[I], r[0], -(s[I] * r[1])); y[1] = fma(s[I], r[0], c[I] * r[1]); y[2] = r[2];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                A[0][k] = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), B[0][k], B[1][k], B[2][k]);
                A[1][k] = k_dot3<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), B[0][k], B[1][k], B[2][k]);
                A[2][k] = k_dot3<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), B[0][k], B[1][k], B[2][k]);
            }
            r[0] = k_dot3_acc<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_T, 0), KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), y[0], y[1], y[2]);
            r[1] = k_dot3_acc<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_T, 1), KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), y[0], y[1], y[2]);
            r[2] = k_dot3_acc<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_T, 2), KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), y[0], y[1], y[2]);
        }
    });
}

#include "rb_dyn_tree.cuh"

// ------------------------------------------------------------------ tip pose (tip-pose cost terms of rollouts)
// Orientation R of the tip frame in the base frame (the frame of rb_jac: the reference's last link frame, tip rotation
// included) and its origin pos (rb_fwd_kin's result, the same operations).  Composed tip -> base along the supporting
// branch (the whole chain for serial chains): A <- R_p Rz A; the last joint's factor starts from the identity and the
// tip rotation is applied at the end, so the exact 0 and +-1 of the fixed rotations drop out of every product.
template <class M>
RB_DI void rb_tip_pose(const typename M::Param& p, const RB_R (&s)[M::N], const RB_R (&c)[M::N], RB_R (&R)[3][3], RB_R (&pos)[3]) {
    constexpr int N = M::N;
    RB_R A[3][3];
    pos[0] = 0.0; pos[1] = 0.0; pos[2] = 0.0;
    rb_for_anc<M, N - 1>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        const RB_R y0 = fma(c[I], pos[0], -(s[I] * pos[1])), y1 = fma(s[I], pos[0], c[I] * pos[1]), y2 = pos[2];
        pos[0] = k_dot3_acc<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_T, 0), KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), y0, y1, y2);
        pos[1] = k_dot3_acc<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_T, 1), KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), y0, y1, y2);
        pos[2] = k_dot3_acc<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_T, 2), KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), y0, y1, y2);
        if constexpr (I == N - 1) {
            // A = R_p Rz(q): columns (c r0 + s r1, c r1 - s r0, r2) of R_p's rows r
            rb_for_up<0, 3>([&](auto rc) {
                constexpr int r = decltype(rc)::value;
                A[r][0] = k_dot3<KC(I, RB_F_R, 3 * r), KC(I, RB_F_R, 3 * r + 1), RB_ZERO>(KV(I, RB_F_R, 3 * r), KV(I, RB_F_R, 3 * r + 1), RB_R(0), c[I], s[I], RB_R(0));
                A[r][1] = k_dot3<KC(I, RB_F_R, 3 * r + 1), KC(I, RB_F_R, 3 * r), RB_ZERO>(KV(I, RB_F_R, 3 * r + 1), KV(I, RB_F_R, 3 * r), RB_R(0), c[I], -s[I], RB_R(0));
                A[r][2] = KV(I, RB_F_R, 3 * r + 2);
            });
        } else {
            RB_R B[3][3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                B[0][k] = fma(c[I], A[0][k], -(s[I] * A[1][k]));
                B[1][k] = fma(s[I], A[0][k], c[I] * A[1][k]);
                B[2][k] = A[2][k];
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                A[0][k] = k_dot3<KC(I, RB_F_R, 0), KC(I, RB_F_R, 1), KC(I, RB_F_R, 2)>(KV(I, RB_F_R, 0), KV(I, RB_F_R, 1), KV(I, RB_F_R, 2), B[0][k], B[1][k], B[2][k]);
                A[1][k] = k_dot3<KC(I, RB_F_R, 3), KC(I, RB_F_R, 4), KC(I, RB_F_R, 5)>(KV(I, RB_F_R, 3), KV(I, RB_F_R, 4), KV(I, RB_F_R, 5), B[0][k], B[1][k], B[2][k]);
                A[2][k] = k_dot3<KC(I, RB_F_R, 6), KC(I, RB_F_R, 7), KC(I, RB_F_R, 8)>(KV(I, RB_F_R, 6), KV(I, RB_F_R, 7), KV(I, RB_F_R, 8), B[0][k], B[1][k], B[2][k]);
            }
        }
    });
    // R = A tip
    rb_for_up<0, 3>([&](auto kc) {
        constexpr int k = decltype(kc)::value;
        constexpr int T0 = M::template tipcls<k>(), T1 = M::template tipcls<3 + k>(), T2 = M::template tipcls<6 + k>();
#pragma unroll
        for (int r = 0; r < 3; ++r)
            R[r][k] = k_dot3<T0, T1, T2>(M::template tip<k>(p), M::template tip<3 + k>(p), M::template tip<6 + k>(p), A[r][0], A[r][1], A[r][2]);
    });
}

// The tip-pose terms of RbTipCost at one state whose tip pose is (R, pos); tw = their row of the cost-weight block
// (RB_TW_* entries).  With x = pos + R offset and e = x - p_ref:
//   run = sum_k w_p[k] e_k^2 + w_R ||R - R_ref||_F^2,   fin = the same with w_p_final, w_R_final.
RB_DI void rb_tip_terms(const double (&R)[3][3], const double (&pos)[3], const double* __restrict__ tw, double& run, double& fin) {
    auto w = [&](int k) { return __ldg(tw + k); };
    double ep = 0.0, epf = 0.0, dR = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double x = fma(R[k][2], w(RB_TW_OFFSET + 2), fma(R[k][1], w(RB_TW_OFFSET + 1), fma(R[k][0], w(RB_TW_OFFSET), pos[k])));
        const double e = x - w(RB_TW_PREF + k);
        ep = fma(w(RB_TW_WP + k) * e, e, ep);
        epf = fma(w(RB_TW_WPF + k) * e, e, epf);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double d = R[k][j] - w(RB_TW_RREF + 3 * k + j);
            dR = fma(d, d, dR);
        }
    }
    run = fma(w(RB_TW_WR), dR, ep);
    fin = fma(w(RB_TW_WRF), dR, epf);
}
