// rb_kernels_deriv.cu -- analytical-derivative kernels (rb_deriv.cuh), one instantiation per chain length
// (inverse dynamics: 1..32 joints; forward dynamics and the rollout adjoint, which also unroll FD itself: 1..12).
// Unlike the other register-resident kernels these are NOT specialised on the model: the algebra runs in the world
// frame, where the zeros of a particular robot's fixed rotations buy little, and real loops over the joints keep the
// code small and the register allocation sane.  The model travels as a __grid_constant__ parameter (<= 6.2 KB).
#include "rb_kernels.cuh"
#include "rb_deriv.cuh"
#include "rb_util.cuh"

#ifndef RB_MINB_DERIV
#define RB_MINB_DERIV 2
#endif
#ifndef RB_MINB_ADJOINT
#define RB_MINB_ADJOINT 2
#endif

// out: [2 N^2][ld]: d tau_r / d q_c at entry r + N c, then d tau_r / d dq_c at N^2 + r + N c.
template <int N>
__global__ void __launch_bounds__(RB_BLOCK, RB_MINB_DERIV)
rb_rnea_deriv_kernel(const __grid_constant__ RbModelK<N> p, const double* __restrict__ q, const double* __restrict__ dq,
                     const double* __restrict__ ddq, double* __restrict__ out, size_t B, size_t ld) {
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    double a[N], b[N], c[N], sn[N], cs[N];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    rb_load<N>(dq, ld, s, b);
    rb_load<N>(ddq, ld, s, c);
    double* o = out + s;
    rb_rnea_derivatives<N>(p, sn, cs, b, c, [&](int blk, int r, int col, double v) { __stcs(o + (size_t)(blk * N * N + r + N * col) * ld, v); });
}

// out: [3 N^2][ld]: d qdd / d q, d qdd / d dq, H^-1 (= d qdd / d tau), each entry r + N c.
//   qdd = FD(q, dq, tau);  d qdd / d x = -H^-1 (d rnea / d x at ddq = qdd).
// The two d rnea matrices pass through `out` (written, then read back column by column by the same thread); the
// factor of H is rebuilt after the derivative sweep rather than kept alive across it (35 doubles of registers).
template <int N>
__global__ void __launch_bounds__(RB_BLOCK, RB_MINB_DERIV)
rb_fd_deriv_kernel(const __grid_constant__ RbModelK<N> p, const double* __restrict__ q, const double* __restrict__ dq,
                   const double* __restrict__ tau, double* __restrict__ out, size_t B, size_t ld, int* __restrict__ status) {
    using M = RtModel<N>;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    double a[N], b[N], x[N], sn[N], cs[N];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    rb_load<N>(dq, ld, s, b);
    rb_load<N>(tau, ld, s, a);
    rb_forward_dynamics<M>(p, sn, cs, b, a, x);              // qdd
    double* o = out + s;
    rb_rnea_derivatives<N>(p, sn, cs, b, x, [&](int blk, int r, int col, double v) { o[(size_t)(blk * N * N + r + N * col) * ld] = v; });
    double H[N][N], dinv[N];
    rb_crba<M>(p, sn, cs, H);
    const bool ok = rb_ldlt_factor<N>(H, dinv);
    if (!ok) atomicOr(status, RB_STATUS_NOT_SPD);
#pragma unroll 1
    for (int c = 0; c < 3 * N; ++c) {                        // columns of the three blocks
        double y[N];
#pragma unroll
        for (int r = 0; r < N; ++r) y[r] = c < 2 * N ? -o[(size_t)(r + N * c) * ld] : (r == c - 2 * N ? 1.0 : 0.0);
        rb_ldlt_apply<N>(H, dinv, y);
#pragma unroll
        for (int r = 0; r < N; ++r) __stcs(o + (size_t)(r + N * c) * ld, ok ? y[r] : rb_nan<double>());
    }
}

// Reverse-mode (vector-Jacobian) pass through the rollout of rb_rollout_kernel, one thread per trajectory.
//   forward step t, u_t = tau[t]:   qdd_t = FD(q_t, dq_t, u_t),  dq_{t+1} = dq_t + dt qdd_t,  q_{t+1} = q_t + dt dq_{t+1}
//   outputs q_traj[t] = q_{t+1}, dq_traj[t] = dq_{t+1}, final = (q_H, dq_H); upstream gradients Gq[t], Gdq[t], Gqf, Gdqf.
//   a_q = Gqf + Gq[H-1],  a_dq = Gdqf + Gdq[H-1]                         (adjoints of q_H, dq_H)
//   for t = H-1 .. 0:                                                    (q_t, dq_t = q_traj[t-1], dq_traj[t-1]; q0, dq0 at t = 0)
//       b    = a_dq + dt a_q                                             (q_{t+1} depends on dq_{t+1})
//       mu   = H(q_t)^-1 (dt b)                                          -> grad_tau[t] = mu
//       a_q  = a_q - (d tau / d q )^T mu     at (q_t, dq_t, ddq = qdd_t)  (rb_rnea_vjp, O(N))
//       a_dq = b   - (d tau / d dq)^T mu
//       t > 0:  a_q += Gq[t-1],  a_dq += Gdq[t-1]
//   grad_q0 = a_q,  grad_dq0 = a_dq.
// QUAD: the upstream gradients of the quadratic cost of RbQuadCost (weights in the engine's cost-weight block cost_w),
// formed here from the stored states:  Gq[t] = 2 dt w_q (q_{t+1} - q_ref),  Gdq[t] = 2 dt w_dq dq_{t+1},
// Gqf = 2 w_q_final (q_H - q_ref),  Gdqf = 2 w_dq_final dq_H;  grad_tau[t] gains the direct term 2 dt w_tau u_t.
// Otherwise they come from g_q / g_dq ([H][N][ld]) and g_qf / g_dqf ([N][ld]); a NULL array is zero.
// TIP (with QUAD): also the tip-pose terms of RbTipCost (row RB_CW_TIP of cost_w): the adjoint of each stored state q_t,
// t >= 1, gains dt times their running gradient, added inside rb_rnea_vjp from the step's own sin/cos; q_H gains the
// running and terminal gradient from one more sin/cos (rb_tip_grad).
// COL (with TIP): also the collision-sphere terms of RbCollisionCost (the block at cost_w + RB_CW_COL), the same way: per
// link wrenches summed in rb_rnea_vjp's inward sweep, and rb_col_grad for q_H.
// These are gradients of the exact-arithmetic map evaluated at the computed states, not of the rounded fma-Euler map.
// One LDL^T of H(q_t) per step serves both solves: qdd_t (operation for operation rb_forward_dynamics) and mu.
// The trajectory (q_traj, dq_traj) has its own leading dimension ld_traj; everything else uses ld.  A trajectory that
// meets a non-SPD mass matrix sets the status bit and gets NaN in every gradient.
template <int N, bool QUAD, bool TIP = false, bool COL = false>
__global__ void __launch_bounds__(RB_BLOCK, RB_MINB_ADJOINT)
rb_rollout_adjoint_kernel(const __grid_constant__ RbModelK<N> p, const double* __restrict__ q0, const double* __restrict__ dq0,
                          const double* __restrict__ tau, const double* __restrict__ q_traj, const double* __restrict__ dq_traj,
                          size_t ld_traj, const double* __restrict__ g_q, const double* __restrict__ g_dq,
                          const double* __restrict__ g_qf, const double* __restrict__ g_dqf, const double* __restrict__ cost_w,
                          double* __restrict__ grad_tau, double* __restrict__ grad_q0, double* __restrict__ grad_dq0,
                          double dt, int horizon, size_t B, size_t ld, int* __restrict__ status) {
    using M = RtModel<N>;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    const size_t step = (size_t)N * ld, step_x = (size_t)N * ld_traj;
    auto w = [&](int row, int i) { return __ldg(cost_w + row * RB_MAX_N + i); };
    double aq[N], adq[N], x[N], xd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) { aq[i] = 0.0; adq[i] = 0.0; }
    if constexpr (QUAD) {                                     // adjoints of (q_H, dq_H) from the terminal and last running cost
        if (horizon > 0) {
            rb_load<N>(q_traj + (size_t)(horizon - 1) * step_x, ld_traj, s, x);
            rb_load<N>(dq_traj + (size_t)(horizon - 1) * step_x, ld_traj, s, xd);
        } else {
            rb_load<N>(q0, ld, s, x);
            rb_load<N>(dq0, ld, s, xd);
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const double e = x[i] - w(RB_CW_QREF, i);
            aq[i] = 2.0 * (w(RB_CW_QF, i) * e);
            adq[i] = 2.0 * (w(RB_CW_DQF, i) * xd[i]);
            if (horizon > 0) {
                aq[i] = fma(2.0 * dt, w(RB_CW_Q, i) * e, aq[i]);
                adq[i] = fma(2.0 * dt, w(RB_CW_DQ, i) * xd[i], adq[i]);
            }
        }
        if constexpr (COL) {
            double sn[N], cs[N];
            rb_sincos_all<N>(x, sn, cs);
            rb_col_grad<N>(p, sn, cs, cost_w + RB_CW_TIP * RB_MAX_N, cost_w + RB_CW_COL, horizon > 0 ? dt : 0.0, 1.0, aq);
        } else if constexpr (TIP) {
            double sn[N], cs[N];
            rb_sincos_all<N>(x, sn, cs);
            rb_tip_grad<N>(p, sn, cs, cost_w + RB_CW_TIP * RB_MAX_N, horizon > 0 ? dt : 0.0, 1.0, aq);
        }
    } else {
        auto add = [&](const double* g, size_t off, double (&acc)[N]) {
            if (!g) return;
#pragma unroll
            for (int i = 0; i < N; ++i) acc[i] += __ldcs(g + off + (size_t)i * ld + s);
        };
        add(g_qf, 0, aq);
        add(g_dqf, 0, adq);
        if (horizon > 0) { add(g_q, (size_t)(horizon - 1) * step, aq); add(g_dq, (size_t)(horizon - 1) * step, adq); }
    }
    bool ok = true;
#pragma unroll 1
    for (int t = horizon - 1; t >= 0; --t) {
        if (t > 0) {                                          // the state before step t
            rb_load<N>(q_traj + (size_t)(t - 1) * step_x, ld_traj, s, x);
            rb_load<N>(dq_traj + (size_t)(t - 1) * step_x, ld_traj, s, xd);
        } else {
            rb_load<N>(q0, ld, s, x);
            rb_load<N>(dq0, ld, s, xd);
        }
        double sn[N], cs[N], qdd[N], mu[N];
        rb_sincos_all<N>(x, sn, cs);
        {
            double Hm[N][N], dinv[N];
            rb_rnea<M, false>(p, sn, cs, xd, xd /*unused*/, qdd);
            rb_load<N>(tau + (size_t)t * step, ld, s, x);                   // u_t (x is reloaded below where needed)
#pragma unroll
            for (int i = 0; i < N; ++i) {
                qdd[i] = x[i] - qdd[i];
                adq[i] = fma(dt, aq[i], adq[i]);                            // b
                mu[i] = dt * adq[i];
            }
            rb_crba<M>(p, sn, cs, Hm);
            ok = rb_ldlt_factor<N>(Hm, dinv) && ok;
            rb_ldlt_apply<N>(Hm, dinv, qdd);
            rb_ldlt_apply<N>(Hm, dinv, mu);
        }
        if (grad_tau) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                double gt = mu[i];
                if constexpr (QUAD) gt = fma(2.0 * dt, w(RB_CW_TAU, i) * __ldcs(tau + (size_t)t * step + (size_t)i * ld + s), gt);
                __stcs(grad_tau + (size_t)t * step + (size_t)i * ld + s, gt);
            }
        }
        if constexpr (COL) rb_rnea_vjp<N, true, true>(p, sn, cs, xd, qdd, mu, aq, adq, cost_w + RB_CW_TIP * RB_MAX_N, t > 0 ? dt : 0.0,
                                                      cost_w + RB_CW_COL);
        else if constexpr (TIP) rb_rnea_vjp<N, true>(p, sn, cs, xd, qdd, mu, aq, adq, cost_w + RB_CW_TIP * RB_MAX_N, t > 0 ? dt : 0.0);
        else rb_rnea_vjp<N>(p, sn, cs, xd, qdd, mu, aq, adq);             // a_q -= (d tau/d q)^T mu,  a_dq = b - (d tau/d dq)^T mu
        if (t > 0) {                                          // upstream gradients of the state before step t
            if constexpr (QUAD) {
                rb_load<N>(q_traj + (size_t)(t - 1) * step_x, ld_traj, s, x);
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    aq[i] = fma(2.0 * dt, w(RB_CW_Q, i) * (x[i] - w(RB_CW_QREF, i)), aq[i]);
                    adq[i] = fma(2.0 * dt, w(RB_CW_DQ, i) * xd[i], adq[i]);
                }
            } else {
                if (g_q) {
#pragma unroll
                    for (int i = 0; i < N; ++i) aq[i] += __ldcs(g_q + (size_t)(t - 1) * step + (size_t)i * ld + s);
                }
                if (g_dq) {
#pragma unroll
                    for (int i = 0; i < N; ++i) adq[i] += __ldcs(g_dq + (size_t)(t - 1) * step + (size_t)i * ld + s);
                }
            }
        }
    }
    if (!ok) {
        atomicOr(status, RB_STATUS_NOT_SPD);
#pragma unroll
        for (int i = 0; i < N; ++i) { aq[i] = rb_nan<double>(); adq[i] = rb_nan<double>(); }
        if (grad_tau)
#pragma unroll 1
            for (int t = 0; t < horizon; ++t) rb_store<N>(grad_tau + (size_t)t * step, ld, s, aq);
    }
    if (grad_q0) rb_store<N>(grad_q0, ld, s, aq);
    if (grad_dq0) rb_store<N>(grad_dq0, ld, s, adq);
}

namespace {
unsigned dgrid(size_t B) { return (unsigned)((B + RB_BLOCK - 1) / RB_BLOCK); }
template <int N>
cudaError_t launch_rnea(const double* flat, const double* q, const double* dq, const double* ddq, double* out, size_t B, size_t ld, cudaStream_t st) {
    RbModelK<N> p;
    memcpy(&p, flat, sizeof(p));
    rb_rnea_deriv_kernel<N><<<dgrid(B), RB_BLOCK, 0, st>>>(p, q, dq, ddq, out, B, ld);
    return cudaGetLastError();
}
template <int N>
cudaError_t launch_fd(const double* flat, const double* q, const double* dq, const double* tau, double* out, size_t B, size_t ld, int* status, cudaStream_t st) {
    RbModelK<N> p;
    memcpy(&p, flat, sizeof(p));
    rb_fd_deriv_kernel<N><<<dgrid(B), RB_BLOCK, 0, st>>>(p, q, dq, tau, out, B, ld, status);
    return cudaGetLastError();
}
// The cost instantiations (QUAD) form their upstream gradients from cost_w; the plain vector-Jacobian product reads g_*.
template <int N, bool QUAD, bool TIP = false, bool COL = false>
cudaError_t launch_adjoint_as(const RbModelK<N>& p, const RbAdjointArgs& a, size_t B, size_t ld, int* status, cudaStream_t st) {
    rb_rollout_adjoint_kernel<N, QUAD, TIP, COL><<<dgrid(B), RB_BLOCK, 0, st>>>(
        p, a.q0, a.dq0, a.tau, a.q_traj, a.dq_traj, a.ld_traj, QUAD ? nullptr : a.g_q, QUAD ? nullptr : a.g_dq,
        QUAD ? nullptr : a.g_qf, QUAD ? nullptr : a.g_dqf, QUAD ? a.cost_w : nullptr, a.grad_tau, a.grad_q0, a.grad_dq0,
        a.dt, a.horizon, B, ld, status);
    return cudaGetLastError();
}
template <int N>
cudaError_t launch_adjoint(const double* flat, const RbAdjointArgs& a, size_t B, size_t ld, int* status, cudaStream_t st) {
    RbModelK<N> p;
    memcpy(&p, flat, sizeof(p));
    if (a.cost_w) switch (a.terms) {
        case RB_COST_TIP_COL: return launch_adjoint_as<N, true, true, true>(p, a, B, ld, status, st);
        case RB_COST_TIP: return launch_adjoint_as<N, true, true>(p, a, B, ld, status, st);
        case RB_COST_QUAD: return launch_adjoint_as<N, true>(p, a, B, ld, status, st);
    }
    return launch_adjoint_as<N, false>(p, a, B, ld, status, st);
}
}  // namespace

#define RB_DERIV_CASES(F, ...) \
    switch (n) { \
        case 1: return F<1>(__VA_ARGS__); case 2: return F<2>(__VA_ARGS__); case 3: return F<3>(__VA_ARGS__); \
        case 4: return F<4>(__VA_ARGS__); case 5: return F<5>(__VA_ARGS__); case 6: return F<6>(__VA_ARGS__); \
        case 7: return F<7>(__VA_ARGS__); case 8: return F<8>(__VA_ARGS__); case 9: return F<9>(__VA_ARGS__); \
        case 10: return F<10>(__VA_ARGS__); case 11: return F<11>(__VA_ARGS__); case 12: return F<12>(__VA_ARGS__); \
        default: return cudaErrorInvalidValue; \
    }

cudaError_t rb_launch_rnea_deriv(int n, const double* flat_model, const double* q, const double* dq, const double* ddq,
                                 double* out, size_t B, size_t ld, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    switch (n) {                                             // the rolled recursion has no per-joint state: any length
        case 13: return launch_rnea<13>(flat_model, q, dq, ddq, out, B, ld, st); case 14: return launch_rnea<14>(flat_model, q, dq, ddq, out, B, ld, st);
        case 15: return launch_rnea<15>(flat_model, q, dq, ddq, out, B, ld, st); case 16: return launch_rnea<16>(flat_model, q, dq, ddq, out, B, ld, st);
        case 17: return launch_rnea<17>(flat_model, q, dq, ddq, out, B, ld, st); case 18: return launch_rnea<18>(flat_model, q, dq, ddq, out, B, ld, st);
        case 19: return launch_rnea<19>(flat_model, q, dq, ddq, out, B, ld, st); case 20: return launch_rnea<20>(flat_model, q, dq, ddq, out, B, ld, st);
        case 21: return launch_rnea<21>(flat_model, q, dq, ddq, out, B, ld, st); case 22: return launch_rnea<22>(flat_model, q, dq, ddq, out, B, ld, st);
        case 23: return launch_rnea<23>(flat_model, q, dq, ddq, out, B, ld, st); case 24: return launch_rnea<24>(flat_model, q, dq, ddq, out, B, ld, st);
        case 25: return launch_rnea<25>(flat_model, q, dq, ddq, out, B, ld, st); case 26: return launch_rnea<26>(flat_model, q, dq, ddq, out, B, ld, st);
        case 27: return launch_rnea<27>(flat_model, q, dq, ddq, out, B, ld, st); case 28: return launch_rnea<28>(flat_model, q, dq, ddq, out, B, ld, st);
        case 29: return launch_rnea<29>(flat_model, q, dq, ddq, out, B, ld, st); case 30: return launch_rnea<30>(flat_model, q, dq, ddq, out, B, ld, st);
        case 31: return launch_rnea<31>(flat_model, q, dq, ddq, out, B, ld, st); case 32: return launch_rnea<32>(flat_model, q, dq, ddq, out, B, ld, st);
        default: break;
    }
    RB_DERIV_CASES(launch_rnea, flat_model, q, dq, ddq, out, B, ld, st)
}
cudaError_t rb_launch_fd_deriv(int n, const double* flat_model, const double* q, const double* dq, const double* tau,
                               double* out, size_t B, size_t ld, int* status, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    RB_DERIV_CASES(launch_fd, flat_model, q, dq, tau, out, B, ld, status, st)
}
cudaError_t rb_launch_rollout_adjoint(int n, const double* flat_model, const RbAdjointArgs& a, size_t B, size_t ld, int* status,
                                      cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    RB_DERIV_CASES(launch_adjoint, flat_model, a, B, ld, status, st)
}
