// rb_kernels_n.cu -- run-time-n kernel family ("generic-n") + the small utility kernels of the engine
// (sampler fill, AoS<->SoA transposes, FP64 peak probe).
//
// generic-n: persistent grid-stride kernels; the model rows sit in global memory (uniform loads, cached in
// L1/constant path); per-thread per-link state goes to a strided scratch [slot][thread] in HBM.
#include <atomic>
#include "rb_kernels.cuh"
#include "rb_dyn_n.cuh"
#include "rb_util.cuh"
#include <cstdlib>
#include <cstring>

int rb_rollout_mode() {
    const char* e = getenv("RIGIDBODY_B200_ROLLOUT");      // read per launch (tests flip it inside one process)
    return e && strcmp(e, "ws") == 0 ? 2 : 0;
}

__global__ void __launch_bounds__(RB_BLOCK)
rbn_rnea_kernel(RbNParam P, const double* __restrict__ q, const double* __restrict__ dq, const double* __restrict__ ddq,
                double* __restrict__ tau, size_t B, size_t ld) {
    const size_t tid = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * RB_BLOCK;
    const int n = P.n;
    const RbJointK* jt = reinterpret_cast<const RbJointK*>(P.model);
    const double* g = P.model + (size_t)n * 24;
    RbScratch sc{P.scratch + tid, P.threads};
    for (size_t s = tid; s < B; s += nthr) {
        for (int i = 0; i < n; ++i) {
            double sn, cs;
            sincos(__ldcs(q + (size_t)i * ld + s), &sn, &cs);
            sc[i] = sn; sc[n + i] = cs;
        }
        RbScratch out{tau + s, ld};
        if (P.tree) rbn_tree_rnea(jt, g, n, sc, RbScratch{P.scratch + tid + (size_t)(8 * n) * P.threads, P.threads}, dq + s, ddq + s, ld, out);
        else rbn_rnea(jt, g, n, sc, dq + s, ddq + s, ld, out);
    }
}

// ---- forward dynamics for long chains, two kernels per chunk of states ----------------------------------------
// A 32-joint mass matrix is 528 doubles: no thread can hold it, and factorising it in a per-thread global scratch
// costs O(n^3) HBM accesses per state (the first version of this family did that: 0.027 G states/s for n = 32).  Instead:
//   1. rbn_fd_prepare_kernel (thread per state, persistent): sin/cos, bias forces -> rhs = tau - rnea(q,dq,0)
//      written into qdd, CRBA -> packed upper triangle of H streamed ONCE to HBM, tile-major
//      ([state / 32][k][state % 32]: a warp writes 256-byte runs and a tile's 135 KB are contiguous);
//   2. rbn_ldlt_tile_kernel: a warp pulls a tile of TS states (all n(n+1)/2 rows, 256-byte runs) into shared
//      memory, lane = state, and runs the dot-product (Crout) LDL^T + both triangular solves entirely on chip:
//      2 shared loads per FMA, no bank conflicts ([k][lane] layout), H read from HBM exactly once.
// HBM traffic per state: 2 * n(n+1)/2 * 8 B for H (8.4 KB at n = 32) + the 32 n algorithmic bytes.
__global__ void __launch_bounds__(RB_BLOCK)
rbn_fd_prepare_kernel(RbNParam P, const double* __restrict__ q, const double* __restrict__ dq, const double* __restrict__ tau,
                      double* __restrict__ qdd, size_t B, size_t ld) {
    const size_t tid = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * RB_BLOCK;
    const int n = P.n;
    const RbJointK* jt = reinterpret_cast<const RbJointK*>(P.model);
    const double* g = P.model + (size_t)n * 24;
    RbScratch sc{P.scratch + tid, P.threads};
    for (size_t s = tid; s < B; s += nthr) {          // B <= P.hpk_states: s doubles as the chunk-local index
        for (int i = 0; i < n; ++i) {
            double sn, cs;
            sincos(__ldcs(q + (size_t)i * ld + s), &sn, &cs);
            sc[i] = sn; sc[n + i] = cs;
        }
        RbScratch x{qdd + s, ld};
        const RbScratch va{P.scratch + tid + (size_t)(8 * n) * P.threads, P.threads};   // trees: link motions, then composites
        if (P.tree) rbn_tree_rnea(jt, g, n, sc, va, dq + s, nullptr, ld, x);  // bias
        else rbn_rnea(jt, g, n, sc, dq + s, nullptr, ld, x);
        for (int i = 0; i < n; ++i) x[i] = __ldcs(tau + (size_t)i * ld + s) - x[i];
        double* hp = P.hpk + (s >> 5) * (size_t)(n * (n + 1) / 2) * 32 + (s & 31);    // tile-major: [s / 32][k][s % 32]
        auto put = [&](int r, int c, double v) { __stcs(hp + (size_t)(r * n - r * (r - 1) / 2 + (c - r)) * 32, v); };
        if (P.tree) rbn_tree_crba(jt, n, sc, va, put);
        else rbn_crba(jt, n, sc, put);
    }
}

// One block = RB_TILE_WARPS warps sharing one tile of TS states; lane = state, warps split the columns.
// Shared memory, all [row][TS]:
//   S : row j holds entries (j, j..n) of the augmented matrix [H | rhs] (column n = right-hand side), packed:
//       entry (j, i) at rowp(j) + i with rowp(j) = j (n + 1) - j (j - 1) / 2 - j;
//   M0, M1 : the multipliers of the current / next row (double-buffered), n each;   DI : 1 / d_j.
// The tile arrives through cp.async (8 bytes per lane per row, every row of the tile in flight at once).
// Factorisation (dot-product / Crout form of H = U^T D U, S = D U): for row j and every column i in [j, n]
//   S(j, i) = A(j, i) - sum_{k<j} m_k S(k, i),   m_k = S(k, j) / d_k,   d_j = S(j, j)
// so the rhs column comes out as D U x (forward substitution for free).  One block barrier per row: the
// multipliers of row j+1 that do not depend on row j are produced while row j is being computed, the last one
// (k = j) is recomputed by every warp after the barrier.
#ifndef RB_TILE_WARPS
#define RB_TILE_WARPS 8
#endif
template <int TS>
__global__ void __launch_bounds__(32 * RB_TILE_WARPS)
rbn_ldlt_tile_kernel(int n, const double* __restrict__ hpk, size_t hpk_states, double* __restrict__ qdd, size_t B, size_t ld,
                     int* __restrict__ status) {
    extern __shared__ double rb_tile[];
    constexpr int W = RB_TILE_WARPS;
    const int np1 = n * (n + 1) / 2 + n;                         // rows of S
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double* S = rb_tile + lane;                                  // this lane's column of every row
    double* Mb[2] = {S + (size_t)np1 * TS, S + (size_t)(np1 + n) * TS};
    double* DI = S + (size_t)(np1 + 2 * n) * TS;
    const size_t tiles = (B + TS - 1) / TS;
    auto rowp = [&](int j) { return j * (n + 1) - j * (j - 1) / 2 - j; };
    bool all_ok = true;
    for (size_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const size_t s = tile * TS + lane;
        const bool live = lane < TS && s < B;
        if (live) {
            for (int j = w; j < n; j += W) {                     // warp w fetches rows w, w + W, ...
                // packed (j, j) of this state's 32-state tile: rows of one tile are contiguous in HBM
                const double* src = hpk + ((s >> 5) * (size_t)(n * (n + 1) / 2) + (size_t)(j * n - j * (j - 1) / 2)) * 32 + (s & 31);
                double* dst = S + (size_t)(rowp(j) + j) * TS;
                for (int i = j; i < n; ++i, src += 32, dst += TS) {
                    const uint32_t d32 = (uint32_t)__cvta_generic_to_shared(dst);
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d32), "l"(src) : "memory");
                }
                const uint32_t d32 = (uint32_t)__cvta_generic_to_shared(dst);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d32), "l"(qdd + (size_t)j * ld + s) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        bool ok = true;
        for (int j = 0; j < n; ++j) {
            double* Mcur = Mb[j & 1];
            double* Mnxt = Mb[(j + 1) & 1];
            if (live) {
                // last multiplier of this row (depends on row j-1, finished at the barrier): every warp, redundantly
                if (j > 0) {
                    const double m = S[(size_t)(rowp(j - 1) + j) * TS] * DI[(size_t)(j - 1) * TS];
                    // columns j + w, j + w + W, ... <= n, two per pass (independent accumulator chains)
                    for (int i = j + w; i <= n; i += 2 * W) {
                        const bool two = i + W <= n;
                        const int off1 = two ? W * TS : 0;
                        double* pj = S + (size_t)(rowp(j) + i) * TS;
                        double a0 = pj[0], a1 = pj[off1];
                        const double* pk = S + (size_t)i * TS;        // (0, i); row k+1 starts n - k doubles later
                        const double* pm = Mcur;
                        int step = n * TS;
#pragma unroll 4
                        for (int k = 0; k < j - 1; ++k) {
                            const double mk = *pm;
                            a0 = fma(-mk, pk[0], a0);
                            a1 = fma(-mk, pk[off1], a1);
                            pk += step; step -= TS; pm += TS;
                        }
                        a0 = fma(-m, pk[0], a0);                       // k = j - 1 with the freshly computed multiplier
                        a1 = fma(-m, pk[off1], a1);
                        pj[0] = a0;
                        if (two) pj[off1] = a1;
                        if (i == j) { ok = ok && (a0 > 0.0); DI[(size_t)j * TS] = 1.0 / a0; }
                    }
                } else if (w == 0) {
                    const double d = S[0];
                    ok = ok && (d > 0.0);
                    DI[0] = 1.0 / d;
                }
                // multipliers of row j + 1 that only need rows < j:  m_k = S(k, j + 1) / d_k
                if (j + 1 < n)
                    for (int k = w; k < j; k += W) Mnxt[(size_t)k * TS] = S[(size_t)(rowp(k) + j + 1) * TS] * DI[(size_t)k * TS];
            }
            __syncthreads();
        }
        // back substitution, column-oriented so the warps split the rows.  X_k := S(k, n) = (D U x)_k:
        //   for k = n-1..0: x_k = X_k / d_k (final);  every i < k: X_i -= S(i, k) x_k
        bool okv = true;
        if (live)
            for (int j = 0; j < n; ++j) { const double v = DI[(size_t)j * TS]; okv = okv && (v > 0.0) && (v < 1.0e300); }
        for (int k = n - 1; k >= 0; --k) {
            if (live) {
                const double xk = S[(size_t)(rowp(k) + n) * TS] * DI[(size_t)k * TS];
                for (int i = w; i < k; i += W) {
                    double* xi = S + (size_t)(rowp(i) + n) * TS;
                    *xi = fma(-S[(size_t)(rowp(i) + k) * TS], xk, *xi);
                }
                if (w == (k & (W - 1))) __stcs(qdd + (size_t)k * ld + s, okv ? xk : __longlong_as_double(0x7ff8000000000000LL));
            }
            __syncthreads();
        }
        all_ok = all_ok && okv;
    }
    if (!all_ok) atomicOr(status, RB_STATUS_NOT_SPD);
}

__global__ void __launch_bounds__(RB_BLOCK)
rbn_crba_kernel(RbNParam P, const double* __restrict__ q, double* __restrict__ Hout, size_t B, size_t ld) {
    const size_t tid = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * RB_BLOCK;
    const int n = P.n;
    const RbJointK* jt = reinterpret_cast<const RbJointK*>(P.model);
    RbScratch sc{P.scratch + tid, P.threads};
    for (size_t s = tid; s < B; s += nthr) {
        for (int i = 0; i < n; ++i) {
            double sn, cs;
            sincos(__ldcs(q + (size_t)i * ld + s), &sn, &cs);
            sc[i] = sn; sc[n + i] = cs;
        }
        for (int c = 0; c < n; ++c)
            for (int r = c + 1; r < n; ++r) __stcs(Hout + (size_t)(r + n * c) * ld + s, 0.0);
        auto put = [&](int r, int c, double v) { __stcs(Hout + (size_t)(r + n * c) * ld + s, v); };
        if (P.tree) rbn_tree_crba(jt, n, sc, RbScratch{P.scratch + tid + (size_t)(8 * n) * P.threads, P.threads}, put);
        else rbn_crba(jt, n, sc, put);
    }
}

__global__ void __launch_bounds__(RB_BLOCK)
rbn_fk_jac_kernel(RbNParam P, const double* __restrict__ q, double* __restrict__ xyz, double* __restrict__ Jout,
                  size_t B, size_t ld) {
    const size_t tid = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * RB_BLOCK;
    const int n = P.n;
    const RbJointK* jt = reinterpret_cast<const RbJointK*>(P.model);
    for (size_t s = tid; s < B; s += nthr) {
        double A[3][3], r[3];
        if (Jout && P.tree)                              // joints that do not support the tip (last link): zero columns
            for (int k = 0; k < 6 * n; ++k) __stcs(Jout + (size_t)k * ld + s, 0.0);
        rbn_tip_pose(jt, P.model + (size_t)n * 24 + 3, n,
                     [&](int i, double* sn, double* cs) { sincos(__ldcs(q + (size_t)i * ld + s), sn, cs); },
                     [&](int i, const double (&A)[3][3], const double (&r)[3]) {
                         if (!Jout) return;
#pragma unroll
                         for (int k = 0; k < 3; ++k) {
                             __stcs(Jout + (size_t)(k + 6 * i) * ld + s, fma(A[1][k], r[0], -(A[0][k] * r[1])));
                             __stcs(Jout + (size_t)(3 + k + 6 * i) * ld + s, A[2][k]);
                         }
                     }, A, r);
        if (xyz) {
            __stcs(xyz + s, r[0]); __stcs(xyz + ld + s, r[1]); __stcs(xyz + 2 * ld + s, r[2]);
        }
    }
}

// Running and terminal tip-pose terms (rb_tip_terms) of a state whose sin/cos sincos_i gives, with the run-time-n tip pose.
template <class SinCos>
RB_DI void rbn_tip_terms(const RbNParam& P, SinCos&& sincos_i, const double* tw, double& run, double& fin) {
    double R[3][3], x[3];
    rbn_tip_pose(reinterpret_cast<const RbJointK*>(P.model), P.model + (size_t)P.n * 24 + 3, P.n, sincos_i,
                 [](int, const double (&)[3][3], const double (&)[3]) {}, R, x);
    rb_tip_terms(R, x, tw, run, fin);
}

// scratch slots: [0,2n) sincos, [2n,8n) f, (trees: [8n,20n) link motions / composites,) then n*n H, n rhs/x, n dinv,
// 2n carried (q, dq).  tip != 0 adds the tip-pose terms of RbTipCost (row RB_CW_TIP of cost_w), each running term of
// q_t from the sin/cos step t computes for q_t, as rb_rollout_kernel does; COL (with tip) adds the collision-sphere
// terms of RbCollisionCost (the block at cost_w + RB_CW_COL) on the same schedule.  The per-step solve
// still factorises H in the per-thread global scratch (slow for long chains; rollouts of long chains are not a
// BASELINE.json configuration).
template <bool COL = false>
__global__ void __launch_bounds__(RB_BLOCK)
rbn_rollout_kernel(RbNParam P, const double* __restrict__ q0, const double* __restrict__ dq0, const double* __restrict__ tau,
                   double dt, int horizon, double* __restrict__ q_traj, double* __restrict__ dq_traj,
                   double* __restrict__ q_fin, double* __restrict__ dq_fin, size_t B, size_t ld, int* __restrict__ status,
                   const double* __restrict__ cost_w, double* __restrict__ cost, int tip) {
    const size_t tid = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * RB_BLOCK;
    const int n = P.n;
    const RbJointK* jt = reinterpret_cast<const RbJointK*>(P.model);
    const double* g = P.model + (size_t)n * 24;
    RbScratch sc{P.scratch + tid, P.threads};
    auto sc_sincos = [&](int i, double* sn, double* cs) { *sn = sc[i]; *cs = sc[n + i]; };
    const int o = P.tree ? 20 * n : 8 * n;           // trees keep 12n link motions / 9n composites at [8n, 20n)
    RbScratch va{P.scratch + tid + (size_t)(8 * n) * P.threads, P.threads};
    RbScratch Hs{P.scratch + tid + (size_t)o * P.threads, P.threads};
    RbScratch x{P.scratch + tid + (size_t)(o + n * n) * P.threads, P.threads};
    RbScratch dinv{P.scratch + tid + (size_t)(o + n + n * n) * P.threads, P.threads};
    RbScratch qs{P.scratch + tid + (size_t)(o + 2 * n + n * n) * P.threads, P.threads};
    RbScratch dqs{P.scratch + tid + (size_t)(o + 3 * n + n * n) * P.threads, P.threads};
    const size_t step = (size_t)n * ld;
    bool all_ok = true;
    for (size_t s = tid; s < B; s += nthr) {
        for (int i = 0; i < n; ++i) { qs[i] = q0[(size_t)i * ld + s]; dqs[i] = dq0[(size_t)i * ld + s]; }
        double J = 0.0;
        bool ok_s = true;
        for (int t = 0; t < horizon; ++t) {
            for (int i = 0; i < n; ++i) {
                double sn, cs;
                sincos(qs[i], &sn, &cs);
                sc[i] = sn; sc[n + i] = cs;
            }
            if (tip && t > 0) {                          // running tip terms of q_t
                double run, fin;
                rbn_tip_terms(P, sc_sincos, cost_w + RB_CW_TIP * RB_MAX_N, run, fin);
                J = fma(dt, run, J);
                if constexpr (COL) J = fma(dt, cost_w[RB_CW_COL + RB_CL_W] * rbn_col_phi(jt, n, sc_sincos, cost_w + RB_CW_COL), J);
            }
            if (P.tree) rbn_tree_rnea(jt, g, n, sc, va, dqs.base, nullptr, dqs.stride, x);
            else rbn_rnea(jt, g, n, sc, dqs.base, nullptr, dqs.stride, x);
            for (int i = 0; i < n; ++i) x[i] = __ldcs(tau + (size_t)t * step + (size_t)i * ld + s) - x[i];
            auto put = [&](int r, int c, double v) { Hs[r * n + c] = v; };
            if (P.tree) rbn_tree_crba(jt, n, sc, va, put);
            else rbn_crba(jt, n, sc, put);
            ok_s = rbn_ldlt_solve(n, Hs, x, dinv) && ok_s;
            double c = 0.0;
            for (int i = 0; i < n; ++i) {
                const double dqn = fma(dt, x[i], dqs[i]);
                const double qn = fma(dt, dqn, qs[i]);
                dqs[i] = dqn; qs[i] = qn;
                if (q_traj) __stcs(q_traj + (size_t)t * step + (size_t)i * ld + s, qn);
                if (dq_traj) __stcs(dq_traj + (size_t)t * step + (size_t)i * ld + s, dqn);
                if (cost) {
                    const double e = qn - cost_w[RB_CW_QREF * RB_MAX_N + i];
                    const double u = __ldcs(tau + (size_t)t * step + (size_t)i * ld + s);
                    c = fma(cost_w[RB_CW_Q * RB_MAX_N + i] * e, e, c);
                    c = fma(cost_w[RB_CW_DQ * RB_MAX_N + i] * dqn, dqn, c);
                    c = fma(cost_w[RB_CW_TAU * RB_MAX_N + i] * u, u, c);
                }
            }
            J = fma(dt, c, J);
        }
        all_ok = all_ok && ok_s;
        if (cost) {
            for (int i = 0; i < n; ++i) {
                const double e = qs[i] - cost_w[RB_CW_QREF * RB_MAX_N + i];
                J = fma(cost_w[RB_CW_QF * RB_MAX_N + i] * e, e, J);
                J = fma(cost_w[RB_CW_DQF * RB_MAX_N + i] * dqs[i], dqs[i], J);
            }
            if (tip) {                                   // q_H: its running term (horizon > 0) and the terminal term
                double run, fin;
                rbn_tip_terms(P, [&](int i, double* sn, double* cs) { sincos(qs[i], sn, cs); }, cost_w + RB_CW_TIP * RB_MAX_N, run, fin);
                if (horizon > 0) J = fma(dt, run, J);
                J += fin;
                if constexpr (COL) {
                    const double phi = rbn_col_phi(jt, n, [&](int i, double* sn, double* cs) { sincos(qs[i], sn, cs); }, cost_w + RB_CW_COL);
                    if (horizon > 0) J = fma(dt, cost_w[RB_CW_COL + RB_CL_W] * phi, J);
                    J = fma(cost_w[RB_CW_COL + RB_CL_WF], phi, J);
                }
            }
            __stcs(cost + s, ok_s ? J : __longlong_as_double(0x7ff8000000000000LL));
        }
        for (int i = 0; i < n; ++i) {
            if (q_fin) q_fin[(size_t)i * ld + s] = qs[i];
            if (dq_fin) dq_fin[(size_t)i * ld + s] = dqs[i];
        }
    }
    if (!all_ok) atomicOr(status, RB_STATUS_NOT_SPD);
}

// ---- rollout of serial chains of <= 32 joints: one forward-dynamics launch (rb_kernels_warp.cu) + one integration
// launch per step.  The per-thread factorisation of rbn_rollout_kernel touches O(n^3) scratch words per step; here the
// state (q, dq) and qdd of all trajectories live in three [n][B] scratch arrays between the launches.
// tip != NULL (the model, RbNParam::model) adds the tip-pose terms of the state reached: forward dynamics runs in
// another kernel, so the pose takes its own sin/cos of q_{t+1} here.  COL (with tip) adds the collision-sphere terms the same way.
template <bool COL = false>
__global__ void __launch_bounds__(RB_BLOCK)
rbn_euler_kernel(int n, double dt, double* __restrict__ qc, double* __restrict__ dqc, const double* __restrict__ qdd,
                 const double* __restrict__ tau_t, double* __restrict__ q_out, double* __restrict__ dq_out, size_t B, size_t ldc,
                 size_t ld, const double* __restrict__ cost_w, double* __restrict__ cost, int first, int last,
                 double* __restrict__ q_fin, double* __restrict__ dq_fin, const double* __restrict__ tip) {
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    double c = 0.0, term = 0.0;
    for (int i = 0; i < n; ++i) {
        const double dqn = fma(dt, qdd[(size_t)i * ldc + s], dqc[(size_t)i * ldc + s]);
        const double qn = fma(dt, dqn, qc[(size_t)i * ldc + s]);
        dqc[(size_t)i * ldc + s] = dqn; qc[(size_t)i * ldc + s] = qn;
        if (q_out) __stcs(q_out + (size_t)i * ld + s, qn);
        if (dq_out) __stcs(dq_out + (size_t)i * ld + s, dqn);
        if (last) {
            if (q_fin) q_fin[(size_t)i * ld + s] = qn;
            if (dq_fin) dq_fin[(size_t)i * ld + s] = dqn;
        }
        if (cost) {
            const double e = qn - cost_w[RB_CW_QREF * RB_MAX_N + i];
            const double u = __ldcs(tau_t + (size_t)i * ld + s);
            c = fma(cost_w[RB_CW_Q * RB_MAX_N + i] * e, e, c);
            c = fma(cost_w[RB_CW_DQ * RB_MAX_N + i] * dqn, dqn, c);
            c = fma(cost_w[RB_CW_TAU * RB_MAX_N + i] * u, u, c);
            if (last) {
                term = fma(cost_w[RB_CW_QF * RB_MAX_N + i] * e, e, term);
                term = fma(cost_w[RB_CW_DQF * RB_MAX_N + i] * dqn, dqn, term);
            }
        }
    }
    if (tip) {
        double R[3][3], x[3], run, fin;
        rbn_tip_pose(reinterpret_cast<const RbJointK*>(tip), tip + (size_t)n * 24 + 3, n,
                     [&](int i, double* sn, double* cs) { sincos(qc[(size_t)i * ldc + s], sn, cs); },
                     [](int, const double (&)[3][3], const double (&)[3]) {}, R, x);
        rb_tip_terms(R, x, cost_w + RB_CW_TIP * RB_MAX_N, run, fin);
        c += run;
        if (last) term += fin;
        if constexpr (COL) {
            const double* col = cost_w + RB_CW_COL;
            const double phi = rbn_col_phi(reinterpret_cast<const RbJointK*>(tip), n,
                                           [&](int i, double* sn, double* cs) { sincos(qc[(size_t)i * ldc + s], sn, cs); }, col);
            c = fma(col[RB_CL_W], phi, c);
            if (last) term = fma(col[RB_CL_WF], phi, term);
        }
    }
    if (cost) {
        const double J = fma(dt, c, first ? 0.0 : cost[s]);
        cost[s] = last ? J + term : J;                       // a non-SPD step leaves NaN in qdd, hence in q, hence here
    }
}

namespace {
unsigned ngrid(const RbNParam* P, size_t B) {
    size_t want = (B + RB_BLOCK - 1) / RB_BLOCK;
    size_t cap = P->threads / RB_BLOCK;
    return (unsigned)(want < cap ? want : cap);
}
cudaError_t n_rnea(const void* param, const double* q, const double* dq, const double* ddq, double* tau, size_t B, size_t ld, cudaStream_t st) {
    const RbNParam* P = (const RbNParam*)param;
    if (B == 0) return cudaSuccess;
    rbn_rnea_kernel<<<ngrid(P, B), RB_BLOCK, 0, st>>>(*P, q, dq, ddq, tau, B, ld);
    return cudaGetLastError();
}
template <int TS>
cudaError_t launch_tile(int n, const double* hpk, size_t hpk_states, double* qdd, size_t cnt, size_t ld, int* status,
                        size_t smem, int dev, int sms, cudaStream_t st) {
    // per device: largest dynamic shared-memory size opted into (atomic: handles may be created from several threads;
    // setting the attribute twice is harmless, a torn read is not)
    static std::atomic<size_t> configured[64];
    if (dev >= 0 && dev < 64 && smem > configured[dev].load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(rbn_ldlt_tile_kernel<TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[dev].store(smem, std::memory_order_release);
    }
    const size_t tiles = (cnt + TS - 1) / TS;
    size_t per_sm = (size_t)(220 * 1024) / (smem + 1024);
    per_sm = per_sm < 1 ? 1 : (per_sm > 16 ? 16 : per_sm);
    const size_t cap = (size_t)sms * per_sm;
    rbn_ldlt_tile_kernel<TS><<<(unsigned)(tiles < cap ? tiles : cap), 32 * RB_TILE_WARPS, smem, st>>>(n, hpk, hpk_states, qdd, cnt, ld, status);
    return cudaGetLastError();
}
}  // namespace

// Solves H x = rhs for `cnt` states: H packed upper in hpk ([n(n+1)/2][hpk_states]), rhs in qdd (overwritten by x).
cudaError_t rb_launch_ldlt_tiles(int n, const double* hpk, size_t hpk_states, double* qdd, size_t cnt, size_t ld,
                                 int* status, cudaStream_t st) {
    if (cnt == 0) return cudaSuccess;
    const size_t rows = (size_t)n * (n + 1) / 2 + 4 * (size_t)n;      // S (with the rhs column) + M0 + M1 + DI
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // widest tile whose shared-memory footprint fits one SM
    if (rows * 32 * sizeof(double) <= 200 * 1024) return launch_tile<32>(n, hpk, hpk_states, qdd, cnt, ld, status, rows * 32 * sizeof(double), dev, sms, st);
    if (rows * 16 * sizeof(double) <= 200 * 1024) return launch_tile<16>(n, hpk, hpk_states, qdd, cnt, ld, status, rows * 16 * sizeof(double), dev, sms, st);
    return launch_tile<8>(n, hpk, hpk_states, qdd, cnt, ld, status, rows * 8 * sizeof(double), dev, sms, st);
}

namespace {
cudaError_t n_fd(const void* param, const double* q, const double* dq, const double* tau, double* qdd, size_t B, size_t ld, int* status, cudaStream_t st) {
    const RbNParam* P = (const RbNParam*)param;
#if RB_WARP_FD
    if (P->n <= 32 && !P->tree)                                      // warp-per-state, nothing leaves the SM (rb_kernels_warp.cu)
        return rb_launch_warp_fd(P->model, P->n, q, dq, tau, qdd, B, ld, status, st);
#endif
    for (size_t off = 0; off < B; off += P->hpk_states) {
        const size_t cnt = (B - off < P->hpk_states) ? (B - off) : P->hpk_states;
        rbn_fd_prepare_kernel<<<ngrid(P, cnt), RB_BLOCK, 0, st>>>(*P, q + off, dq + off, tau + off, qdd + off, cnt, ld);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        e = rb_launch_ldlt_tiles(P->n, P->hpk, P->hpk_states, qdd + off, cnt, ld, status, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}
cudaError_t n_crba(const void* param, const double* q, double* H, size_t B, size_t ld, cudaStream_t st) {
    const RbNParam* P = (const RbNParam*)param;
    if (B == 0) return cudaSuccess;
    rbn_crba_kernel<<<ngrid(P, B), RB_BLOCK, 0, st>>>(*P, q, H, B, ld);
    return cudaGetLastError();
}
cudaError_t n_fk(const void* param, const double* q, double* xyz, size_t B, size_t ld, cudaStream_t st) {
    const RbNParam* P = (const RbNParam*)param;
    if (B == 0) return cudaSuccess;
    rbn_fk_jac_kernel<<<ngrid(P, B), RB_BLOCK, 0, st>>>(*P, q, xyz, nullptr, B, ld);
    return cudaGetLastError();
}
cudaError_t n_jac(const void* param, const double* q, double* J, size_t B, size_t ld, cudaStream_t st) {
    const RbNParam* P = (const RbNParam*)param;
    if (B == 0) return cudaSuccess;
    rbn_fk_jac_kernel<<<ngrid(P, B), RB_BLOCK, 0, st>>>(*P, q, nullptr, J, B, ld);
    return cudaGetLastError();
}
cudaError_t n_rollout_any(const void* param, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                          double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                          const double* cost_w, double* cost, bool tip, bool col, cudaStream_t st) {
    const RbNParam* P = (const RbNParam*)param;
    if (B == 0) return cudaSuccess;
#if RB_WARP_FD
    if (P->n <= 32 && !P->tree && horizon > 0) {
        const int n = P->n;
        const size_t cap = P->slots * P->threads / ((size_t)4 * n);          // trajectories the scratch holds at once
        for (size_t off = 0; off < B; off += cap) {
            const size_t cnt = B - off < cap ? B - off : cap;
            double* qc = P->scratch; double* dqc = qc + (size_t)n * cnt; double* tc = dqc + (size_t)n * cnt; double* acc = tc + (size_t)n * cnt;
            cudaError_t e = cudaMemcpy2DAsync(qc, cnt * sizeof(double), q0 + off, ld * sizeof(double), cnt * sizeof(double), n, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return e;
            e = cudaMemcpy2DAsync(dqc, cnt * sizeof(double), dq0 + off, ld * sizeof(double), cnt * sizeof(double), n, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return e;
            const size_t step = (size_t)n * ld;
            for (int t = 0; t < horizon; ++t) {
                const double* tau_t = tau + (size_t)t * step + off;
                // tau rows have stride ld, the carried state stride cnt: one kernel call wants one stride
                e = cudaMemcpy2DAsync(tc, cnt * sizeof(double), tau_t, ld * sizeof(double), cnt * sizeof(double), n, cudaMemcpyDeviceToDevice, st);
                if (e != cudaSuccess) return e;
                e = rb_launch_warp_fd(P->model, n, qc, dqc, tc, acc, cnt, cnt, status, st);
                if (e != cudaSuccess) return e;
                (col ? rbn_euler_kernel<true> : rbn_euler_kernel<false>)<<<(unsigned)((cnt + RB_BLOCK - 1) / RB_BLOCK), RB_BLOCK, 0, st>>>(
                    n, dt, qc, dqc, acc, tau_t, q_traj ? q_traj + (size_t)t * step + off : nullptr,
                    dq_traj ? dq_traj + (size_t)t * step + off : nullptr, cnt, cnt, ld, cost_w, cost ? cost + off : nullptr,
                    t == 0, t == horizon - 1, q_fin ? q_fin + off : nullptr, dq_fin ? dq_fin + off : nullptr, tip ? P->model : nullptr);
                e = cudaGetLastError();
                if (e != cudaSuccess) return e;
            }
        }
        return cudaSuccess;
    }
#endif
    (col ? rbn_rollout_kernel<true> : rbn_rollout_kernel<false>)<<<ngrid(P, B), RB_BLOCK, 0, st>>>(
        *P, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost, tip ? 1 : 0);
    return cudaGetLastError();
}
cudaError_t n_rollout(const void* param, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                      double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                      const double* cost_w, double* cost, cudaStream_t st) {
    return n_rollout_any(param, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost, false, false, st);
}
cudaError_t n_rollout_tip(const void* param, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                          double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                          const double* cost_w, double* cost, cudaStream_t st) {
    return n_rollout_any(param, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost, true, false, st);
}
cudaError_t n_rollout_col(const void* param, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                          double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                          const double* cost_w, double* cost, cudaStream_t st) {
    return n_rollout_any(param, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost, true, true, st);
}
}  // namespace

const RbOps* rb_ops_generic_n() {
    static const RbOps ops = [] {
        RbOps o{};
        o.name = "generic-n"; o.param_bytes = sizeof(RbNParam); o.shared_scratch = true;
        o.rnea = &n_rnea; o.fd = &n_fd; o.crba = &n_crba; o.fwd_kin = &n_fk; o.jac = &n_jac; o.rollout = &n_rollout;
        o.rollout_tip = &n_rollout_tip; o.rollout_col = &n_rollout_col;
        return o;
    }();
    return &ops;
}

// ------------------------------------------------------------------ utility kernels (declared in rb_util.cuh)
__global__ void rb_fill_kernel(double* __restrict__ out, uint64_t seed, uint32_t field, int n, RbFillRange rg,
                               size_t first, size_t count, size_t ld) {
    const size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= count) return;
    for (int i = 0; i < n; ++i) {
        const uint64_t ctr = ((uint64_t)field << 58) | ((uint64_t)i << 50) | ((first + s) & ((1ULL << 50) - 1));
        uint64_t z = seed + 0x9E3779B97F4A7C15ULL * (ctr + 1ULL);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        z = z ^ (z >> 31);
        const double u = (double)(z >> 11) * 0x1.0p-53;
        out[(size_t)i * ld + s] = fma(rg.hi[i] - rg.lo[i], u, rg.lo[i]);
    }
}

// [B][n] (AoS) <-> [n][ld] (SoA): `spb` states per block pass through shared memory so both the global reads
// and the global writes are contiguous runs.
__global__ void rb_aos_to_soa_kernel(const double* __restrict__ aos, double* __restrict__ soa, int n, size_t B, size_t ld, int spb) {
    extern __shared__ double tile[];               // [spb][n] as in memory
    const size_t s0 = (size_t)blockIdx.x * spb;
    const size_t cnt = (B - s0 < (size_t)spb) ? (B - s0) : (size_t)spb;
    const size_t tot = cnt * (size_t)n;
    for (size_t k = threadIdx.x; k < tot; k += blockDim.x) tile[k] = aos[s0 * n + k];
    __syncthreads();
    for (size_t k = threadIdx.x; k < tot; k += blockDim.x) {
        const size_t i = k / cnt, s = k % cnt;
        soa[i * ld + s0 + s] = tile[s * n + i];
    }
}
__global__ void rb_soa_to_aos_kernel(const double* __restrict__ soa, double* __restrict__ aos, int n, size_t B, size_t ld, int spb) {
    extern __shared__ double tile[];
    const size_t s0 = (size_t)blockIdx.x * spb;
    const size_t cnt = (B - s0 < (size_t)spb) ? (B - s0) : (size_t)spb;
    const size_t tot = cnt * (size_t)n;
    for (size_t k = threadIdx.x; k < tot; k += blockDim.x) {
        const size_t i = k / cnt, s = k % cnt;
        tile[s * n + i] = soa[i * ld + s0 + s];
    }
    __syncthreads();
    for (size_t k = threadIdx.x; k < tot; k += blockDim.x) aos[s0 * n + k] = tile[k];
}

// Register-only DFMA chains: 8 independent accumulators per thread, RB_PEAK_INNER fused multiply-adds each
// per outer iteration.  2 flops per DFMA.
__global__ void __launch_bounds__(256) rb_fp64_peak_kernel(double* out, int iters, double a_in, double b_in) {
    // multiplier and addend in REGISTERS: as kernel parameters they become constant-bank operands of every DFMA, and the
    // probe then reads 6 % below what the same chains reach with register operands (tools/ubench_fp64_peak.cu)
    double a, b;
    asm volatile("mov.f64 %0, %1;" : "=d"(a) : "d"(a_in));
    asm volatile("mov.f64 %0, %1;" : "=d"(b) : "d"(b_in));
    double x0 = threadIdx.x * 1e-9, x1 = x0 + 1.0, x2 = x0 + 2.0, x3 = x0 + 3.0;
    double x4 = x0 + 4.0, x5 = x0 + 5.0, x6 = x0 + 6.0, x7 = x0 + 7.0;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < RB_PEAK_INNER; ++k) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    const double r = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (r == 123.456) out[0] = r;   // keeps the chains live without a store in the common case
}

cudaError_t rb_launch_fill(double* out, uint64_t seed, uint32_t field, int n, const RbFillRange& rg,
                           size_t first, size_t count, size_t ld, cudaStream_t st) {
    if (count == 0) return cudaSuccess;
    rb_fill_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(out, seed, field, n, rg, first, count, ld);
    return cudaGetLastError();
}
static int rb_tr_spb(int n) { int spb = 4096 / n; return spb < 1 ? 1 : (spb > 128 ? 128 : spb); }
cudaError_t rb_launch_aos_to_soa(const double* aos, double* soa, int n, size_t B, size_t ld, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    const int spb = rb_tr_spb(n);
    rb_aos_to_soa_kernel<<<(unsigned)((B + spb - 1) / spb), 256, (size_t)spb * n * sizeof(double), st>>>(aos, soa, n, B, ld, spb);
    return cudaGetLastError();
}
cudaError_t rb_launch_soa_to_aos(const double* soa, double* aos, int n, size_t B, size_t ld, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    const int spb = rb_tr_spb(n);
    rb_soa_to_aos_kernel<<<(unsigned)((B + spb - 1) / spb), 256, (size_t)spb * n * sizeof(double), st>>>(soa, aos, n, B, ld, spb);
    return cudaGetLastError();
}
cudaError_t rb_launch_fp64_peak(double* out, int blocks, int threads, int iters, cudaStream_t st) {
    rb_fp64_peak_kernel<<<blocks, threads, 0, st>>>(out, iters, 0.999999, 1e-7);
    return cudaGetLastError();
}
