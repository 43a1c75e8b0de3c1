// rb_kernels.cuh -- __global__ kernels over SoA batches for an unrolled model policy M, and the RbOps
// table through which the C ABI (rb_api.cu) reaches whichever kernel family serves a chain.
//
// Data layout in HBM: joint-major SoA.  Array x of a batch is [n][ld] doubles; state s of joint i is
// x[i*ld + s].  Thread t of the grid owns state s = t: consecutive lanes read consecutive doubles, so each
// warp-level load/store is one fully used 256-byte run, and each array is streamed exactly once
// (ld.global.cs / st.global.cs, no reuse, no smem staging needed).
#pragma once
// RB_DEVICE_ONLY (defined by the run-time compiler, rb_jit.cu) drops everything that is host code: NVRTC
// compiles the kernels of this header for one uploaded chain and has neither the CUDA runtime API nor <stdint.h>.
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <type_traits>
#else
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef unsigned long uintptr_t;
#endif
#include "rb_dyn.cuh"

#ifndef RB_BLOCK
#define RB_BLOCK 128
#endif
// Minimum resident blocks per SM requested from ptxas (register cap = 65536 / (RB_BLOCK * min_blocks)).
#ifndef RB_MINB_RNEA
#define RB_MINB_RNEA 4     // 126 registers, no spills.  (5 blocks / 96 registers won by 4 % with the per-joint library sincos;
#endif                     //  with the batched sincos 4 blocks win by 3 %: profiles/r2_kbench_launch_bounds.jsonl)
#ifndef RB_MINB_FD
#define RB_MINB_FD 4
#endif
// The run-time-constant family executes ~1.7-2x the instructions with more live values: it wants more registers.
// chains of 9..12 joints (run-time specialised): fewer, fatter blocks (profiles/r1_kbench_jit_launch_bounds.txt)
#ifndef RB_MINB_RNEA_LONG
#define RB_MINB_RNEA_LONG 4
#endif
#ifndef RB_MINB_RNEA_XLONG
#define RB_MINB_RNEA_XLONG 3   // 15..18 joints
#endif
#ifndef RB_MINB_FD_LONG
#define RB_MINB_FD_LONG 2      // 12 joints: the 78-entry matrix wants all 255 registers
#endif
#ifndef RB_MINB_RNEA_RT
#define RB_MINB_RNEA_RT 3
#endif
#ifndef RB_MINB_FD_RT
#define RB_MINB_FD_RT 2
#endif
#ifndef RB_STREAM
#define RB_STREAM 0        // 1 = route full tiles through the persistent TMA-fed kernels (experiments/, measured slower)
#endif
#ifndef RB_PREFETCH
#define RB_PREFETCH 0      // 1 = persistent kernels with register prefetch (experiments/, measured slower)
#endif

#ifndef RB_DEVICE_ONLY
struct RbOps {
    const char* name;
    size_t param_bytes;    // bytes of model parameter the launchers expect behind `param`
    bool shared_scratch;   // kernels work in engine-owned scratch: launches must be ordered across streams
    cudaError_t (*rnea)(const void* param, const double* q, const double* dq, const double* ddq, double* tau,
                        size_t B, size_t ld, cudaStream_t st);
    cudaError_t (*fd)(const void* param, const double* q, const double* dq, const double* tau, double* qdd,
                      size_t B, size_t ld, int* status, cudaStream_t st);
    // optional: the same two on state-major AoS batches [B][n] (null = the API transposes around the SoA kernels)
    cudaError_t (*rnea_aos)(const void* param, const double* q, const double* dq, const double* ddq, double* tau,
                            size_t B, cudaStream_t st);
    cudaError_t (*fd_aos)(const void* param, const double* q, const double* dq, const double* tau, double* qdd,
                          size_t B, int* status, cudaStream_t st);
    cudaError_t (*crba)(const void* param, const double* q, double* H, size_t B, size_t ld, cudaStream_t st);
    cudaError_t (*fwd_kin)(const void* param, const double* q, double* xyz, size_t B, size_t ld, cudaStream_t st);
    cudaError_t (*jac)(const void* param, const double* q, double* J, size_t B, size_t ld, cudaStream_t st);
    cudaError_t (*rollout)(const void* param, const double* q0, const double* dq0, const double* tau, double dt,
                           int horizon, double* q_traj, double* dq_traj, double* q_fin, double* dq_fin,
                           size_t B, size_t ld, int* status, const double* cost_w, double* cost, cudaStream_t st);
    // the same rollout with the tip-pose terms of RbTipCost added to the cost (cost_w carries the RB_CW_TIP row)
    cudaError_t (*rollout_tip)(const void* param, const double* q0, const double* dq0, const double* tau, double dt,
                               int horizon, double* q_traj, double* dq_traj, double* q_fin, double* dq_fin,
                               size_t B, size_t ld, int* status, const double* cost_w, double* cost, cudaStream_t st);
    // ... with the collision-sphere terms of RbCollisionCost added as well (cost_w carries the tip row and the block at RB_CW_COL)
    cudaError_t (*rollout_col)(const void* param, const double* q0, const double* dq0, const double* tau, double dt,
                               int horizon, double* q_traj, double* dq_traj, double* q_fin, double* dq_fin,
                               size_t B, size_t ld, int* status, const double* cost_w, double* cost, cudaStream_t st);
    // optional fp32 mode (BASELINE.json: "an optional fp32 mode is held to a stated 1e-4 tolerance"): the same kernels
    // instantiated with Real = float, device-resident SoA batches only (null = family has no fp32 kernels)
    cudaError_t (*rnea_f32)(const void* param, const float* q, const float* dq, const float* ddq, float* tau,
                            size_t B, size_t ld, cudaStream_t st);
    cudaError_t (*fd_f32)(const void* param, const float* q, const float* dq, const float* tau, float* qdd,
                          size_t B, size_t ld, int* status, cudaStream_t st);
    // optional: tau = rnea(q, dq, ddq) and qdd = fd(q, dq, tau_in) in ONE pass over SoA batches, out = [2n][ld]
    // (null = the API issues the rnea and fd launches back to back)
    cudaError_t (*rnea_fd)(const void* param, const double* q, const double* dq, const double* ddq, const double* tau_in,
                           double* out, size_t B, size_t ld, int* status, cudaStream_t st);
};

// $RIGIDBODY_B200_ROLLOUT, read at every launch: "ws" = 2 selects the two-warp kernel of experiments/rb_rollout_ws.cuh
// in builds made with -DRB_ROLLOUT_WS=1; anything else = 0, the product kernel (rb_rollout_kernel).
int rb_rollout_mode();
const RbOps* rb_ops_fr3();        // compile-time FR3 model (rb_kernels_fr3.cu)
const RbOps* rb_ops_rt7();        // any 7-joint chain, run-time constants (rb_kernels_rt.cu)
const RbOps* rb_ops_generic_n();  // any chain length (rb_kernels_n.cu)
const double* rb_fr3_table();     // the 7x24 table + 3 gravity doubles the FR3 kernels were compiled for
const RbOps* rb_ops_chain32();    // compile-time 32-joint chain, long-chain layout (rb_kernels_c32.cu)
const double* rb_chain32_table();
#endif  // RB_DEVICE_ONLY

#define RB_STATUS_NOT_SPD 1

// Parameter block of the run-time-n family (rb_kernels_n.cu); rb_api.cu fills it when a chain is uploaded.
struct RbNParam {
    const double* model;     // device: n rows of 24 doubles + g[3] + tip[9]
    int n;
    double* scratch;         // per-thread strided scratch: `slots` doubles per thread, element k at scratch[k*threads + tid]
    size_t threads;          // threads the scratch was sized for (persistent grid * block)
    size_t slots;
    double* hpk;             // packed upper triangles of H for one chunk of states, tile-major [state / 32][n(n+1)/2][state % 32]
    size_t hpk_states;       // states per chunk
    int tree;                // 1 = some joint's parent is not the previous joint: rbn_tree_* recursions, no warp kernel
};

// Quiet NaN of the scalar type (marks states whose mass matrix was not positive definite).
template <class T> RB_DI T rb_nan();
template <> RB_DI double rb_nan<double>() { return __longlong_as_double(0x7ff8000000000000LL); }
template <> RB_DI float rb_nan<float>() { return __int_as_float(0x7fc00000); }

template <int N, class T>
RB_DI void rb_load(const T* __restrict__ x, size_t ld, size_t s, T (&v)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __ldcs(x + (size_t)i * ld + s);
}
template <int N, class T>
RB_DI void rb_store(T* __restrict__ x, size_t ld, size_t s, const T (&v)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) __stcs(x + (size_t)i * ld + s, v[i]);
}

// AoS batches ([B][N], the reference's RB_R[7] repeated): a block stages its RB_BLOCK states through shared
// memory so the global accesses stay contiguous runs; thread t then reads its N values at stride N (odd N: no
// bank conflicts).  No extra pass over HBM, unlike a separate transpose.
template <int N, class T>
RB_DI void rb_aos_load3(const T* __restrict__ x0, const T* __restrict__ x1, const T* __restrict__ x2,
                        size_t B, T* buf, T (&a)[N], T (&b)[N], T (&c)[N]) {
    const size_t base = (size_t)blockIdx.x * RB_BLOCK * N;
    const size_t rest = B * N - base;
    const int cnt = rest < (size_t)RB_BLOCK * N ? (int)rest : RB_BLOCK * N;
    T* b0 = buf; T* b1 = buf + RB_BLOCK * N; T* b2 = buf + 2 * RB_BLOCK * N;
    for (int k = threadIdx.x; k < cnt; k += RB_BLOCK) {
        b0[k] = __ldcs(x0 + base + k); b1[k] = __ldcs(x1 + base + k); b2[k] = __ldcs(x2 + base + k);
    }
    __syncthreads();
    const int o = threadIdx.x * N;
    if (o < cnt) {
#pragma unroll
        for (int i = 0; i < N; ++i) { a[i] = b0[o + i]; b[i] = b1[o + i]; c[i] = b2[o + i]; }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) { a[i] = T(0); b[i] = T(0); c[i] = T(0); }
    }
    __syncthreads();
}
template <int N, class T>
RB_DI void rb_aos_store(T* __restrict__ out, size_t B, T* buf, const T (&v)[N]) {
    const size_t base = (size_t)blockIdx.x * RB_BLOCK * N;
    const size_t rest = B * N - base;
    const int cnt = rest < (size_t)RB_BLOCK * N ? (int)rest : RB_BLOCK * N;
    const int o = threadIdx.x * N;
#pragma unroll
    for (int i = 0; i < N; ++i) buf[o + i] = v[i];
    __syncthreads();
    for (int k = threadIdx.x; k < cnt; k += RB_BLOCK) __stcs(out + base + k, buf[k]);
}

template <class M, bool AOS = false>
__global__ void __launch_bounds__(RB_BLOCK, !M::kSpecialised ? RB_MINB_RNEA_RT : (M::N <= 8 ? RB_MINB_RNEA : (M::N <= 14 ? RB_MINB_RNEA_LONG : (M::N <= 18 ? RB_MINB_RNEA_XLONG : 2))))
rb_rnea_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q, const RB_R* __restrict__ dq,
               const RB_R* __restrict__ ddq, RB_R* __restrict__ tau, size_t B, size_t ld) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    RB_R a[N], b[N], c[N], sn[N], cs[N], t[N];
    if constexpr (AOS) {
        extern __shared__ double rb_aos_raw[];
        RB_R* rb_aos_buf = reinterpret_cast<RB_R*>(rb_aos_raw);
        rb_aos_load3<N>(q, dq, ddq, B, rb_aos_buf, a, b, c);
        rb_sincos_all<N>(a, sn, cs);
        rb_rnea<M, true>(p, sn, cs, b, c, t);
        rb_aos_store<N>(tau, B, rb_aos_buf, t);
    } else {
        if (s >= B) return;
        rb_load<N>(q, ld, s, a);
        rb_load<N>(dq, ld, s, b);
        rb_load<N>(ddq, ld, s, c);
        rb_sincos_all<N>(a, sn, cs);
        rb_rnea<M, true>(p, sn, cs, b, c, t);
        rb_store<N>(tau, ld, s, t);
    }
}

template <class M, bool AOS = false>
__global__ void __launch_bounds__(RB_BLOCK, !M::kSpecialised ? RB_MINB_FD_RT : (M::N <= 11 ? RB_MINB_FD : RB_MINB_FD_LONG))
rb_fd_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q, const RB_R* __restrict__ dq,
             const RB_R* __restrict__ tau, RB_R* __restrict__ qdd, size_t B, size_t ld, int* __restrict__ status) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    RB_R a[N], b[N], c[N], sn[N], cs[N], x[N];
    if constexpr (AOS) {
        extern __shared__ double rb_aos_raw[];
        RB_R* rb_aos_buf = reinterpret_cast<RB_R*>(rb_aos_raw);
        rb_aos_load3<N>(q, dq, tau, B, rb_aos_buf, a, b, c);
    } else {
        if (s >= B) return;
        rb_load<N>(q, ld, s, a);
        rb_load<N>(dq, ld, s, b);
        rb_load<N>(tau, ld, s, c);
    }
    rb_sincos_all<N>(a, sn, cs);
    const bool ok = rb_forward_dynamics<M>(p, sn, cs, b, c, x);
    if (!ok) {
        if (s < B) atomicOr(status, RB_STATUS_NOT_SPD);     // padding threads of an AoS tail block do not count
#pragma unroll
        for (int i = 0; i < N; ++i) x[i] = rb_nan<RB_R>();
    }
    if constexpr (AOS) {
        extern __shared__ double rb_aos_raw[];
        RB_R* rb_aos_buf = reinterpret_cast<RB_R*>(rb_aos_raw);
        rb_aos_store<N>(qdd, B, rb_aos_buf, x);
    } else {
        rb_store<N>(qdd, ld, s, x);
    }
}

// Inverse + forward dynamics of the same states in one pass (multibody_rnea_fd_batch): 4n doubles in, 2n out
// (336 B per FR3 state instead of the 448 B of two launches), shared sin/cos, bias recursion and mass matrix
// (rb_rnea_fd_fused).  out holds tau in rows 0..n-1 and qdd in rows n..2n-1.
#ifndef RB_MINB_FUSED
#define RB_MINB_FUSED 3    // 168 registers, no spills (4 blocks: 128 registers, 148 B of spills, 2 % slower)
#endif
template <class M>
__global__ void __launch_bounds__(RB_BLOCK, !M::kSpecialised ? RB_MINB_FD_RT : (M::N <= 11 ? RB_MINB_FUSED : RB_MINB_FD_LONG))
rb_rnea_fd_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q, const RB_R* __restrict__ dq,
                  const RB_R* __restrict__ ddq, const RB_R* __restrict__ tau_in, RB_R* __restrict__ out,
                  size_t B, size_t ld, int* __restrict__ status) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    RB_R a[N], b[N], c[N], d[N], sn[N], cs[N], t[N], x[N];
    rb_load<N>(q, ld, s, a);
    rb_load<N>(dq, ld, s, b);
    rb_load<N>(ddq, ld, s, c);
    rb_load<N>(tau_in, ld, s, d);
    rb_sincos_all<N>(a, sn, cs);
    const bool ok = rb_rnea_fd_fused<M>(p, sn, cs, b, c, d, t, x);
    rb_store<N>(out, ld, s, t);
    if (!ok) {
        atomicOr(status, RB_STATUS_NOT_SPD);
#pragma unroll
        for (int i = 0; i < N; ++i) x[i] = rb_nan<RB_R>();
    }
    rb_store<N>(out + (size_t)N * ld, ld, s, x);
}

#if RB_STREAM || RB_PREFETCH
#include "experiments/rb_experiments.cuh"   // measured dead ends (DESIGN.md 4.5), not part of the default build
#endif

// H out: reference convention, n*n entries per state, entry k = r + n*c, upper filled, strict lower 0.
template <class M>
__global__ void __launch_bounds__(RB_BLOCK)
rb_crba_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q, RB_R* __restrict__ Hout,
               size_t B, size_t ld) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    RB_R a[N], sn[N], cs[N], H[N][N];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    rb_crba<M>(p, sn, cs, H);
#pragma unroll
    for (int c = 0; c < N; ++c)
#pragma unroll
        for (int r = 0; r < N; ++r) __stcs(Hout + (size_t)(r + N * c) * ld + s, r <= c ? H[r][c] : RB_R(0));
}

template <class M>
__global__ void __launch_bounds__(RB_BLOCK)
rb_fwd_kin_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q, RB_R* __restrict__ xyz,
                  size_t B, size_t ld) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    RB_R a[N], sn[N], cs[N], pos[3];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    rb_fwd_kin<M>(p, sn, cs, pos);
    rb_store<3>(xyz, ld, s, pos);
}

template <class M>
__global__ void __launch_bounds__(RB_BLOCK)
rb_jac_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q, RB_R* __restrict__ Jout,
              size_t B, size_t ld) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    RB_R a[N], sn[N], cs[N], J[N][6];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    rb_jac<M>(p, sn, cs, J);
#pragma unroll
    for (int c = 0; c < N; ++c)
#pragma unroll
        for (int r = 0; r < 6; ++r) __stcs(Jout + (size_t)(r + 6 * c) * ld + s, J[c][r]);
}

// MPC rollout (SURVEY.md a14): the trajectory's (q, dq) stay in registers for the whole horizon; per step the
// kernel reads tau[t] (n doubles) and writes the new (q, dq) (2n doubles).
// TIP adds the tip-pose terms of RbTipCost (row RB_CW_TIP of cost_w).  The pose of q_t needs sin/cos of q_t, which step t
// computes for forward dynamics anyway: the running term of q_t is added at the top of step t (t >= 1) from that step's
// sin/cos, and only q_H takes one more sin/cos after the last step (running and terminal term from one pose).  Computing
// the pose of q_{t+1} right after the integration would pay a second sin/cos of every joint per step instead.
// COL (with TIP) adds the collision-sphere terms of RbCollisionCost (the block at cost_w + RB_CW_COL, RB_CL_* entries) on
// the same schedule: dt w Phi(q_t) at the top of step t >= 1 from that step's sin/cos, and dt w Phi(q_H) + w_final Phi(q_H)
// after the last step.  Without collision terms the caller runs the TIP kernel (same bits as the tip-cost call).
#ifndef RB_MINB_ROLLOUT
#define RB_MINB_ROLLOUT 2   // measured on B200 (profiles/r1_kbench_rollout.jsonl): 255 regs, 2 blocks per SM is fastest
#endif
// Rows of the cost-weight block a rollout may carry: cost_w[row * RB_MAX_N + joint] (see RbQuadCost in rigidbody.h).
enum : int { RB_CW_QREF = 0, RB_CW_Q, RB_CW_DQ, RB_CW_TAU, RB_CW_QF, RB_CW_DQF, RB_CW_ROWS };
// ... and behind them the tip-pose terms of RbTipCost (RB_TW_* entries of one row, rb_model.h)
enum : int { RB_CW_TIP = RB_CW_ROWS, RB_CW_ROWS_TIP };
// ... and behind those rows the collision block (RB_CL_* entries, rb_model.h): offset and size in doubles
enum : int { RB_CW_COL = RB_CW_ROWS_TIP * RB_MAX_N, RB_CW_DOUBLES_COL = RB_CW_COL + RB_CL_COUNT };
#ifndef RB_ROLLOUT_WS
#define RB_ROLLOUT_WS 0
#endif
#ifndef RB_RO_BLOCK
#define RB_RO_BLOCK 32      // threads per rollout block: one warp (warps of small blocks are spread over the four SM
                            // sub-partitions like those of large ones, profiles/r2_ubench_smsp_mapping.txt)
#endif
#ifndef RB_RO_MINB
#define RB_RO_MINB (RB_MINB_ROLLOUT * (128 / RB_RO_BLOCK))
#endif
template <class M, bool TIP = false, bool COL = false>
__global__ void __launch_bounds__(RB_RO_BLOCK, RB_RO_MINB)
rb_rollout_kernel(const __grid_constant__ typename M::Param p, const RB_R* __restrict__ q0, const RB_R* __restrict__ dq0,
                  const RB_R* __restrict__ tau, RB_R dt, int horizon, RB_R* __restrict__ q_traj,
                  RB_R* __restrict__ dq_traj, RB_R* __restrict__ q_fin, RB_R* __restrict__ dq_fin,
                  size_t B, size_t ld, int* __restrict__ status, const RB_R* __restrict__ cost_w, RB_R* __restrict__ cost) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_RO_BLOCK + threadIdx.x;
    if (s >= B) return;
    RB_R q[N], dq[N];
    rb_load<N>(q0, ld, s, q);
    rb_load<N>(dq0, ld, s, dq);
    bool ok = true;
    RB_R J = RB_R(0);                                // running quadratic cost (sampling-based MPC), see RbQuadCost
    const size_t step = (size_t)N * ld;
    RB_R u[N];
    if (horizon > 0) rb_load<N>(tau, ld, s, u);            // horizon == 0: no step, tau is not read (may be NULL)
    for (int t = 0; t < horizon; ++t) {
        RB_R sn[N], cs[N], qdd[N];
        RB_R un[N];
        // prefetch the next step's torques so the load latency hides behind this step's arithmetic
        if (t + 1 < horizon) rb_load<N>(tau + (size_t)(t + 1) * step, ld, s, un);
        rb_sincos_all<N>(q, sn, cs);
        if constexpr (TIP) {
            if (t > 0) {                               // running tip terms of q_t
                RB_R R[3][3], pos[3], run, fin;
                rb_tip_pose<M>(p, sn, cs, R, pos);
                rb_tip_terms(R, pos, cost_w + RB_CW_TIP * RB_MAX_N, run, fin);
                J = fma(dt, run, J);
                if constexpr (COL) J = fma(dt, __ldg(cost_w + RB_CW_COL + RB_CL_W) * rb_col_phi<M>(p, sn, cs, cost_w + RB_CW_COL), J);
            }
        }
        ok = rb_forward_dynamics<M>(p, sn, cs, dq, u, qdd) && ok;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            dq[i] = fma(dt, qdd[i], dq[i]);
            q[i] = fma(dt, dq[i], q[i]);
        }
        if (q_traj) rb_store<N>(q_traj + (size_t)t * step, ld, s, q);
        if (dq_traj) rb_store<N>(dq_traj + (size_t)t * step, ld, s, dq);
        if (cost) {                                    // stage cost of the state reached and the torque applied
            RB_R c = RB_R(0);
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const RB_R e = q[i] - __ldg(cost_w + RB_CW_QREF * RB_MAX_N + i);
                c = fma(__ldg(cost_w + RB_CW_Q * RB_MAX_N + i) * e, e, c);
                c = fma(__ldg(cost_w + RB_CW_DQ * RB_MAX_N + i) * dq[i], dq[i], c);
                c = fma(__ldg(cost_w + RB_CW_TAU * RB_MAX_N + i) * u[i], u[i], c);
            }
            J = fma(dt, c, J);
        }
        if (t + 1 < horizon) {
#pragma unroll
            for (int i = 0; i < N; ++i) u[i] = un[i];
        }
    }
    if (cost) {                                        // terminal cost
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const RB_R e = q[i] - __ldg(cost_w + RB_CW_QREF * RB_MAX_N + i);
            J = fma(__ldg(cost_w + RB_CW_QF * RB_MAX_N + i) * e, e, J);
            J = fma(__ldg(cost_w + RB_CW_DQF * RB_MAX_N + i) * dq[i], dq[i], J);
        }
        if constexpr (TIP) {                           // q_H: its running term (horizon > 0) and the terminal term
            RB_R sn[N], cs[N], R[3][3], pos[3], run, fin;
            rb_sincos_all<N>(q, sn, cs);
            rb_tip_pose<M>(p, sn, cs, R, pos);
            rb_tip_terms(R, pos, cost_w + RB_CW_TIP * RB_MAX_N, run, fin);
            if (horizon > 0) J = fma(dt, run, J);
            J += fin;
            if constexpr (COL) {                       // the same for the collision terms
                const RB_R phi = rb_col_phi<M>(p, sn, cs, cost_w + RB_CW_COL);
                if (horizon > 0) J = fma(dt, __ldg(cost_w + RB_CW_COL + RB_CL_W) * phi, J);
                J = fma(__ldg(cost_w + RB_CW_COL + RB_CL_WF), phi, J);
            }
        }
        __stcs(cost + s, ok ? J : rb_nan<RB_R>());
    }
    if (q_fin) rb_store<N>(q_fin, ld, s, q);
    if (dq_fin) rb_store<N>(dq_fin, ld, s, dq);
    if (!ok) atomicOr(status, RB_STATUS_NOT_SPD);
}

#if RB_ROLLOUT_WS
#include "experiments/rb_rollout_ws.cuh"      // two warps per 32 trajectories: measured slower (DESIGN.md 4.5), not part of the default build
#endif

#ifndef RB_DEVICE_ONLY
// ------------------------------------------------------------------ launchers for policy M
template <class M>
struct RbLaunch {
    using P = typename M::Param;
    static unsigned grid(size_t B) { return (unsigned)((B + RB_BLOCK - 1) / RB_BLOCK); }
    // SM count of the current device (cached per device ordinal).
    static int sm_count() {
        static std::atomic<int> cache[64];
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
        int v = cache[dev].load(std::memory_order_relaxed);
        if (v == 0) {
            if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
            cache[dev].store(v, std::memory_order_relaxed);
        }
        return v;
    }
    static cudaError_t rnea(const void* param, const double* q, const double* dq, const double* ddq, double* tau,
                            size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        size_t done = 0;
#if RB_STREAM || RB_PREFETCH
        { cudaError_t e = RbExperimentLaunch<M>::rnea(*(const P*)param, q, dq, ddq, tau, B, ld, st, sm_count(), &done); if (e != cudaSuccess || done == B) return e; }
#endif
        rb_rnea_kernel<M><<<grid(B - done), RB_BLOCK, 0, st>>>(*(const P*)param, q + done, dq + done, ddq + done, tau + done, B - done, ld);
        return cudaGetLastError();
    }
    static cudaError_t fd(const void* param, const double* q, const double* dq, const double* tau, double* qdd,
                          size_t B, size_t ld, int* status, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        size_t done = 0;
#if RB_STREAM || RB_PREFETCH
        { cudaError_t e = RbExperimentLaunch<M>::fd(*(const P*)param, q, dq, tau, qdd, B, ld, status, st, sm_count(), &done); if (e != cudaSuccess || done == B) return e; }
#endif
        rb_fd_kernel<M><<<grid(B - done), RB_BLOCK, 0, st>>>(*(const P*)param, q + done, dq + done, tau + done, qdd + done, B - done, ld, status);
        return cudaGetLastError();
    }
    static cudaError_t rnea_fd(const void* param, const double* q, const double* dq, const double* ddq, const double* tau_in,
                               double* out, size_t B, size_t ld, int* status, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_rnea_fd_kernel<M><<<grid(B), RB_BLOCK, 0, st>>>(*(const P*)param, q, dq, ddq, tau_in, out, B, ld, status);
        return cudaGetLastError();
    }
    static constexpr size_t aos_smem = (size_t)3 * RB_BLOCK * M::N * sizeof(double);
    static cudaError_t rnea_aos(const void* param, const double* q, const double* dq, const double* ddq, double* tau,
                                size_t B, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_rnea_kernel<M, true><<<grid(B), RB_BLOCK, aos_smem, st>>>(*(const P*)param, q, dq, ddq, tau, B, 0);
        return cudaGetLastError();
    }
    static cudaError_t fd_aos(const void* param, const double* q, const double* dq, const double* tau, double* qdd,
                              size_t B, int* status, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_fd_kernel<M, true><<<grid(B), RB_BLOCK, aos_smem, st>>>(*(const P*)param, q, dq, tau, qdd, B, 0, status);
        return cudaGetLastError();
    }
    static cudaError_t crba(const void* param, const double* q, double* H, size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_crba_kernel<M><<<grid(B), RB_BLOCK, 0, st>>>(*(const P*)param, q, H, B, ld);
        return cudaGetLastError();
    }
    static cudaError_t fwd_kin(const void* param, const double* q, double* xyz, size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_fwd_kin_kernel<M><<<grid(B), RB_BLOCK, 0, st>>>(*(const P*)param, q, xyz, B, ld);
        return cudaGetLastError();
    }
    static cudaError_t jac(const void* param, const double* q, double* J, size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_jac_kernel<M><<<grid(B), RB_BLOCK, 0, st>>>(*(const P*)param, q, J, B, ld);
        return cudaGetLastError();
    }
    static cudaError_t rollout(const void* param, const double* q0, const double* dq0, const double* tau, double dt,
                               int horizon, double* q_traj, double* dq_traj, double* q_fin, double* dq_fin,
                               size_t B, size_t ld, int* status, const double* cost_w, double* cost, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
#if RB_ROLLOUT_WS
        if constexpr (M::N <= RB_RO2_MAX_N) {
            if (rb_rollout_mode() == 2) {
                rb_rollout_ws_kernel<M><<<(unsigned)((B + 63) / 64), 128, 0, st>>>(*(const P*)param, q0, dq0, tau, dt, horizon, q_traj, dq_traj,
                                                                                  q_fin, dq_fin, B, ld, status, cost_w, cost);
                return cudaGetLastError();
            }
        }
#endif
        rb_rollout_kernel<M><<<(unsigned)((B + RB_RO_BLOCK - 1) / RB_RO_BLOCK), RB_RO_BLOCK, 0, st>>>(
            *(const P*)param, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost);
        return cudaGetLastError();
    }
    static cudaError_t rollout_tip(const void* param, const double* q0, const double* dq0, const double* tau, double dt,
                                   int horizon, double* q_traj, double* dq_traj, double* q_fin, double* dq_fin,
                                   size_t B, size_t ld, int* status, const double* cost_w, double* cost, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_rollout_kernel<M, true><<<(unsigned)((B + RB_RO_BLOCK - 1) / RB_RO_BLOCK), RB_RO_BLOCK, 0, st>>>(
            *(const P*)param, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost);
        return cudaGetLastError();
    }
    static cudaError_t rollout_col(const void* param, const double* q0, const double* dq0, const double* tau, double dt,
                                   int horizon, double* q_traj, double* dq_traj, double* q_fin, double* dq_fin,
                                   size_t B, size_t ld, int* status, const double* cost_w, double* cost, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_rollout_kernel<M, true, true><<<(unsigned)((B + RB_RO_BLOCK - 1) / RB_RO_BLOCK), RB_RO_BLOCK, 0, st>>>(
            *(const P*)param, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld, status, cost_w, cost);
        return cudaGetLastError();
    }
    // M32 = the same policy with Real = float (fp32 mode)
    template <class M32>
    static cudaError_t rnea_f32(const void* param, const float* q, const float* dq, const float* ddq, float* tau,
                                size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_rnea_kernel<M32, false><<<grid(B), RB_BLOCK, 0, st>>>(*(const typename M32::Param*)param, q, dq, ddq, tau, B, ld);
        return cudaGetLastError();
    }
    template <class M32>
    static cudaError_t fd_f32(const void* param, const float* q, const float* dq, const float* tau, float* qdd,
                              size_t B, size_t ld, int* status, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_fd_kernel<M32, false><<<grid(B), RB_BLOCK, 0, st>>>(*(const typename M32::Param*)param, q, dq, tau, qdd, B, ld, status);
        return cudaGetLastError();
    }
    template <class M32 = void>
    static RbOps ops(const char* name) {
        RbOps o{};
        o.name = name; o.param_bytes = sizeof(P);
        o.rnea = &rnea; o.fd = &fd; o.rnea_aos = &rnea_aos; o.fd_aos = &fd_aos;
        o.crba = &crba; o.fwd_kin = &fwd_kin; o.jac = &jac; o.rollout = &rollout; o.rollout_tip = &rollout_tip;
        o.rollout_col = &rollout_col;
        o.rnea_fd = &rnea_fd;
        if constexpr (!std::is_void<M32>::value) { o.rnea_f32 = &rnea_f32<M32>; o.fd_f32 = &fd_f32<M32>; }
        return o;
    }
};
#endif  // RB_DEVICE_ONLY
