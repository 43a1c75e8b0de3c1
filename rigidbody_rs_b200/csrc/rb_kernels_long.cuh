// rb_kernels_long.cuh -- unrolled kernels for chains too long to keep per-state data in registers
// (BASELINE.json configs[4]: the synthetic 32-joint serial chain).
//
// Same model-policy templates as rb_kernels.cuh (CtModel / RtModel, constants from the instruction stream or the
// constant bank, never from global memory: the first loop-based 32-joint kernels were bound by the ~14
// model/sin-cos load instructions each force transform needed).  What changes for long chains:
//   * RNEA: the 6(N-1) force components live in the thread's local frame (ptxas spills what does not fit;
//     spills are private, interleaved per thread, hence coalesced);
//   * forward dynamics is not here: H (528 doubles at N = 32) cannot be held by a thread, and a 400 KB unrolled
//     "CRBA to HBM" kernel plus a tile solver ran at 0.089 G evals/s.  The run-time-n family's lane-per-joint kernels
//     (rb_kernels_warp.cu, 0.32 G evals/s) serve it through the fallback table.
#pragma once
#include "rb_kernels.cuh"
#ifndef RB_DEVICE_ONLY
#include "rb_util.cuh"
#endif

#ifndef RB_MINB_LONG
#define RB_MINB_LONG 2
#endif

template <class M>
__global__ void __launch_bounds__(RB_BLOCK, RB_MINB_LONG)
rb_long_rnea_kernel(const __grid_constant__ typename M::Param p, const double* __restrict__ q, const double* __restrict__ dq,
                    const double* __restrict__ ddq, double* __restrict__ tau, size_t B, size_t ld) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    double a[N], b[N], c[N], sn[N], cs[N], t[N];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    rb_load<N>(dq, ld, s, b);
    rb_load<N>(ddq, ld, s, c);
    rb_rnea<M, true>(p, sn, cs, b, c, t);
    rb_store<N>(tau, ld, s, t);
}

// H out in the reference convention (entry r + N*c, strict lower triangle 0), written entry by entry.
template <class M>
__global__ void __launch_bounds__(RB_BLOCK, RB_MINB_LONG)
rb_long_crba_kernel(const __grid_constant__ typename M::Param p, const double* __restrict__ q, double* __restrict__ Hout,
                    size_t B, size_t ld) {
    constexpr int N = M::N;
    const size_t s = (size_t)blockIdx.x * RB_BLOCK + threadIdx.x;
    if (s >= B) return;
    double a[N], sn[N], cs[N];
    rb_load<N>(q, ld, s, a);
    rb_sincos_all<N>(a, sn, cs);
    for (int c = 0; c < N; ++c)
        for (int r = c + 1; r < N; ++r) __stcs(Hout + (size_t)(r + N * c) * ld + s, 0.0);
    rb_crba_put<M>(p, sn, cs, [&](auto jc, auto ic, double v) {
        constexpr int J = decltype(jc)::value, I = decltype(ic)::value;
        __stcs(Hout + (size_t)(J + N * I) * ld + s, v);
    });
}

#ifndef RB_DEVICE_ONLY
template <class M>
struct RbLaunchLong {
    using MP = typename M::Param;
    static unsigned grid(size_t B) { return (unsigned)((B + RB_BLOCK - 1) / RB_BLOCK); }
    static cudaError_t rnea(const void* param, const double* q, const double* dq, const double* ddq, double* tau,
                            size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_long_rnea_kernel<M><<<grid(B), RB_BLOCK, 0, st>>>(*(const MP*)param, q, dq, ddq, tau, B, ld);
        return cudaGetLastError();
    }
    static cudaError_t crba(const void* param, const double* q, double* H, size_t B, size_t ld, cudaStream_t st) {
        if (B == 0) return cudaSuccess;
        rb_long_crba_kernel<M><<<grid(B), RB_BLOCK, 0, st>>>(*(const MP*)param, q, H, B, ld);
        return cudaGetLastError();
    }
    // fd / fwd_kin / jac / rollout are served by the run-time-n family (null here = use the fallback table).
    static RbOps ops(const char* name) {
        RbOps o{};
        o.name = name; o.param_bytes = sizeof(MP);
        o.rnea = &rnea; o.crba = &crba;
        return o;
    }
};
#endif  // RB_DEVICE_ONLY
