// rb_kernels_mppi.cu -- the model-agnostic kernels of one MPPI step (multibody_mppi_step): the sampler of the perturbed
// torque sequences, the per-problem softmin weights, and the weighted mean of the samples.  The rollout between the
// sampler and the weights is the engine's own cost launcher, unchanged.  Every sum runs in an order fixed by (K, H, n)
// alone, with no atomics, so the results do not depend on chunking, layout or memory kind.
#include <stdint.h>

#include "rb_util.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWThreads = 1024;          // the weights kernel: one block per problem, up to 65 536 samples in it
constexpr int kTile = 4 * kThreads;      // samples per tile of the update's first stage (4 per thread)
constexpr int kRows = 8;                 // rows (t, i) per block of the update's first stage

// The normal draw of counter c (include/rigidbody.h multibody_mppi_step): the splitmix64 mixer of multibody_gpu_fill,
// then Box-Muller on the two 32-bit halves.
__device__ __forceinline__ double mppi_normal(uint64_t seed, uint64_t c) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ULL * (c + 1ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    z = z ^ (z >> 31);
    const double u1 = ((double)(z >> 32) + 0.5) * 0x1.0p-32;
    const double u2 = (double)(z & 0xffffffffULL) * 0x1.0p-32;
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

// Fixed-order sum of one value per thread over the block: shuffle tree per warp, then the warp sums in order by thread 0.
// `red` holds one double per warp.  Every thread gets the result.
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = red[0];
        for (unsigned w = 1; w < blockDim.x / 32; ++w) s += red[w];
        red[0] = s;
    }
    __syncthreads();
    return red[0];
}

}  // namespace

// One thread per (sample j of the chunk, joint i): the start state, then tau over t.  j = p K + k with p the chunk's
// problem; the global sample index is (p_first + p) K + k.
__global__ void __launch_bounds__(kThreads) rb_mppi_sample_kernel(const __grid_constant__ RbMppiParam P, const double* __restrict__ q0,
                                                                  const double* __restrict__ dq0, const double* __restrict__ u_nom,
                                                                  size_t ld, size_t p_first, size_t cnt, double* __restrict__ tau,
                                                                  double* __restrict__ q0s, double* __restrict__ dq0s, size_t ldS) {
    const size_t j = (size_t)blockIdx.x * kThreads + threadIdx.x;
    const int i = blockIdx.y;
    const size_t K = P.K;
    if (j >= cnt * K) return;
    const size_t p = j / K, k = j - p * K;
    q0s[(size_t)i * ldS + j] = q0[(size_t)i * ld + p];
    dq0s[(size_t)i * ldS + j] = dq0[(size_t)i * ld + p];
    const int n = P.n, H = P.H;
    const double sg = P.sigma[i], lo = P.lower[i], hi = P.upper[i];
    const uint64_t s = (uint64_t)(p_first + p) * K + k;
    for (int t = 0; t < H; ++t) {
        const size_t row = (size_t)t * n + i;
        const double u = u_nom[row * ld + p];
        double x = u;
        if (k != 0) x = fma(sg, mppi_normal(P.seed, ((uint64_t)s * H + t) * n + i), u);
        tau[row * ldS + j] = x < lo ? lo : (x > hi ? hi : x);      // NaN passes through
    }
}

// One block per problem: m = min of the finite costs, w_k = exp((m - c_k) / lambda) (0 for a non-finite cost),
// eta = sum w.  Writes w and eta, and w / eta to `sw` when it is not NULL.
__global__ void __launch_bounds__(kWThreads) rb_mppi_weights_kernel(const double* __restrict__ cost, size_t K, double lambda,
                                                                    double* __restrict__ w, double* __restrict__ eta,
                                                                    double* __restrict__ sw) {
    __shared__ double red[kWThreads / 32];
    const size_t p = blockIdx.x;
    const double* c = cost + p * K;
    double m = INFINITY;
#pragma unroll 4
    for (size_t k = threadIdx.x; k < K; k += kWThreads) {
        const double ck = c[k];
        if (isfinite(ck)) m = fmin(m, ck);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_down_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = red[0];
    for (int v = 1; v < kWThreads / 32; ++v) m = fmin(m, red[v]);
    double acc = 0.0;
#pragma unroll 4
    for (size_t k = threadIdx.x; k < K; k += kWThreads) {
        const double ck = c[k];
        const double wk = isfinite(ck) ? exp((m - ck) / lambda) : 0.0;
        w[p * K + k] = wk;
        acc += wk;
    }
    const double e = block_sum(acc, red);
    if (threadIdx.x == 0) eta[p] = e;
    if (sw)
        for (size_t k = threadIdx.x; k < K; k += kWThreads) sw[p * K + k] = w[p * K + k] / e;
}

// First stage of the update: block (tile, row group, problem) sums w_k tau_k over the tile's samples for kRows rows
// (t, i) of tau [rows][ldS]; each thread adds its 4 samples in order, then block_sum.  part: [problem][tile][rows].
// blockIdx.x = row group * ntiles + tile, blockIdx.y = problem.
__global__ void __launch_bounds__(kThreads) rb_mppi_update_tiles_kernel(const double* __restrict__ tau, size_t ldS, size_t K, int rows,
                                                                        size_t ntiles, const double* __restrict__ w,
                                                                        double* __restrict__ part) {
    __shared__ double red[kThreads / 32];
    const size_t tile = blockIdx.x % ntiles, p = blockIdx.y;
    const int r0 = (int)(blockIdx.x / ntiles) * kRows;
    const size_t k0 = tile * kTile + threadIdx.x;
    double wk[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) wk[a] = k0 + (size_t)a * kThreads < K ? w[p * K + k0 + (size_t)a * kThreads] : 0.0;
    double acc[kRows];
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
        acc[r] = 0.0;
        if (r0 + r >= rows) continue;
        const double* row = tau + (size_t)(r0 + r) * ldS + p * K;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const size_t k = k0 + (size_t)a * kThreads;
            if (k < K) acc[r] = fma(wk[a], row[k], acc[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
        const double s = block_sum(acc[r], red);
        if (threadIdx.x == 0 && r0 + r < rows) part[(p * ntiles + tile) * rows + r0 + r] = s;
    }
}

// Second stage: one thread per (row, problem) adds the tiles' partials in order and divides by eta.
__global__ void __launch_bounds__(kThreads) rb_mppi_update_final_kernel(const double* __restrict__ part, size_t ntiles, int rows,
                                                                        const double* __restrict__ eta, size_t cnt,
                                                                        double* __restrict__ u_new, size_t ld) {
    const size_t x = (size_t)blockIdx.x * kThreads + threadIdx.x;
    if (x >= (size_t)rows * cnt) return;
    const size_t p = x / rows, r = x - p * rows;
    double s = 0.0;
    for (size_t tile = 0; tile < ntiles; ++tile) s += part[(p * ntiles + tile) * rows + r];
    u_new[r * ld + p] = s / eta[p];
}

size_t rb_mppi_tiles(size_t K) { return (K + kTile - 1) / kTile; }

cudaError_t rb_launch_mppi_sample(const RbMppiParam& P, const double* q0, const double* dq0, const double* u_nom, size_t ld,
                                  size_t p_first, size_t cnt, double* tau, double* q0s, double* dq0s, size_t ldS, cudaStream_t st) {
    const size_t J = cnt * P.K;
    if (J == 0) return cudaSuccess;
    rb_mppi_sample_kernel<<<dim3((unsigned)((J + kThreads - 1) / kThreads), (unsigned)P.n), kThreads, 0, st>>>(
        P, q0, dq0, u_nom, ld, p_first, cnt, tau, q0s, dq0s, ldS);
    return cudaGetLastError();
}

cudaError_t rb_launch_mppi_weights(const double* cost, size_t K, double lambda, size_t cnt, double* w, double* eta, double* sw,
                                   cudaStream_t st) {
    if (cnt == 0) return cudaSuccess;
    rb_mppi_weights_kernel<<<(unsigned)cnt, kWThreads, 0, st>>>(cost, K, lambda, w, eta, sw);
    return cudaGetLastError();
}

cudaError_t rb_launch_mppi_update(const double* tau, size_t ldS, size_t K, int rows, const double* w, const double* eta, size_t cnt,
                                  double* part, double* u_new, size_t ld, cudaStream_t st) {
    if (cnt == 0 || rows == 0) return cudaSuccess;
    const size_t ntiles = rb_mppi_tiles(K);
    rb_mppi_update_tiles_kernel<<<dim3((unsigned)(ntiles * ((rows + kRows - 1) / kRows)), (unsigned)cnt), kThreads, 0, st>>>(
        tau, ldS, K, rows, ntiles, w, part);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const size_t X = (size_t)rows * cnt;
    rb_mppi_update_final_kernel<<<(unsigned)((X + kThreads - 1) / kThreads), kThreads, 0, st>>>(part, ntiles, rows, eta, cnt, u_new, ld);
    return cudaGetLastError();
}
