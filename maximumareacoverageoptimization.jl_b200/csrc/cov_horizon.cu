// cov_horizon.cu -- the two kernels of cov_run_horizon (receding-horizon MADS on the device, FullSimulation.py
// lines 72-107 per timestep) that no existing launcher covers:
//   horizon_start_kernel   steps 2-4 of timestep t: the r_max rule, cons3's previous swarm := cur, and the S starts
//                          with their initial meshes (the solver's MadsArgs X0 / a0 / b0);
//   horizon_commit_kernel  step 6: the winner of the S solves becomes cur (row t of X_out), its stats row, and the
//                          thresholds [x; y; T(R)] of cur that the next timestep's rmvCoveredPOI reads.
// rmvCoveredPOI, the repack of the bit planes, the solves and the objective of cur are the existing launchers.
// Both kernels use the FP64 operations the host forms (cov_set_params, FullSimulation.py, cov_api.cu's initial_mesh)
// one by one, so a host replay of the same horizon gives the same bits.  Both take E scenarios side by side
// (cov_run_horizon_ensemble): blockIdx.y (start) or blockIdx.x (commit) is the scenario.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "cov_device.cuh"
#include "cov_kernel_common.cuh"
#include "cov_kernels.cuh"

namespace cov {

namespace {
constexpr int kHorizonThreads = 256;
constexpr int kStartMaxBlocks = 148 * 8;

__device__ __forceinline__ double max_host(double a, double b) { return (a < b) ? b : a; } // std::max

__device__ __forceinline__ double p10(const double *pow10, int b) { return pow10[b - kMadsPow10Min]; }
} // namespace

__global__ void __launch_bounds__(kHorizonThreads)
horizon_start_kernel(const HorizonStep s, const double *__restrict__ cur_all, double *__restrict__ params_all,
                     double *__restrict__ X0_all, double *__restrict__ a0_all, int *__restrict__ b0_all)
{
    const int N = s.N, n = 3 * N;
    for (long long e = blockIdx.y; e < s.E; e += gridDim.y) {
        const double *cur = cur_all + e * n;
        double *params = params_all + e * 5 * N, *X0 = X0_all + e * s.S * n, *a0 = a0_all + e * s.S * n;
        int *b0 = b0_all + e * s.S * n;
        const unsigned long long seed = s.seed + (unsigned long long)e * s.seed_stride;
        if (blockIdx.x == 0) {
            for (int i = threadIdx.x; i < N; i += blockDim.x) {
                const double x = cur[i], y = cur[N + i], R = cur[2 * N + i];
                // FullSimulation.py:80-87, from the second timestep on
                if (s.t >= 2 && s.n_boxes > 0 && fabs(__dsub_rn(s.h_focus, __ddiv_rn(R, s.tan_half_fov))) < 1.0) {
                    const double m = __dmul_rn(s.h_max, s.tan_half_fov);
                    bool near = false;
                    for (int k = 0; k < s.n_boxes; ++k) {
                        const double *bx = s.boxes + 4 * k; // x_LB, x_UB, y_LB, y_UB
                        near |= x < __dadd_rn(bx[1], m) && x > __dsub_rn(bx[0], m) && y < __dadd_rn(bx[3], m) &&
                                y > __dsub_rn(bx[2], m);
                    }
                    params[i] = near ? __dmul_rn(s.h_focus, s.tan_half_fov) : m;
                }
                params[N + i] = x; // cons3's previous swarm, as cov_set_params stores it
                params[2 * N + i] = y;
                params[3 * N + i] = __ddiv_rn(R, s.tan_half_fov);
            }
        }
        const long long total = s.S * (long long)n;
        for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < total;
             q += (long long)gridDim.x * blockDim.x) {
            const long long k = q / n;
            const int v = (int)(q - k * n);
            double x = cur[v];
            if (k > 0 && v < 2 * N) { // x_i and y_i of start k >= 1: cur + spread * z, snapped to the mesh
                unsigned long long sum = 0;
#pragma unroll
                for (uint32_t j = 0; j < 3; ++j) {
                    uint32_t r[4];
                    philox4x32_10((uint32_t)s.t, (uint32_t)k, (uint32_t)v, 3u + j, (uint32_t)seed,
                                  (uint32_t)(seed >> 32), r);
                    sum += (unsigned long long)r[0] + r[1] + r[2] + r[3];
                }
                const double z = __dsub_rn(__dmul_rn((double)sum, 2.3283064365386962890625e-10), 6.0);
                x = __dadd_rn(x, __dmul_rn(s.spread, z));
                if (s.granularity > 0) x = __dmul_rn(rint(__ddiv_rn(x, s.granularity)), s.granularity);
            }
            X0[q] = x;
            // cov_api.cu's initial_mesh with floor(log10(target)) read off the host-libm table: the largest b >= 0
            // with 10^b <= target (target >= 1)
            const double target = max_host(max_host(__ddiv_rn(fabs(x), 10.0), 1.0), s.granularity);
            int b = 0;
            while (b < -kMadsPow10Min && p10(s.pow10, b + 1) <= target) ++b;
            const double mant = __ddiv_rn(target, p10(s.pow10, b));
            a0[q] = mant < 2 ? 1.0 : (mant < 5 ? 2.0 : 5.0);
            b0[q] = b;
        }
    }
}

// One CTA: the solve with the smallest barrier value (NaN counts as +Inf, ties to the smallest k, k = 0 when none is
// finite) becomes cur.  stats_row[0..2] = winner, evaluations over the S solves, solves with a feasible point
// (stats_row[3], the entries removed, is the removal kernel's).
__global__ void __launch_bounds__(kHorizonThreads)
horizon_commit_kernel(long long S, int N, const double *__restrict__ Xs_all, const double *__restrict__ objs_all,
                      const long long *__restrict__ mstats_all, double *__restrict__ cur_all,
                      long long *__restrict__ stats_all, double *__restrict__ xyT_all, long long row_stride)
{
    __shared__ double s_best[kHorizonThreads];
    __shared__ long long s_k[kHorizonThreads], s_ev[kHorizonThreads], s_feas[kHorizonThreads];
    const int tid = threadIdx.x, n = 3 * N;
    const long long e = blockIdx.x;
    const double *Xs = Xs_all + e * S * n, *objs = objs_all + e * S;
    const long long *mstats = mstats_all + e * S * 4;
    double *cur = cur_all + e * n, *xyT = xyT_all + e * n;
    long long *stats_row = stats_all + e * row_stride;
    double best = __longlong_as_double(0x7ff0000000000000ll);
    long long kb = -1, ev = 0, feas = 0;
    for (long long k = tid; k < S; k += blockDim.x) { // increasing k: a strict < keeps the smallest
        const double f = objs[k];
        if (f < best) {
            best = f;
            kb = k;
        }
        ev += mstats[4 * k + 1];
        feas += isfinite(f) ? 1 : 0;
    }
    s_best[tid] = best;
    s_k[tid] = kb;
    s_ev[tid] = ev;
    s_feas[tid] = feas;
    __syncthreads();
    for (int off = blockDim.x / 2; off > 0; off >>= 1) {
        if (tid < off) {
            const double fb = s_best[tid + off];
            const long long kk = s_k[tid + off];
            if (kk >= 0 && (s_k[tid] < 0 || fb < s_best[tid] || (fb == s_best[tid] && kk < s_k[tid]))) {
                s_best[tid] = fb;
                s_k[tid] = kk;
            }
            s_ev[tid] += s_ev[tid + off];
            s_feas[tid] += s_feas[tid + off];
        }
        __syncthreads();
    }
    const long long w = s_k[0] >= 0 ? s_k[0] : 0;
    for (int i = tid; i < n; i += blockDim.x) cur[i] = Xs[w * n + i];
    for (int c = tid; c < N; c += blockDim.x) {
        xyT[c] = Xs[w * n + c];
        xyT[N + c] = Xs[w * n + N + c];
        xyT[2 * N + c] = threshold(Xs[w * n + 2 * N + c]);
    }
    if (tid == 0) {
        stats_row[0] = w;
        stats_row[1] = s_ev[0];
        stats_row[2] = s_feas[0];
    }
}

cudaError_t launch_horizon_start(const HorizonStep &s, const double *cur, double *params, double *X0, double *a0,
                                 int *b0, cudaStream_t stream)
{
    const long long total = s.S * 3LL * s.N;
    const int gy = (int)std::min<long long>(s.E, 65535);
    const int grid = (int)std::max<long long>(1, std::min<long long>((total + kHorizonThreads - 1) / kHorizonThreads,
                                                                      std::max(kStartMaxBlocks / gy, 1)));
    horizon_start_kernel<<<dim3(grid, gy), kHorizonThreads, 0, stream>>>(s, cur, params, X0, a0, b0);
    return cudaGetLastError();
}

cudaError_t launch_horizon_commit(long long S, int N, const double *Xs, const double *objs, const long long *mstats,
                                  double *cur, long long *stats_row, double *xyT, cudaStream_t stream, long long E,
                                  long long row_stride)
{
    horizon_commit_kernel<<<(unsigned)E, kHorizonThreads, 0, stream>>>(S, N, Xs, objs, mstats, cur, stats_row, xyT,
                                                                       row_stride);
    return cudaGetLastError();
}

} // namespace cov
