// cov_region.cu -- the grid-free static objective's kernels (sm_100a): the arcs of the covered set's boundary
// (cov_set_region, once per region) and the batch evaluation (cov_eval_region_batch, one warp per candidate).  The
// device MADS on this objective is region_solve_kernel in cov_mads.cu.  The geometry is in cov_region.cuh.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "cov_kernel_common.cuh"
#include "cov_region.cuh"
#include "cov_kernels.cuh"

namespace cov {

// The arcs of every covered circle m that lie inside the domain and inside no other covered disc, in circle order
// and, per circle, in list order of their starts: one warp walks the circles (M <= kRegionMaxCovered, run once per
// region).  Writes at most cap arcs and the count of all of them.
__global__ void __launch_bounds__(32) region_arcs_kernel(const __grid_constant__ RegionDesc r, RegionArc *out, int cap,
                                                         int *count)
{
    extern __shared__ __align__(16) double arcs_list[]; // ia, ib: region_list_cap(0, M) doubles each
    const int M = r.M;
    const uint32_t lane = lane_id();
    double *ia = arcs_list, *ib = arcs_list + region_list_cap(0, M);
    const RegionView v{r.discs, r.discs + M, r.discs + 2 * M, nullptr, M, 0, r.x_lo, r.y_lo, r.x_hi, r.y_hi};
    int K = 0;
    for (int m = 0; m < M; ++m) {
        const double cx = v.cx[m], cy = v.cy[m], R = v.cr[m];
        int n = 0;
        bool whole = false;
        for (int j0 = 0; j0 < M + 4 && !whole; j0 += 32) {
            const int j = j0 + (int)lane;
            int rel = 0;
            double phi = 0.0, alpha = 0.0;
            if (j < M) {
                if (j != m) rel = circle_vs_disc(cx, cy, R, v.cx[j], v.cy[j], v.cr[j], m < j, phi, alpha);
            } else if (j < M + 4) {
                rel = circle_vs_edge(v, j - M, cx, cy, R, phi, alpha);
            }
            whole = __any_sync(0xffffffffu, rel == 2);
            double a0 = 0, b0 = 0, a1 = 0, b1 = 0;
            const int k = rel == 1 ? wrap_interval(phi, alpha, a0, b0, a1, b1) : 0;
            n = warp_append(ia, ib, n, k, a0, b0, a1, b1);
        }
        __syncwarp();
        if (!whole)
            for_each_exposed(ia, ib, n, 0.0, kTwoPi, [&](bool has, double pos, double nxt) {
                const uint32_t bal = __ballot_sync(0xffffffffu, has);
                const int at = K + __popc(bal & ((1u << lane) - 1u));
                if (has && at < cap) out[at] = RegionArc{pos, nxt, m, 0};
                K += __popc(bal);
            });
        __syncwarp();
    }
    if (lane == 0) *count = K;
}

cudaError_t launch_region_arcs(const RegionDesc &r, RegionArc *out, int cap, int *count, cudaStream_t s)
{
    const int smem = 16 * region_list_cap(0, r.M);
    cudaError_t err = cudaFuncSetAttribute(region_arcs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    region_arcs_kernel<<<1, 32, smem, s>>>(r, out, cap, count);
    return cudaGetLastError();
}

// obj / area / feasible of B candidates (each nullable), one warp per candidate, persistent CTAs.
template <int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS)
region_eval_kernel(const __grid_constant__ RegionDesc r, const __grid_constant__ ObjParams o, const double *__restrict__ X,
                   long long B, double *obj, double *area, unsigned char *feasible)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const RegionView v = region_stage(r, smem_raw);
    const int N = o.N, W = blockDim.x >> 5, warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    unsigned char *wbase = smem_raw + region_smem_bytes(r.M, r.K) + (size_t)warp * region_warp_bytes(N, r.M);
    double *stage = reinterpret_cast<double *>(wbase);
    double *ia = reinterpret_cast<double *>(wbase + round_up(3 * N * 8, 16)), *ib = ia + region_list_cap(N, r.M);
    __syncthreads();
    for (long long b = (long long)blockIdx.x * W + warp; b < B; b += (long long)gridDim.x * W) {
        for (int t = lane; t < 3 * N; t += 32) stage[t] = __ldg(X + b * 3 * N + t);
        __syncwarp();
        double A;
        int feas;
        const double f = region_objective(v, o, stage, ia, ib, A, feas);
        if (lane == 0) {
            if (obj) obj[b] = f;
            if (area) area[b] = A;
            if (feasible) feasible[b] = (unsigned char)feas;
        }
        __syncwarp(); // the stage is rewritten for the warp's next candidate
    }
}

cudaError_t launch_region_eval(const RegionDesc &r, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                               long long B, double *obj, double *area, unsigned char *feasible, cudaStream_t s)
{
    if (B <= 0) return cudaSuccess;
    int warps = 0, smem = 0;
    if (o.N > kRegionMaxUavs || !region_plan(o.N, r.M, r.K, 0, cfg.max_smem_optin - 1024 /* the kernel's static shared memory */, &warps, &smem))
        return cudaErrorInvalidConfiguration;
    auto kern = region_eval_kernel<kRegionThreads, kRegionCtas>;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem);
    if (err != cudaSuccess) return err;
    const int grid = (int)std::min<long long>((B + warps - 1) / warps, (long long)cfg.num_sms * std::max(per_sm, 1));
    kern<<<grid, warps * 32, smem, s>>>(r, o, dX, B, obj, area, feasible);
    return cudaGetLastError();
}

} // namespace cov
