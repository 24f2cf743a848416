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
    double *ia = arcs_list, *ib = arcs_list + region_list_cap(0, M);
    const RegionView v{r.discs, r.discs + M, r.discs + 2 * M, nullptr, M, 0, r.x_lo, r.y_lo, r.x_hi, r.y_hi};
    covered_arcs(v, ia, ib, out, cap, count);
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

// ---- cov_run_horizon_region: step 1 and step 7 of a timestep ----
// Step 1 of timestep t, by one warp: cur's discs with R > 0 appended to the covered set in UAV order (cov_set_region's
// filter), then the arcs of its boundary (covered_arcs, region_arcs_kernel's walk) and K_t to stats_row[3].  A
// non-finite value in cur or more than kRegionMaxArcs arcs is recorded in c.ctl with t; every later kernel of the call
// then returns at once.
__global__ void __launch_bounds__(32) cover_arcs_kernel(const __grid_constant__ CoverSet c, const double *__restrict__ cur,
                                                        int N, long long t, long long *stats_row)
{
    extern __shared__ __align__(16) double arcs_list[]; // ia, ib: region_list_cap(0, c.pitch) doubles each
    if (c.ctl[2]) return;
    const uint32_t lane = lane_id();
    int M = c.ctl[0];
    bool bad = false;
    for (int i0 = 0; i0 < N; i0 += 32) {
        const int i = i0 + (int)lane;
        double x = 0.0, y = 0.0, R = 0.0;
        if (i < N) {
            x = cur[i];
            y = cur[N + i];
            R = cur[2 * N + i];
            bad |= !(isfinite(x) && isfinite(y) && isfinite(R));
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, i < N && R > 0.0);
        const int at = M + __popc(bal & ((1u << lane) - 1u));
        if (i < N && R > 0.0 && at < c.pitch) {
            c.discs[at] = x;
            c.discs[c.pitch + at] = y;
            c.discs[2 * c.pitch + at] = R;
        }
        M += __popc(bal);
    }
    if (__any_sync(0xffffffffu, bad)) {
        if (lane == 0) {
            c.ctl[2] = kCoverBadDisc;
            c.ctl[3] = (int)t;
        }
        return;
    }
    M = min(M, c.pitch); // the host sized the buffer for every disc the call can append
    __syncwarp();        // the appended discs are read by every lane
    double *ia = arcs_list, *ib = arcs_list + region_list_cap(0, c.pitch);
    const RegionView v{c.discs, c.discs + c.pitch, c.discs + 2 * c.pitch, nullptr, M, 0, c.x_lo, c.y_lo, c.x_hi, c.y_hi};
    const int K = covered_arcs(v, ia, ib, c.arcs, kRegionMaxArcs, c.ctl + 1);
    if (lane == 0) {
        c.ctl[0] = M;
        stats_row[3] = K;
        if (K > kRegionMaxArcs) {
            c.ctl[2] = kCoverManyArcs;
            c.ctl[3] = (int)t;
        }
    }
}

// Step 7, by one warp: the region objective without the barrier of the committed swarm x on the covered set and arcs
// as step 1 left them, read through L2 (one candidate: nothing to stage).  Shared memory: region_warp_bytes(N, pitch).
// The launch bounds are region_eval_kernel's, so region_area is compiled for the same register budget.
__global__ void __launch_bounds__(kRegionThreads, kRegionCtas)
cover_eval_kernel(const __grid_constant__ CoverSet c, const __grid_constant__ ObjParams o, const double *__restrict__ x,
                  double *obj)
{
    extern __shared__ __align__(16) unsigned char cover_ws[];
    if (c.ctl[2]) return;
    const int N = o.N;
    const uint32_t lane = lane_id();
    const RegionView v{c.discs, c.discs + c.pitch, c.discs + 2 * c.pitch, c.arcs, c.ctl[0], min(c.ctl[1], kRegionMaxArcs),
                       c.x_lo, c.y_lo, c.x_hi, c.y_hi};
    double *stage = reinterpret_cast<double *>(cover_ws);
    double *ia = reinterpret_cast<double *>(cover_ws + round_up(3 * N * 8, 16)), *ib = ia + region_list_cap(N, c.pitch);
    for (int i = lane; i < 3 * N; i += 32) stage[i] = x[i];
    __syncwarp();
    double A;
    int feas;
    const double f = region_objective(v, o, stage, ia, ib, A, feas);
    if (lane == 0) *obj = f;
}

cudaError_t launch_cover_arcs(const CoverSet &c, const double *cur, int N, long long t, long long *stats_row,
                              cudaStream_t s)
{
    cover_arcs_kernel<<<1, 32, 16 * region_list_cap(0, c.pitch), s>>>(c, cur, N, t, stats_row);
    return cudaGetLastError();
}

cudaError_t launch_cover_eval(const CoverSet &c, const ObjParams &o, const double *x, double *obj, cudaStream_t s)
{
    cover_eval_kernel<<<1, 32, region_warp_bytes(o.N, c.pitch), s>>>(c, o, x, obj);
    return cudaGetLastError();
}

} // namespace cov
