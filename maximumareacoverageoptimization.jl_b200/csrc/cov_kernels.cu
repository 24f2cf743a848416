// cov_kernels.cu -- the batched coverage-objective kernels of libcoverage_cuda (sm_100a).
//
// What is computed, per candidate x = [x_1..x_N, y_1..y_N, R_1..R_N] (all citations relative to
// /root/reference/):
//   area   = sum over list entries p of w_p * [exists c: sqrt((px-cx)^2 + (py-cy)^2) < R_c]
//                                                    src/AreaCoverageCalculation.jl:63-110
//   obj    = -area + penalty_scale * sum_i |R_i - r_max_i|      src/TDM_STATIC_opt.jl:82-100
//   cons3  : sqrt(dx^2+dy^2+dz^2) > d_lim[i] rejects, z = R/tan(FOV/2)   src/TDM_Constraints.jl:54-75
//   cons7  : y < 200 and R > 19*tan(FOV/2) rejects                      src/TDM_Constraints.jl:142-154
//   cons8  : sqrt((xi-xj)^2+(yi-yj)^2) < sep rejects                    src/TDM_Constraints.jl:157-172
//   cons1_progressive = sum max(R_i - r_max_i, 0)                       src/TDM_Constraints.jl:182-195
//
// The list lives on a lattice, so it is held as bit planes (cov_types.h).  This file holds the two
// cell-sweeping kernels and the launcher; the span kernels (the default) are in
// cov_span_small.cu / cov_span_cta.cu.
//   brute  every cell against every disc (north_star's formulation): FP32 test with a certified
//          error band, FP64 for band cells, ballot + popc.
//   exact  every cell against every disc in FP64 only (cross-check for the others).
// One warp owns one candidate at a time; a CTA is a batch of warps sharing the staged planes.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "cov_device.cuh"
#include "cov_kernel_common.cuh"
#include "cov_candidate.cuh"
#include "cov_kernels.cuh"
#include "../../include/coverage_cuda.h"

namespace cov {

// ------------------------------------------------------------------------------------------
// brute kernel (north_star's formulation): every cell of every word that holds a list entry is
// tested against every disc.  Lane b of a warp owns cell 32w + b + 1 of the word being swept; the
// discs come from the warp's shared memory as one broadcast 16-byte load each
// (cx, tlo, thi, dy^2 for the current row); FP32 test with the certified band, FP64 for band
// cells only; ballot + popc against the plane words.
// ------------------------------------------------------------------------------------------
template <bool MULTI, bool PLANES_SMEM>
__global__ void __launch_bounds__(256)
brute_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
             const double *__restrict__ X, long long B, EvalOut out, unsigned long long *counter,
             int force_exact, int unit)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N;
    const int planes_bytes = PLANES_SMEM ? g.n_planes * g.plane_words * 4 : 0;
    const int warp_bytes = round_up(3 * N * 8, 16) + N * 32 + N * 16;
    uint32_t *planes_s = reinterpret_cast<uint32_t *>(smem_raw);
    unsigned char *wbase = smem_raw + planes_bytes + (size_t)warp * warp_bytes;
    double *stage = reinterpret_cast<double *>(wbase);
    DiscParam *dp = reinterpret_cast<DiscParam *>(wbase + round_up(3 * N * 8, 16));
    float4 *row = reinterpret_cast<float4 *>(wbase + round_up(3 * N * 8, 16) + N * 32);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + planes_bytes + (size_t)warps * warp_bytes);

    if (PLANES_SMEM) stage_planes(g, planes_s, bar, planes_bytes);
    const uint32_t *planes = PLANES_SMEM ? planes_s : g.planes;

    // unit = candidates a warp takes per grab: 32 (coalesced result stores) for big batches, 1 when the batch
    // would otherwise leave warps idle (one candidate is already ~10^5 tests)
    const long long n_chunks = (B + unit - 1) / unit;
    const int cstride = 3 * N;
    for (;;) {
        unsigned long long chunk = 0;
        if (lane == 0) chunk = atomicAdd(counter, 1ull);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
        if ((long long)chunk >= n_chunks) break;
        const long long base = (long long)chunk * unit;
        const int in_chunk = (int)min((long long)unit, B - base);
        double my_obj = 0.0, my_prog = 0.0;
        long long my_cnt = 0;
        long long my_cls[kMaxClasses];
#pragma unroll
        for (int k = 0; k < kMaxClasses; ++k) my_cls[k] = 0;
        int my_feas = 0;

        for (int kc = 0; kc < in_chunk; ++kc) {
            const double *xc = X + (base + kc) * cstride;
            for (int t = lane; t < cstride; t += 32) stage[t] = __ldg(xc + t);
            __syncwarp();
            const CandScalars cs = candidate_prologue<true>(g, o, stage, dp, out.progressive != nullptr);
            __syncwarp();
            for (int c = lane; c < N; c += 32) {
                const DiscParam d = dp[c];
                row[c] = make_float4(d.cxf, force_exact ? -1.0f : d.tlo,
                                     force_exact ? __int_as_float(0x7f800000) : d.thi, 0.0f);
            }
            long long cls_total[kMaxClasses];
#pragma unroll
            for (int k = 0; k < kMaxClasses; ++k) cls_total[k] = 0;
            uint32_t cnt[MULTI ? kMaxClasses : 1];
#pragma unroll
            for (int k = 0; k < (MULTI ? kMaxClasses : 1); ++k) cnt[k] = 0;

            for (int j = 1; j <= g.ny; ++j) {
                const float pyf = fmaf(int_to_float_small(j), g.dyf, -g.hdyf);
                __syncwarp();
                for (int c = lane; c < N; c += 32) {
                    const float ddy = pyf - dp[c].cyf;
                    row[c].w = ddy * ddy;
                }
                __syncwarp();
                const uint32_t *prow = planes + (size_t)(j - 1) * g.stride;
                for (int w = 0; w < g.wpr; ++w) {
                    uint32_t fire = ld_plane<PLANES_SMEM>(prow + w);
                    if (MULTI)
                        for (int l = 1; l < g.n_planes; ++l)
                            fire |= ld_plane<PLANES_SMEM>(prow + (size_t)l * g.plane_words + w);
                    if (fire == 0) continue; // no list entry on these 32 cells
                    const int i = 32 * w + (int)lane + 1;
                    const float pxf = fmaf(int_to_float_small(i), g.dxf, -g.hdxf);
                    bool covered = false, band = false;
#pragma unroll 4
                    for (int c = 0; c < N; ++c) {
                        const float4 r = row[c];
                        const float x = pxf - r.x;
                        const float sf = fmaf(x, x, r.w);
                        const bool in = sf < r.y;
                        covered |= in;
                        band |= !(in || sf > r.z);
                    }
                    const bool need = band && !covered && i <= g.nx;
                    if (__any_sync(0xffffffffu, need)) {
                        if (need) {
                            const double px = cell_centre(i, g.dx, g.hdx);
                            const double py = cell_centre(j, g.dy, g.hdy);
                            for (int c = 0; c < N; ++c)
                                if (radicand(px, py, stage[c], stage[N + c]) < dp[c].T) {
                                    covered = true;
                                    break;
                                }
                        }
                    }
                    const uint32_t m = __ballot_sync(0xffffffffu, covered && i <= g.nx);
                    if (!MULTI) {
                        cnt[0] += __popc(m & fire);
                    } else {
                        for (int l = 0; l < g.n_planes; ++l) {
                            const uint32_t v =
                                __popc(m & ld_plane<PLANES_SMEM>(prow + (size_t)l * g.plane_words + w)) *
                                g.plane_mult[l];
                            const int kcls = g.plane_class[l];
#pragma unroll
                            for (int k = 0; k < kMaxClasses; ++k) cnt[k] += (k == kcls) ? v : 0u;
                        }
                    }
                }
                if ((j & 1023) == 0) { // keep the 32-bit partial counts far from overflow
#pragma unroll
                    for (int k = 0; k < (MULTI ? kMaxClasses : 1); ++k) {
                        cls_total[k] += cnt[k];
                        cnt[k] = 0;
                    }
                }
            }
            long long total = 0;
#pragma unroll
            for (int k = 0; k < kMaxClasses; ++k) {
                if (k < (MULTI ? kMaxClasses : 1)) cls_total[k] += cnt[k]; // ballot counts are warp-uniform
                total += cls_total[k];
            }
            const double objv = assemble_objective(g, o, cls_total, cs.violation);
            if ((int)lane == kc) {
                my_obj = objv;
                my_cnt = total;
                my_feas = cs.feasible;
                my_prog = cs.progressive;
#pragma unroll
                for (int k = 0; k < kMaxClasses; ++k) my_cls[k] = cls_total[k];
            }
            __syncwarp();
        }
        if ((int)lane < in_chunk) {
            const long long bidx = base + lane;
            out.obj[bidx] = my_obj;
            store_mirrors(out, bidx, my_obj, my_feas);
            if (out.count) out.count[bidx] = my_cnt;
            if (out.feasible) out.feasible[bidx] = (unsigned char)my_feas;
            if (out.progressive) out.progressive[bidx] = my_prog;
            if (out.class_count)
                for (int k = 0; k < g.n_classes; ++k) out.class_count[bidx * g.n_classes + k] = my_cls[k];
        }
    }
}

// ------------------------------------------------------------------------------------------
// exact kernel: every cell against every disc, FP64 only. Slow by design; the cross-check.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
exact_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
             const double *__restrict__ X, long long B, EvalOut out, unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N;
    const int warp_bytes = round_up(3 * N * 8, 16) + round_up(N * 8, 16);
    double *stage = reinterpret_cast<double *>(smem_raw + (size_t)warp * warp_bytes);
    double *Ts = reinterpret_cast<double *>(smem_raw + (size_t)warp * warp_bytes + round_up(3 * N * 8, 16));
    const int cstride = 3 * N;
    for (;;) {
        unsigned long long cand = 0;
        if (lane == 0) cand = atomicAdd(counter, 1ull);
        cand = __shfl_sync(0xffffffffu, cand, 0);
        if ((long long)cand >= B) break;
        const double *xc = X + (long long)cand * cstride;
        for (int t = lane; t < cstride; t += 32) stage[t] = xc[t];
        __syncwarp();
        for (int c = lane; c < N; c += 32) Ts[c] = threshold(stage[2 * N + c]);
        const CandScalars cs = candidate_prologue<false>(g, o, stage, nullptr, out.progressive != nullptr);
        __syncwarp();
        long long cls_total[kMaxClasses];
#pragma unroll
        for (int k = 0; k < kMaxClasses; ++k) cls_total[k] = 0;
        for (int j = 1; j <= g.ny; ++j) {
            const double py = cell_centre(j, g.dy, g.hdy);
            for (int w = 0; w < g.wpr; ++w) {
                uint32_t any_bits = 0;
                for (int l = 0; l < g.n_planes; ++l)
                    any_bits |= g.planes[(size_t)l * g.plane_words + (size_t)(j - 1) * g.stride + w];
                if (!any_bits) continue;
                const int i = 32 * w + lane + 1;
                bool cov_cell = false;
                if (i <= g.nx) {
                    const double px = cell_centre(i, g.dx, g.hdx);
                    for (int c = 0; c < N; ++c) {
                        if (radicand(px, py, stage[c], stage[N + c]) < Ts[c]) {
                            cov_cell = true;
                            break;
                        }
                    }
                }
                const uint32_t m = __ballot_sync(0xffffffffu, cov_cell);
                for (int l = 0; l < g.n_planes; ++l) {
                    const uint32_t pw = g.planes[(size_t)l * g.plane_words + (size_t)(j - 1) * g.stride + w];
                    cls_total[g.plane_class[l] & (kMaxClasses - 1)] += (long long)__popc(m & pw) * g.plane_mult[l];
                }
            }
        }
        if (lane == 0) {
            long long total = 0;
            for (int k = 0; k < g.n_classes; ++k) total += cls_total[k];
            const double my_obj = assemble_objective(g, o, cls_total, cs.violation);
            out.obj[cand] = my_obj;
            store_mirrors(out, cand, my_obj, cs.feasible);
            if (out.count) out.count[cand] = total;
            if (out.feasible) out.feasible[cand] = (unsigned char)cs.feasible;
            if (out.progressive) out.progressive[cand] = cs.progressive;
            if (out.class_count)
                for (int k = 0; k < g.n_classes; ++k) out.class_count[cand * g.n_classes + k] = cls_total[k];
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// ordered kernel: the reference's own loop (src/AreaCoverageCalculation.jl:63-110) over the point LIST --
// for each entry in list order, the first covering disc adds the entry's weight to a Float64 running sum and
// breaks.  FP64 only.  This is the kernel for stores whose weights are not dyadic (the high-interest weight
// (h_max tan(FOV/2))^2 pi, src/CellFunctions.jl:41-45): there the value of the sum depends on the order of the
// additions, so it is replayed in list order, one warp per candidate, 32 entries tested at a time and the covered
// ones added one after the other (every lane forms the same sum; ordered_area in cov_candidate.cuh).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ordered_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
               const double *__restrict__ X, long long B, EvalOut out, unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N;
    const int warp_bytes = round_up(3 * N * 8, 16) + round_up(N * 8, 16);
    double *stage = reinterpret_cast<double *>(smem_raw + (size_t)warp * warp_bytes);
    double *Ts = reinterpret_cast<double *>(smem_raw + (size_t)warp * warp_bytes + round_up(3 * N * 8, 16));
    const int cstride = 3 * N;
    for (;;) {
        unsigned long long cand = 0;
        if (lane == 0) cand = atomicAdd(counter, 1ull);
        cand = __shfl_sync(0xffffffffu, cand, 0);
        if ((long long)cand >= B) break;
        const double *xc = X + (long long)cand * cstride;
        for (int t = lane; t < cstride; t += 32) stage[t] = xc[t];
        __syncwarp();
        for (int c = lane; c < N; c += 32) Ts[c] = threshold(stage[2 * N + c]);
        const CandScalars cs = candidate_prologue<false>(g, o, stage, nullptr, out.progressive != nullptr);
        __syncwarp();
        long long cls_total[kMaxClasses];
        const double area = ordered_area(g, N, stage, Ts, cls_total);
        if (lane == 0) {
            long long total = 0;
            for (int k = 0; k < g.n_classes; ++k) total += cls_total[k];
            const double my_obj = __dadd_rn(-area, __dmul_rn(cs.violation, o.penalty_scale));
            out.obj[cand] = my_obj;
            store_mirrors(out, cand, my_obj, cs.feasible);
            if (out.count) out.count[cand] = total;
            if (out.feasible) out.feasible[cand] = (unsigned char)cs.feasible;
            if (out.progressive) out.progressive[cand] = cs.progressive;
            if (out.class_count)
                for (int k = 0; k < g.n_classes; ++k) out.class_count[cand * g.n_classes + k] = cls_total[k];
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// launcher
// ------------------------------------------------------------------------------------------
template <typename K>
static cudaError_t set_smem(K kernel, int bytes)
{
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

cudaError_t launch_eval(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                        long long B, const EvalOut &out, unsigned long long *counter,
                        cudaStream_t stream, LaunchInfo *info)
{
    if (B <= 0) return cudaSuccess;
    cudaError_t err = cudaSuccess; // `counter` is a fresh zeroed slot of the handle's counter ring
    const int N = o.N;
    LaunchInfo li{};
    li.plane_mode = -1;
    if (cfg.ordered || cfg.kernel == COV_KERNEL_ORDERED) {
        if (!g.ent_cell && g.n_ent > 0) return cudaErrorInvalidValue; // the caller uploads the list first
        int warps = 8;
        while (warps > 1 && warps * (round_up(3 * N * 8, 16) + round_up(N * 8, 16)) > 96 * 1024) warps /= 2;
        const int smem = warps * (round_up(3 * N * 8, 16) + round_up(N * 8, 16));
        err = set_smem(ordered_kernel, smem);
        if (err != cudaSuccess) return err;
        const long long want = (B + warps - 1) / warps;
        const int grid = (int)std::min<long long>(want, (long long)cfg.num_sms * 8);
        ordered_kernel<<<grid, warps * 32, smem, stream>>>(g, o, dX, B, out, counter);
        li.grid = grid;
        li.block = warps * 32;
        li.smem_bytes = smem;
        li.kernel = COV_KERNEL_ORDERED;
        if (info) *info = li;
        return cudaGetLastError();
    }
    if (cfg.kernel == COV_KERNEL_EXACT) {
        int warps = 8;
        while (warps > 1 && warps * (round_up(3 * N * 8, 16) + round_up(N * 8, 16)) > 96 * 1024) warps /= 2;
        const int smem = warps * (round_up(3 * N * 8, 16) + round_up(N * 8, 16));
        err = set_smem(exact_kernel, smem);
        if (err != cudaSuccess) return err;
        long long want = (B + warps - 1) / warps;
        const int grid = (int)std::min<long long>(want, (long long)cfg.num_sms * 8);
        exact_kernel<<<grid, warps * 32, smem, stream>>>(g, o, dX, B, out, counter);
        li.grid = grid;
        li.block = warps * 32;
        li.smem_bytes = smem;
        li.kernel = COV_KERNEL_EXACT;
        if (info) *info = li;
        return cudaGetLastError();
    }
    if (cfg.kernel == COV_KERNEL_BRUTE) {
        const bool multi = !(g.n_planes == 1 && g.n_classes == 1 && g.plane_mult[0] == 1);
        int warps = cfg.warps_per_cta > 0 ? min(cfg.warps_per_cta, 8) : 8;
        const int per_warp = round_up(3 * N * 8, 16) + N * 32 + N * 16;
        const int planes_bytes = g.n_planes * g.plane_words * 4;
        while (warps > 1 && warps * per_warp + 16 > cfg.max_smem_optin) warps /= 2;
        if (warps * per_warp + 16 > cfg.max_smem_optin) return cudaErrorInvalidConfiguration;
        const bool planes_smem = planes_bytes + warps * per_warp + 16 <= cfg.max_smem_optin;
        const int smem = (planes_smem ? planes_bytes : 0) + warps * per_warp + 16;
        const int per_sm = max(1, min(8, cfg.max_smem_optin / max(smem, 1)));
        const int unit = (B / 32 >= 4ll * cfg.num_sms * per_sm * warps) ? 32 : 1;
        const long long chunks = (B + unit - 1) / unit;
        const long long want = (chunks + warps - 1) / warps;
        const int grid = (int)std::min<long long>(want, (long long)cfg.num_sms * per_sm);
        li.grid = grid;
        li.block = warps * 32;
        li.smem_bytes = smem;
        li.planes_in_smem = planes_smem;
        li.kernel = COV_KERNEL_BRUTE;
        if (info) *info = li;
#define COV_LAUNCH_BRUTE(M, S)                                                                      \
    do {                                                                                            \
        err = set_smem(brute_kernel<M, S>, smem);                                                   \
        if (err != cudaSuccess) return err;                                                         \
        brute_kernel<M, S><<<grid, warps * 32, smem, stream>>>(g, o, dX, B, out, counter,           \
                                                               cfg.force_exact, unit);              \
    } while (0)
        if (multi) {
            if (planes_smem) COV_LAUNCH_BRUTE(true, true);
            else COV_LAUNCH_BRUTE(true, false);
        } else {
            if (planes_smem) COV_LAUNCH_BRUTE(false, true);
            else COV_LAUNCH_BRUTE(false, false);
        }
#undef COV_LAUNCH_BRUTE
        return cudaGetLastError();
    }
    // span kernels: the small-swarm variant when it applies, else one CTA per candidate
    bool small = cfg.kernel != COV_KERNEL_SPAN_GENERAL && span_small_applies(g, N, cfg, B, nullptr, nullptr);
    // AUTO: a batch of up to one or two thousand candidates finishes sooner with one CTA per candidate (9 us
    // up to 444 candidates, +3.5 us per further 444) than with the warp-per-unit kernel, whose shortest launch
    // (every warp one 4-candidate unit, spread over all SMs) lasts 17-21 us for 5 UAVs and 23-27 us for 8;
    // measured crossover on B200 1 100 - 1 700 candidates for 5 UAVs, 2 000 - 2 300 for 8
    // (tools/small_batch_routing.py).  COV_KERNEL_SPAN keeps the small-swarm kernel from 128 on.
    if (small && cfg.kernel == COV_KERNEL_AUTO && B < 128ll * N + 768) small = false;
    if (small) return launch_span_small(g, o, cfg, dX, B, out, counter, stream, info);
    return launch_span_cta(g, o, cfg, dX, B, out, counter, stream, info);
}

} // namespace cov
