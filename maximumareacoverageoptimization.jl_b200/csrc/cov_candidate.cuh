// cov_candidate.cuh -- per-candidate pieces executed by one warp, shared by the objective kernels
// (cov_kernels.cu) and the device MADS solver (cov_mads.cu): the prologue (penalty sum and the fused
// extreme constraints) and the reference's ordered list loop.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "cov_device.cuh"
#include "cov_kernel_common.cuh"

namespace cov {

// ------------------------------------------------------------------------------------------
// per-disc parameters, one 32-byte record per disc in the owning warp's shared memory
// ------------------------------------------------------------------------------------------
struct __align__(16) DiscParam {
    double T;        // s < T  <=>  sqrt(s) < R
    float cxf, cyf;  // FP32 roundings of the centre
    float tlo, thi;  // FP32 radicand below tlo: certainly inside; above thi: certainly outside
    float Tf;        // (float)T, for the span-end estimate
    uint32_t rows;   // r0 | r1 << 16: rows that can hold covered cells (1-based); r0 > r1: none
};
static_assert(sizeof(DiscParam) == 32, "DiscParam must be 32 bytes");

// Results of the prologue that every lane holds after the call.
struct CandScalars {
    double violation;   // sum |R_i - r_max_i| in index order
    double progressive; // sum max(R_i - r_max_i, 0)
    int feasible;
};

// Per-candidate prologue, executed by one warp.
//   stage : the candidate's 3N doubles in shared memory (already visible to the warp)
//   dp    : N DiscParam records to fill
//   poff  : offset of the parameter block read through o's five arrays (cov_run_horizon_ensemble's scenarios)
template <bool WANT_DP>
__device__ __forceinline__ CandScalars candidate_prologue(const GridDesc &g, const ObjParams &o,
                                                          const double *stage, DiscParam *dp,
                                                          bool want_progressive, long long poff = 0)
{
    const int N = o.N;
    const uint32_t lane = lane_id();
    if (WANT_DP) {
        for (int c = lane; c < N; c += 32) {
            const double cx = stage[c], cy = stage[N + c], R = stage[2 * N + c];
            const double T = threshold(R);
            DiscParam d;
            d.T = T;
            d.cxf = (float)cx;
            d.cyf = (float)cy;
            d.Tf = (float)T;
            bool live = (T > 0.0) && (fabs(cx) <= 1.7976931348623157e308) &&
                        (fabs(cy) <= 1.7976931348623157e308);
            int r0 = 1, r1 = 0;
            if (live) {
                if (isinf(R)) {
                    r0 = 1;
                    r1 = g.ny;
                } else {
                    // rows j with |py_j - cy| < R, widened by one row and by the FP64 absorption
                    // error of fl(py - cy) for far-away centres
                    const double extra = (fabs(cy) + R) * 8.8817841970012523e-16 * g.inv_dy; // 2^-50
                    double lo = floor((cy - R) * g.inv_dy + 0.5 - extra);
                    double hi = ceil((cy + R) * g.inv_dy + 0.5 + extra);
                    if (!(lo <= (double)g.ny) || !(hi >= 1.0)) {
                        live = false;
                    } else {
                        lo = fmax(lo, 1.0);
                        hi = fmin(hi, (double)g.ny);
                        r0 = (int)lo;
                        r1 = (int)hi;
                    }
                }
            }
            if (!live) {
                r0 = 1;
                r1 = 0;
            }
            d.rows = (uint32_t)r0 | ((uint32_t)r1 << 16);
            // FP32 error band on the radicand (derivation in DESIGN.md):
            //   |s_f32 - s_real| <= 4*sqrt(s)*E + 2*E^2 + 2^-21*s,  E = 2^-21 * max(|cx|,|cy|,extent)
            // doubled for slack. Outside the window where that algebra holds, certify nothing.
            const float M = fmaxf(fmaxf(fabsf(d.cxf), fabsf(d.cyf)), g.extent);
            const float E = M * 4.76837158203125e-07f; // 2^-21
            const float Tf = d.Tf;
            if (Tf < 1e30f && M < 1e12f) {
                const float delta = 2.0f * (4.0f * sqrtf(Tf) * E + 2.0f * E * E + Tf * 9.5367431640625e-07f);
                d.thi = Tf + delta;
                d.tlo = (Tf > 64.0f * E * E) ? (Tf - delta) : -1.0f;
            } else {
                d.thi = __int_as_float(0x7f800000); // +Inf: nothing is certainly outside
                d.tlo = -1.0f;                      // nothing is certainly inside
            }
            dp[c] = d;
        }
    }
    CandScalars r;
    // --- penalty: strictly sequential FP64 sum in index order (one lane), then broadcast ---
    double viol = 0.0, prog = 0.0;
    if (lane == 0) {
        for (int i = 0; i < N; ++i) {
            const double diff = __dsub_rn(stage[2 * N + i], o.r_max[poff + i]);
            viol = __dadd_rn(viol, fabs(diff));
        }
        if (want_progressive)
            for (int i = 0; i < N; ++i) {
                const double diff = __dsub_rn(stage[2 * N + i], o.r_max[poff + i]);
                if (prog_takes(o, i)) prog = __dadd_rn(prog, julia_max0(diff));
            }
    }
    r.violation = __shfl_sync(0xffffffffu, viol, 0);
    r.progressive = __shfl_sync(0xffffffffu, prog, 0);
    // --- extreme constraints: order-free (a conjunction), so lane-parallel ---
    bool bad = false;
    if (o.use_cons3) {
        for (int i = lane; i < N; i += 32) {
            const double ax = __dsub_rn(o.prev_x[poff + i], stage[i]);
            const double ay = __dsub_rn(o.prev_y[poff + i], stage[N + i]);
            const double z2 = __ddiv_rn(stage[2 * N + i], o.tan_half_fov);
            const double az = __dsub_rn(o.prev_z[poff + i], z2);
            const double s =
                __dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az));
            bad |= (s >= o.cons3_G[poff + i]);
        }
    }
    if (o.use_cons7) {
        for (int i = lane; i < N; i += 32)
            bad |= (stage[N + i] < 200.0) && (stage[2 * N + i] > o.cons7_R);
    }
    if (o.use_cons8) {
        // (xi-xj)^2 is symmetric in i, j, so unordered pairs decide the ordered-pair loop
        for (int i = 0; i < N - 1; ++i) {
            const double xi = stage[i], yi = stage[N + i];
            for (int j = i + 1 + lane; j < N; j += 32) {
                const double ax = __dsub_rn(xi, stage[j]);
                const double ay = __dsub_rn(yi, stage[N + j]);
                const double s = __dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay));
                bad |= (s < o.sep_T);
            }
            if (__any_sync(0xffffffffu, bad)) break;
        }
    }
    r.feasible = !__any_sync(0xffffffffu, bad);
    return r;
}

// The store's own point list (g.ent_cell / g.ent_cls / g.n_ent), every entry live.
struct StoreList {
    const GridDesc &g;
    __device__ __forceinline__ long long size() const { return g.n_ent; }
    __device__ __forceinline__ bool get(long long p, int &cell, int &k) const
    {
        cell = g.ent_cell[p];
        k = g.ent_cls[p] & (kMaxClasses - 1);
        return true;
    }
};

// The reference's own loop (src/AreaCoverageCalculation.jl:63-110) over the point LIST for one candidate, executed
// by one warp: for each entry in list order, the first covering disc adds the entry's weight to a Float64 running
// sum.  32 entries are tested at a time and the covered ones added one after the other (every lane forms the same
// sum).  stage: the candidate's 3N doubles, Ts: the N thresholds T(R_c) (shared memory, visible to the warp).
// Returns the area; cls_total receives the covered entries per weight class.  list: the sequence walked, list.size()
// entries of which list.get(p, cell, k) reads entry p and says whether it is in the list (a dead entry adds nothing,
// so the sum is the one over the live entries alone, in the same order).
template <class List>
__device__ __forceinline__ double ordered_area(const GridDesc &g, int N, const double *stage, const double *Ts,
                                               long long *cls_total, const List &list)
{
    const uint32_t lane = lane_id();
    const double w0 = g.class_weight[0], w1 = g.class_weight[1], w2 = g.class_weight[2], w3 = g.class_weight[3];
#pragma unroll
    for (int k = 0; k < kMaxClasses; ++k) cls_total[k] = 0;
    double area = 0.0;
    const long long n_ent = list.size();
    for (long long p0 = 0; p0 < n_ent; p0 += 32) {
        const long long p = p0 + lane;
        bool cov_entry = false;
        int k = 0;
        int cell = 0;
        if (p < n_ent && list.get(p, cell, k)) {
            const double px = cell_centre(cell % g.nx + 1, g.dx, g.hdx);
            const double py = cell_centre(cell / g.nx + 1, g.dy, g.hdy);
            for (int c = 0; c < N; ++c) {
                if (radicand(px, py, stage[c], stage[N + c]) < Ts[c]) {
                    cov_entry = true;
                    break;
                }
            }
        }
        uint32_t m = __ballot_sync(0xffffffffu, cov_entry);
#pragma unroll
        for (int q = 0; q < kMaxClasses; ++q)
            cls_total[q] += __popc(__ballot_sync(0xffffffffu, cov_entry && k == q));
        while (m) { // list order = ascending lane
            const int b = __ffs(m) - 1;
            m &= m - 1;
            const int kb = __shfl_sync(0xffffffffu, k, b);
            area = __dadd_rn(area, kb == 0 ? w0 : (kb == 1 ? w1 : (kb == 2 ? w2 : w3)));
        }
    }
    return area;
}
__device__ __forceinline__ double ordered_area(const GridDesc &g, int N, const double *stage, const double *Ts,
                                               long long *cls_total)
{
    return ordered_area(g, N, stage, Ts, cls_total, StoreList{g});
}

} // namespace cov
