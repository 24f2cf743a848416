// cov_region.cuh -- the grid-free static objective (cov_set_region / cov_eval_region_batch /
// cov_mads_solve_batch_region): the exact area A(x) = |(D_1 u ... u D_N) n Omega \ C| of the part of the domain
// Omega (a rectangle) that the candidate's discs D_i cover and the earlier swarms' discs C do not, by one warp.
//
// Green's theorem: A = 1/2 of the integral of (x dy - y dx) over the boundary of that region, which has three
// families of pieces:
//   1. arcs of candidate circle i inside Omega, outside the other candidate discs and outside C (counter-clockwise);
//   2. arcs of C's boundary inside Omega (the precomputed arc list) that lie inside some candidate disc (clockwise);
//   3. pieces of Omega's four edges inside some candidate disc and outside C (Omega's counter-clockwise sense).
// Each family is a set of covered parameter intervals (an angle on a circle, a coordinate on an edge).  The covered
// intervals go to the warp's list in shared memory (warp-aggregated appends, in lane order); an exposed piece starts
// at an interval end no other interval covers (or at the start of the range) and runs to the nearest interval start
// after it -- the method and tie rules of union_area_kernel / union_area_big_kernel (cov_grid_kernels.cu):
// `contained` is <=, and of identical discs the lower index survives, the covered discs counting before the candidate
// ones (so a candidate disc identical to a covered disc adds nothing).  Every lane sums its pieces in a fixed order and
// the lanes are reduced in a fixed order, so a candidate's area has the same bits wherever it is evaluated.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "cov_kernel_common.cuh"
#include "cov_candidate.cuh"
#include "cov_types.h"

namespace cov {

constexpr int kRegionMaxUavs = 64;      // N (one warp per candidate, lanes over the discs)
constexpr int kRegionMaxCovered = 512;  // M
constexpr int kRegionMaxArcs = 2048;    // arcs of C's boundary inside the domain
constexpr double kTwoPi = 6.283185307179586;
constexpr int kRegionThreads = 256; // 8 warps per CTA at most (fewer when the region's lists do not fit)
constexpr int kRegionCtas = 2;      // co-resident CTAs per SM the register budget is compiled for

// Shared memory: [covered discs 3M doubles | K arcs] once per CTA, then per warp [stage 3N doubles | 2 x cap doubles]
__host__ __device__ inline int region_list_cap(int N, int M) { return 2 * (N + M + 4) + 2; }
__host__ __device__ inline int region_smem_bytes(int M, int K) { return round_up(3 * M * 8 + K * 24, 16); }
__host__ __device__ inline int region_warp_bytes(int N, int M) { return round_up(3 * N * 8, 16) + 16 * region_list_cap(N, M); }

// Warps per CTA and dynamic shared-memory bytes for `fixed` bytes of other state; false when not even one warp fits.
inline bool region_plan(int N, int M, int K, int fixed, int max_smem, int *warps, int *smem)
{
    const int base = fixed + region_smem_bytes(M, K), per = region_warp_bytes(N, M);
    int w = kRegionThreads / 32;
    while (w > 1 && base + w * per > max_smem) --w;
    if (base + w * per > max_smem) return false;
    *warps = w;
    *smem = base + w * per;
    return true;
}

struct RegionView {
    const double *cx, *cy, *cr;
    const RegionArc *arcs;
    int M, K;
    double x_lo, y_lo, x_hi, y_hi;
};

// Copies the region into the CTA's shared memory (every thread takes part; the caller synchronises afterwards).
__device__ __forceinline__ RegionView region_stage(const RegionDesc &r, unsigned char *smem)
{
    double *d = reinterpret_cast<double *>(smem);
    RegionArc *arcs = reinterpret_cast<RegionArc *>(smem + 3 * r.M * 8);
    for (int t = threadIdx.x; t < 3 * r.M; t += blockDim.x) d[t] = r.discs[t];
    for (int t = threadIdx.x; t < r.K; t += blockDim.x) arcs[t] = r.arcs[t];
    return RegionView{d, d + r.M, d + 2 * r.M, arcs, r.M, r.K, r.x_lo, r.y_lo, r.x_hi, r.y_hi};
}

// region_stage for cov_run_horizon_region's covered set: M discs held at pitch `pitch` (r.discs: [x | y | R], each
// pitch doubles) and K arcs at r.arcs, both counts read on the device.  The shared-memory layout is region_stage's.
__device__ __forceinline__ RegionView cover_stage(const RegionDesc &r, int pitch, int M, int K, unsigned char *smem)
{
    double *d = reinterpret_cast<double *>(smem);
    RegionArc *arcs = reinterpret_cast<RegionArc *>(smem + 3 * M * 8);
    for (int t = threadIdx.x; t < M; t += blockDim.x) {
        d[t] = r.discs[t];
        d[M + t] = r.discs[pitch + t];
        d[2 * M + t] = r.discs[2 * pitch + t];
    }
    for (int t = threadIdx.x; t < K; t += blockDim.x) arcs[t] = r.arcs[t];
    return RegionView{d, d + M, d + 2 * M, arcs, M, K, r.x_lo, r.y_lo, r.x_hi, r.y_hi};
}

// 1/2 integral of (x dy - y dx) over the arc [t1, t2] of the circle (cx, cy, R), counter-clockwise.
__device__ __forceinline__ double arc_term(double R, double cx, double cy, double t1, double t2)
{
    double s1, c1, s2, c2;
    sincos(t1, &s1, &c1);
    sincos(t2, &s2, &c2);
    return 0.5 * (R * R * (t2 - t1) + R * (cx * (s2 - s1) - cy * (c2 - c1)));
}

// What disc j covers of circle i: 0 nothing (or a point), 1 the arc phi +- alpha, 2 all of it.  survives: circle i
// keeps its boundary when the two discs are identical (it has the lower index).
__device__ __forceinline__ int circle_vs_disc(double cxi, double cyi, double Ri, double cxj, double cyj, double Rj,
                                              bool survives, double &phi, double &alpha)
{
    const double dx = cxj - cxi, dy = cyj - cyi;
    const double d = hypot(dx, dy);
    if (d >= Ri + Rj) return 0;
    if (d + Ri <= Rj) return (d + Rj <= Ri && survives) ? 0 : 2;
    if (d + Rj <= Ri) return 0;
    phi = atan2(dy, dx);
    const double c = (Ri * Ri + d * d - Rj * Rj) / (2.0 * Ri * d);
    alpha = acos(fmax(-1.0, fmin(1.0, c)));
    return 1;
}

// Edge e of the domain: 0 bottom (y = y_lo), 1 right (x = x_hi), 2 top (y = y_hi), 3 left (x = x_lo).
// s: signed distance of (cx, cy) from the edge's line, positive on the domain's side.
__device__ __forceinline__ double edge_side(const RegionView &r, int e, double cx, double cy)
{
    return e == 0 ? cy - r.y_lo : (e == 1 ? r.x_hi - cx : (e == 2 ? r.y_hi - cy : cx - r.x_lo));
}

// What lies beyond edge e of circle (cx, cy, R): same codes as circle_vs_disc (the outward normal is phi).
__device__ __forceinline__ int circle_vs_edge(const RegionView &r, int e, double cx, double cy, double R, double &phi,
                                              double &alpha)
{
    const double s = edge_side(r, e, cx, cy);
    if (s >= R) return 0;
    if (s <= -R) return 2;
    phi = e == 0 ? 4.71238898038469 : (e == 1 ? 0.0 : (e == 2 ? 1.5707963267948966 : 3.141592653589793));
    alpha = acos(s / R);
    return 1;
}

// The chord of disc (cx, cy, R) on edge e as an interval of the edge coordinate (x - x_lo or y - y_lo), clipped to
// the edge; false when the disc does not reach the edge's inside.
__device__ __forceinline__ bool edge_chord(const RegionView &r, int e, double cx, double cy, double R, double &lo,
                                           double &hi)
{
    const double h = fabs(edge_side(r, e, cx, cy));
    if (!(h < R)) return false;
    const double w = sqrt((R - h) * (R + h));
    const double uc = (e & 1) ? cy - r.y_lo : cx - r.x_lo;
    const double L = (e & 1) ? r.y_hi - r.y_lo : r.x_hi - r.x_lo;
    lo = fmax(uc - w, 0.0);
    hi = fmin(uc + w, L);
    return lo < hi;
}

// phi +- alpha as one or two intervals of [0, 2 pi]; returns how many.
__device__ __forceinline__ int wrap_interval(double phi, double alpha, double &a0, double &b0, double &a1, double &b1)
{
    double a = fmod(phi - alpha, kTwoPi);
    if (a < 0.0) a += kTwoPi;
    const double e = a + 2.0 * alpha;
    a0 = a;
    if (e > kTwoPi) {
        b0 = kTwoPi;
        a1 = 0.0;
        b1 = e - kTwoPi;
        return 2;
    }
    b0 = e;
    return 1;
}

// Appends k (0, 1 or 2) intervals of every lane to the warp's list in lane order; returns the new length (warp-uniform).
__device__ __forceinline__ int warp_append(double *ia, double *ib, int n, int k, double a0, double b0, double a1,
                                           double b1)
{
    const uint32_t lane = lane_id();
    int incl = k;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, off);
        if ((int)lane >= off) incl += v;
    }
    const int at = n + incl - k;
    if (k >= 1) {
        ia[at] = a0;
        ib[at] = b0;
    }
    if (k == 2) {
        ia[at + 1] = a1;
        ib[at + 1] = b1;
    }
    return n + __shfl_sync(0xffffffffu, incl, 31);
}

// The exposed pieces of [lo, hi] given the n intervals of the list (all inside [lo, hi], visible to the warp):
// fn(has, pos, nxt) is called by every lane the same number of times, has = the lane holds the exposed piece
// [pos, nxt].  Among intervals with the same end the lowest list position speaks for all, and lo speaks for every
// end at lo.
template <class F>
__device__ __forceinline__ void for_each_exposed(const double *ia, const double *ib, int n, double lo, double hi, F &&fn)
{
    const int lane = (int)lane_id();
    for (int p0 = -1; p0 < n; p0 += 32) {
        const int p = p0 + lane;
        bool has = false;
        double pos = lo, nxt = hi;
        if (p < n) {
            pos = p < 0 ? lo : ib[p];
            bool covered = !(pos < hi) || (p >= 0 && pos == lo);
            for (int q = 0; q < n && !covered; ++q) {
                const double aq = ia[q], bq = ib[q];
                if (q != p && aq <= pos && (pos < bq || (pos == bq && q < p))) covered = true;
                if (aq > pos && aq < nxt) nxt = aq;
            }
            has = !covered && nxt > pos;
        }
        fn(has, pos, nxt);
    }
}

// The arcs of every covered circle m of r (r.M discs; r.arcs / r.K unused) that lie inside the domain and inside no
// other covered disc, in circle order and, per circle, in list order of their starts, by one warp; ia / ib: the warp's
// list, region_list_cap(0, M) doubles each.  Writes at most cap arcs to out and the count of all of them to *count
// (lane 0); every lane returns that count.
__device__ __forceinline__ int covered_arcs(const RegionView &v, double *ia, double *ib, RegionArc *out, int cap,
                                            int *count)
{
    const int M = v.M;
    const uint32_t lane = lane_id();
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
    return K;
}

// A(x) of the candidate in `st` (3N doubles, shared memory, visible to the warp), by one warp; ia / ib: the warp's
// list, region_list_cap(N, M) doubles each.  Every lane returns the area.
static __device__ __noinline__ double region_area(const RegionView &r, const double *st, int N, double *ia, double *ib)
{
    const uint32_t lane = lane_id();
    const double *sx = st, *sy = st + N, *sr = st + 2 * N;
    double acc = 0.0; // this lane's pieces, in a fixed order
    // 1. candidate arcs: blockers are the other candidate discs, the covered discs and the four edges
    const int nb = N + r.M + 4;
    for (int i = 0; i < N; ++i) {
        const double cxi = sx[i], cyi = sy[i], Ri = sr[i];
        if (!(Ri > 0.0)) continue; // warp-uniform
        int n = 0;
        bool whole = false;
        for (int j0 = 0; j0 < nb && !whole; j0 += 32) {
            const int j = j0 + (int)lane;
            int rel = 0;
            double phi = 0.0, alpha = 0.0;
            if (j < N) {
                if (j != i && sr[j] > 0.0) rel = circle_vs_disc(cxi, cyi, Ri, sx[j], sy[j], sr[j], i < j, phi, alpha);
            } else if (j < N + r.M) {
                const int m = j - N;
                rel = circle_vs_disc(cxi, cyi, Ri, r.cx[m], r.cy[m], r.cr[m], false, phi, alpha);
            } else if (j < nb) {
                rel = circle_vs_edge(r, j - N - r.M, cxi, cyi, Ri, phi, alpha);
            }
            whole = __any_sync(0xffffffffu, rel == 2);
            double a0 = 0, b0 = 0, a1 = 0, b1 = 0;
            const int k = rel == 1 ? wrap_interval(phi, alpha, a0, b0, a1, b1) : 0;
            n = warp_append(ia, ib, n, k, a0, b0, a1, b1);
        }
        __syncwarp();
        if (!whole)
            for_each_exposed(ia, ib, n, 0.0, kTwoPi, [&](bool has, double pos, double nxt) {
                if (has) acc += arc_term(Ri, cxi, cyi, pos, nxt);
            });
        __syncwarp(); // the list is rewritten for the next circle
    }
    // 2. arcs of C's boundary: the part of [a, b] inside the candidate discs = [a, b] less its exposed pieces, where
    //    the rest of the circle ([0, a] and [b, 2 pi]) counts as covered
    for (int k = 0; k < r.K; ++k) {
        const RegionArc arc = r.arcs[k];
        const double cxm = r.cx[arc.m], cym = r.cy[arc.m], Rm = r.cr[arc.m];
        int n = 0;
        if (lane == 0) {
            if (arc.a > 0.0) {
                ia[n] = 0.0;
                ib[n++] = arc.a;
            }
            if (arc.b < kTwoPi) {
                ia[n] = arc.b;
                ib[n++] = kTwoPi;
            }
        }
        n = __shfl_sync(0xffffffffu, n, 0);
        bool whole = false, touched = false;
        for (int j0 = 0; j0 < N && !whole; j0 += 32) {
            const int j = j0 + (int)lane;
            int rel = 0;
            double phi = 0.0, alpha = 0.0;
            if (j < N && sr[j] > 0.0) rel = circle_vs_disc(cxm, cym, Rm, sx[j], sy[j], sr[j], true, phi, alpha);
            whole = __any_sync(0xffffffffu, rel == 2);
            touched |= __any_sync(0xffffffffu, rel == 1);
            double a0 = 0, b0 = 0, a1 = 0, b1 = 0;
            const int q = rel == 1 ? wrap_interval(phi, alpha, a0, b0, a1, b1) : 0;
            n = warp_append(ia, ib, n, q, a0, b0, a1, b1);
        }
        __syncwarp();
        if (whole) {
            if (lane == 0) acc -= arc_term(Rm, cxm, cym, arc.a, arc.b);
        } else if (touched) {
            double ex = 0.0;
            for_each_exposed(ia, ib, n, 0.0, kTwoPi, [&](bool has, double pos, double nxt) {
                if (has) ex += arc_term(Rm, cxm, cym, pos, nxt);
            });
            acc -= (lane == 0 ? arc_term(Rm, cxm, cym, arc.a, arc.b) : 0.0) - ex;
        }
        __syncwarp();
    }
    // 3. edges: the length of (candidate chords) less (covered chords) = exposed(C) - exposed(C and candidates)
    for (int e = 0; e < 4; ++e) {
        bool reach = false;
        for (int j = (int)lane; j < N; j += 32) {
            double lo, hi;
            if (sr[j] > 0.0 && edge_chord(r, e, sx[j], sy[j], sr[j], lo, hi)) reach = true;
        }
        if (!__any_sync(0xffffffffu, reach)) continue;
        const double L = (e & 1) ? r.y_hi - r.y_lo : r.x_hi - r.x_lo;
        const double coef = e == 0 ? -0.5 * r.y_lo : (e == 1 ? 0.5 * r.x_hi : (e == 2 ? 0.5 * r.y_hi : -0.5 * r.x_lo));
        int n = 0;
        for (int j0 = 0; j0 < r.M; j0 += 32) { // the covered chords
            const int j = j0 + (int)lane;
            double lo = 0, hi = 0;
            const bool has = j < r.M && edge_chord(r, e, r.cx[j], r.cy[j], r.cr[j], lo, hi);
            n = warp_append(ia, ib, n, has ? 1 : 0, lo, hi, 0.0, 0.0);
        }
        __syncwarp();
        for_each_exposed(ia, ib, n, 0.0, L, [&](bool has, double pos, double nxt) {
            if (has) acc += coef * (nxt - pos);
        });
        for (int j0 = 0; j0 < N; j0 += 32) { // and the candidates' after them
            const int j = j0 + (int)lane;
            double lo = 0, hi = 0;
            const bool has = j < N && sr[j] > 0.0 && edge_chord(r, e, sx[j], sy[j], sr[j], lo, hi);
            n = warp_append(ia, ib, n, has ? 1 : 0, lo, hi, 0.0, 0.0);
        }
        __syncwarp();
        for_each_exposed(ia, ib, n, 0.0, L, [&](bool has, double pos, double nxt) {
            if (has) acc -= coef * (nxt - pos);
        });
        __syncwarp();
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
    return __shfl_sync(0xffffffffu, acc, 0);
}

// The objective of the candidate in `stage` by one warp: obj = -A + penalty_scale * sum |R_i - r_max_i| in the grid
// objective's FP64 order, with A and the fused constraints' verdict.  The constraints are candidate_prologue's.
__device__ __forceinline__ double region_objective(const RegionView &r, const ObjParams &o, const double *stage,
                                                   double *ia, double *ib, double &area, int &feasible)
{
    const CandScalars cs = candidate_prologue<false>(GridDesc{}, o, stage, nullptr, false); // reads no grid
    area = region_area(r, stage, o.N, ia, ib);
    feasible = cs.feasible;
    return objective_from_area(area, cs.violation, o);
}

} // namespace cov
