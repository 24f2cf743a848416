// cov_kernel_common.cuh -- device helpers shared by the coverage kernels (cov_kernels.cu: general
// span / brute / exact kernels; cov_span_small.cu: the small-swarm span kernel).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "cov_device.cuh"
#include "cov_types.h"

namespace cov {

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ float int_to_float_small(int i)
{
    // exact for 0 <= i < 2^23, one LOP3 + one FADD instead of an I2F conversion
    return __int_as_float(0x4B000000 | i) - 8388608.0f;
}

// Julia's max(a, 0.0) for Float64: NaN propagates, max(-0.0, 0.0) = 0.0.
__device__ __forceinline__ double julia_max0(double v) { return (v != v) ? v : (v > 0.0 ? v : 0.0); }

// The term UAV i (0-based) adds to the progressive output: every UAV for cons1_progressive, one fixed UAV for
// cons2_progressive / cons3_progressive (src/TDM_Constraints.jl:182-221; `0 + v` is exact, so the single-term
// forms equal max(R_k - r_max_k, 0.0) itself).
__device__ __forceinline__ bool prog_takes(const ObjParams &o, int i) { return o.prog_which == 0 || o.prog_which == i + 1; }

__host__ __device__ inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// The mirrors of EvalOut (device copies of objective and feasibility for the winner reduction).
__device__ __forceinline__ void store_mirrors(const EvalOut &out, long long idx, double obj, int feasible)
{
    if (out.obj_mirror) {
        out.obj_mirror[idx] = obj;
        out.feasible_mirror[idx] = (unsigned char)feasible;
    }
}

// obj = -area + violation*scale (src/TDM_STATIC_opt.jl:89-97)
__device__ __forceinline__ double objective_from_area(double area, double violation, const ObjParams &o)
{
    return __dadd_rn(-area, __dmul_rn(violation, o.penalty_scale));
}

// obj = -area + violation*scale, area from exact integer counts (see cov_grid_info.area_exact)
__device__ __forceinline__ double assemble_objective(const GridDesc &g, const ObjParams &o,
                                                     const long long *class_cnt, double violation)
{
    double area = 0.0;
    if (g.n_classes == 1) {
        area = __dmul_rn(g.class_weight[0], (double)class_cnt[0]);
    } else {
        for (int k = 0; k < g.n_classes; ++k)
            area = __dadd_rn(area, __dmul_rn(g.class_weight[k], (double)class_cnt[k]));
    }
    return objective_from_area(area, violation, o);
}

// ------------------------------------------------------------------------------------------
// exact FP64 pieces of the span search
// ------------------------------------------------------------------------------------------
struct RowExact {
    double cx, T, dy2, dx, hdx;
    int nx;
    __device__ __forceinline__ double px(int i) const { return cell_centre(i, dx, hdx); }
    __device__ __forceinline__ bool inside(int i) const
    {
        const double ddx = __dsub_rn(px(i), cx);
        return __dadd_rn(__dmul_rn(ddx, ddx), dy2) < T;
    }
};

// Exact [lo, hi] (1-based, inclusive; lo > hi: empty) of the covered columns of one row, walking
// from the estimates. Correct for ANY estimates: the covered set is contiguous and, if not empty,
// contains a cell next to the centre, because the FP64 radicand is non-increasing in i while
// px_i <= cx and non-decreasing while px_i >= cx (every rounding involved is monotone).
static __device__ __noinline__ void exact_span(const RowExact r, int lo_e, int hi_e, int &lo_out, int &hi_out)
{
    int i = min(max(lo_e, 1), r.nx);
    bool found = false;
    if (r.inside(i)) {
        found = true;
    } else if (r.px(i) < r.cx) { // left of the centre: the span, if any, starts to the right
        for (;;) {
            ++i;
            if (i > r.nx) break;
            if (r.inside(i)) {
                found = true;
                break;
            }
            if (!(r.px(i) < r.cx)) break; // passed the centre without a hit: empty row
        }
    } else { // at or right of the centre
        for (;;) {
            --i;
            if (i < 1) break;
            if (r.inside(i)) {
                found = true;
                break;
            }
            if (!(r.px(i) > r.cx)) break;
        }
    }
    if (!found) {
        lo_out = 1;
        hi_out = 0;
        return;
    }
    int lo = i;
    while (lo > 1 && r.inside(lo - 1)) --lo;
    int h = min(max(hi_e, i), r.nx);
    if (r.inside(h)) {
        while (h < r.nx && r.inside(h + 1)) ++h;
    } else {
        while (!r.inside(h)) --h; // stops at i at the latest
    }
    lo_out = lo;
    hi_out = h;
}

// ------------------------------------------------------------------------------------------
// shared-memory plumbing
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// TMA bulk copy global -> shared (1-D, 16-byte granular), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

template <bool SMEM>
__device__ __forceinline__ uint32_t ld_plane(const uint32_t *p)
{
    return SMEM ? *p : __ldg(p);
}

__device__ __forceinline__ void stage_planes(const GridDesc &g, uint32_t *planes_s, uint64_t *bar,
                                             int planes_bytes)
{
    // one elected thread issues TMA bulk copies of the (pre-padded) planes; everyone waits
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, (uint32_t)planes_bytes);
        const char *src = reinterpret_cast<const char *>(g.planes);
        char *dst = reinterpret_cast<char *>(planes_s);
        int left = planes_bytes;
        while (left > 0) {
            const int n = left > 65536 ? 65536 : left;
            bulk_g2s(dst, src, (uint32_t)n, bar);
            dst += n;
            src += n;
            left -= n;
        }
    }
    mbar_wait(bar, 0);
}


} // namespace cov
