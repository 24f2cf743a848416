// cov_mads.cu -- the device-resident multi-start MADS solver of libcoverage_cuda (sm_100a): S independent solves
// in ONE launch (cov_mads_solve_batch).
//
// Persistent CTAs take solves from an atomic dispenser; a CTA runs one solve from its first evaluation to its
// result, then takes the next.  No CTA talks to another.  Per iteration of a solve:
//   1. warp 0 draws the Householder vector v (Irwin-Hall(12) normals from Philox, see coverage_cuda.h) and
//      normalises it; every thread sets the mesh and poll sizes of its variables;
//   2. __syncthreads;
//   3. warp w builds poll points k = w, w + W, ... (column k mod n of I - 2 v v^T, scaled, rounded onto the mesh,
//      sign + for k < n, - after) into its own stage and applies cov_mads_solve's drop rules;
//   4. the warp evaluates every kept point (candidate_prologue, then the row spans of make_sdisc / fast_span /
//      slow_item painted into the warp's framebuffer, or the list-order loop for non-dyadic weights) and stores
//      the barrier value f[k] (NaN marks a dropped point);
//   5. __syncthreads;
//   6. thread 0 picks the first strict minimum in generation order; the incumbent is re-built from its index
//      (the same arithmetic, so the same bits) and the mesh enlarged, or the mesh refined / the solve stopped.
// Everything is cov_mads_solve's loop (cov_api.cu) in the same FP64 operations and order, so a host model can
// replay every iterate bit for bit; only the direction stream and the absence of a cache differ.
// region_solve_kernel (cov_mads_solve_batch_region) runs the same loop (mads_solves) with step 4 replaced by the
// region objective of cov_region.cuh, the device function cov_eval_region_batch's kernel calls.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "cov_device.cuh"
#include "cov_kernel_common.cuh"
#include "cov_candidate.cuh"
#include "cov_span_common.cuh"
#include "cov_kernels.cuh"
#include "cov_region.cuh"

namespace cov {

constexpr int kMadsThreads = 256; // 8 warps: 30 poll points of a 5-UAV swarm are 4 rounds of one point per warp
constexpr int kMadsCtas = 2;      // co-resident CTAs per SM the register budget is compiled for

// Shared memory of a CTA: [planes (optional)] [solve state] [W x per-warp] [mbarrier]
__host__ __device__ inline int mads_state_bytes(int n) { return round_up(7 * n * 8 + 2 * n * 4, 16) + 64; }
__host__ __device__ inline int mads_fb_bytes(const GridDesc &g, int N)
{
    const int fb = round_up(g.ny * g.stride * 4, 16), ts = round_up(N * 8, 16);
    return fb > ts ? fb : ts; // the list-order path keeps the N thresholds there instead
}
__host__ __device__ inline int mads_warp_bytes(const GridDesc &g, int N)
{
    return round_up(3 * N * 8, 16) + N * 32 + round_up(N * 4, 16) + mads_fb_bytes(g, N);
}

struct MadsShared {
    double fx, nrm;
    unsigned long long solve;
    int kb, feasible_found;
};

__device__ __forceinline__ double max_host(double a, double b) { return (a < b) ? b : a; } // std::max

__device__ __forceinline__ double pow10_of(const MadsArgs &a, int b)
{
    b = b < kMadsPow10Min ? kMadsPow10Min : (b > -kMadsPow10Min ? -kMadsPow10Min : b);
    return __ldg(a.pow10 + (b - kMadsPow10Min));
}

// v_i = (sum of the 12 words of the blocks (t lo, t hi, i, 0..2)) * 2^-32 - 6: exact in binary64
__device__ __forceinline__ double irwin_hall(uint32_t k0, uint32_t k1, unsigned long long t, int i)
{
    unsigned long long s = 0;
#pragma unroll
    for (uint32_t q = 0; q < 3; ++q) {
        uint32_t r[4];
        philox4x32_10((uint32_t)t, (uint32_t)(t >> 32), (uint32_t)i, q, k0, k1, r);
        s += (unsigned long long)r[0] + r[1] + r[2] + r[3];
    }
    return __dsub_rn(__dmul_rn((double)s, 2.3283064365386962890625e-10), 6.0);
}

// Poll point kk (column kk mod n, sign + for kk < n) of cov_mads_solve, built by one warp into dst (which may be x
// itself).  Returns whether cov_mads_solve keeps it: some rounded direction component is non-zero and the snapped
// point differs from x.
__device__ __forceinline__ bool poll_point(int kk, int n, const double *x, const double *v, const double *rho,
                                           const double *delta, double gran, double *dst)
{
    const uint32_t lane = lane_id();
    const bool neg = kk >= n;
    const int j = neg ? kk - n : kk;
    const double sgn = neg ? -1.0 : 1.0;
    const double vj = v[j];
    double hmax = 0.0; // a maximum of non-NaN values (NaN components never win std::max), so any order gives it
    for (int i = lane; i < n; i += 32) {
        const double H = __dsub_rn(i == j ? 1.0 : 0.0, __dmul_rn(__dmul_rn(2.0, v[i]), vj));
        hmax = max_host(hmax, fabs(H));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) hmax = max_host(hmax, __shfl_xor_sync(0xffffffffu, hmax, off));
    bool any = false, moved = false;
    for (int i = lane; i < n; i += 32) {
        const double H = __dsub_rn(i == j ? 1.0 : 0.0, __dmul_rn(__dmul_rn(2.0, v[i]), vj));
        const double d = rint(__ddiv_rn(__dmul_rn(rho[i], H), hmax));
        any |= d != 0.0;
        const double xi = x[i];
        double p = __dadd_rn(xi, __dmul_rn(__dmul_rn(sgn, d), delta[i]));
        if (gran > 0) p = __dmul_rn(rint(__ddiv_rn(p, gran)), gran);
        moved |= p != xi;
        dst[i] = p;
    }
    return __any_sync(0xffffffffu, any) && __any_sync(0xffffffffu, moved);
}

// The objective with the extreme barrier for the candidate in `stage`, by one warp: +Inf where a fused constraint
// fails (its coverage is never counted) or the objective is NaN.  fb: the warp's framebuffer, all-zero on entry and
// on return (the list-order path keeps the thresholds there instead and never paints it).  poff: the parameter
// block's offset (candidate_prologue); barrier = false: AreaMaxObjective itself, as the objective kernels give it.
template <bool MULTI, bool PLANES_SMEM>
__device__ double mads_eval(const GridDesc &g, const ObjParams &o, const double *stage, SDisc *sd, int *pre,
                            uint32_t *fb, const uint32_t *planes, int force_exact, int ordered, long long poff = 0,
                            bool barrier = true)
{
    const int N = o.N;
    const uint32_t lane = lane_id();
    const CandScalars cs = candidate_prologue<false>(g, o, stage, nullptr, false, poff);
    if (barrier && !cs.feasible) return __longlong_as_double(0x7ff0000000000000ll);
    double obj;
    long long cls[kMaxClasses];
    if (ordered) {
        double *Ts = reinterpret_cast<double *>(fb);
        for (int c = lane; c < N; c += 32) Ts[c] = threshold(stage[2 * N + c]);
        __syncwarp();
        const double area = ordered_area(g, N, stage, Ts, cls);
        __syncwarp();
        obj = __dadd_rn(-area, __dmul_rn(cs.violation, o.penalty_scale));
    } else {
        for (int c = lane; c < N; c += 32) make_sdisc(g, stage[c], stage[N + c], stage[2 * N + c], sd[c]);
        __syncwarp();
        // (disc, row) items flattened over the lanes: inclusive prefix of the discs' row counts, and the rows the
        // framebuffer has to be cleared on afterwards
        int total = 0, rmin = g.ny + 1, rmax = 0;
        if (lane == 0) {
            for (int c = 0; c < N; ++c) {
                const int r0 = (int)(sd[c].rows & 0xffffu), r1 = (int)(sd[c].rows >> 16);
                if (r1 >= r0) {
                    total += r1 - r0 + 1;
                    rmin = min(rmin, r0);
                    rmax = max(rmax, r1);
                }
                pre[c] = total;
            }
        }
        total = __shfl_sync(0xffffffffu, total, 0);
        rmin = __shfl_sync(0xffffffffu, rmin, 0);
        rmax = __shfl_sync(0xffffffffu, rmax, 0);
        __syncwarp();
        uint32_t cnt[MULTI ? kMaxClasses : 1];
#pragma unroll
        for (int k = 0; k < (MULTI ? kMaxClasses : 1); ++k) cnt[k] = 0;
        const FbLayout fl{g.stride, 0};
        for (int tb = 0; tb < total; tb += 32) {
            const int t = tb + (int)lane;
            const bool has = t < total;
            int c = 0;
            if (has)
                while (pre[c] <= t) ++c;
            const SDisc d = sd[c];
            const int j = has ? (int)(d.rows & 0xffffu) + t - (c ? pre[c - 1] : 0) : 1;
            int lo, hi;
            int st = fast_span(g, d, j, force_exact, lo, hi);
            if (!has) st = kEmpty;
            if (st == kSlow) {
                slow_item(g, stage, N, c, j, (d.flags & 1u) || force_exact, lo, hi);
                if (lo <= hi) st = kSpan;
                else {
                    st = kEmpty;
                    lo = hi = 1;
                }
            }
            // every disc goes through the framebuffer: a lane counts only the bits it was first to set
            paint_span<MULTI, PLANES_SMEM>(g, fb, planes, j, lo, hi, st == kSpan, true, cnt, 1, fl);
        }
        __syncwarp();
        if (rmax >= rmin)
            for (int w = (rmin - 1) * g.stride + (int)lane; w < rmax * g.stride; w += 32) fb[w] = 0u;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < kMaxClasses; ++k)
            cls[k] = k < (MULTI ? kMaxClasses : 1) ? (long long)__reduce_add_sync(0xffffffffu, cnt[MULTI ? k : 0]) : 0;
        obj = assemble_objective(g, o, cls, cs.violation);
    }
    return (obj == obj || !barrier) ? obj : __longlong_as_double(0x7ff0000000000000ll);
}

// The solves of cov_mads_solve_batch from the dispenser `counter` until none is left, by the whole CTA: the loop
// shared by mads_kernel (the grid objective), scenario_solve_kernel (the grid objective of several stores) and
// region_solve_kernel (the region objective).  state: mads_state_bytes(n) bytes of shared memory; stage: the calling
// warp's 3N doubles; key_of(k): the Philox key of solve k, called by every thread before the solve's first evaluation;
// eval(p): the barrier value of the point p (shared memory) by the calling warp.
template <class Key, class Eval>
__device__ __forceinline__ void mads_solves(const MadsArgs &a, int n, unsigned char *state, double *stage,
                                            unsigned long long *counter, const Key &key_of, const Eval &eval)
{
    const int W = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    double *x = reinterpret_cast<double *>(state);
    double *v = x + n, *rho = v + n, *delta = rho + n, *am = delta + n, *f = am + n; // f: 2n
    int *bm = reinterpret_cast<int *>(f + 2 * n), *bz = bm + n;
    MadsShared *sh = reinterpret_cast<MadsShared *>(state + round_up(7 * n * 8 + 2 * n * 4, 16));
    const double gran = a.granularity;
    const int tid = threadIdx.x, nthr = blockDim.x;

    for (;;) {
        if (tid == 0) sh->solve = atomicAdd(counter, 1ull);
        __syncthreads();
        const unsigned long long k = sh->solve;
        if ((long long)k >= a.S) break;
        const unsigned long long key = key_of(k);
        const double *x0 = a.X0 + (long long)k * n;
        for (int i = tid; i < n; i += nthr) {
            x[i] = x0[i];
            am[i] = a.a0[(long long)k * n + i];
            bm[i] = bz[i] = a.b0[(long long)k * n + i];
        }
        __syncthreads();
        if (warp == 0) {
            const double f0 = eval(x);
            if (lane == 0) {
                sh->fx = f0;
                sh->feasible_found = isfinite(f0) ? 1 : 0;
            }
        }
        long long iterations = 0, evaluations = 1, successes = 0; // kept by thread 0
        int converged = 0;
        for (long long it = 0; it < a.n_iter; ++it) {
            ++iterations;
            for (int i = tid; i < n; i += nthr) {
                const double Delta = max_host(__dmul_rn(am[i], pow10_of(a, bm[i])), gran);
                const int e = bm[i] - abs(bm[i] - bz[i]);
                delta[i] = max_host(pow10_of(a, e), gran);
                rho[i] = max_host(rint(__ddiv_rn(Delta, delta[i])), 1.0);
            }
            if (warp == 0) {
                for (int i = lane; i < n; i += 32) v[i] = irwin_hall((uint32_t)key, (uint32_t)(key >> 32), it, i);
                __syncwarp();
                if (lane == 0) {
                    double s = 0.0;
                    for (int i = 0; i < n; ++i) s = __dadd_rn(s, __dmul_rn(v[i], v[i]));
                    sh->nrm = __dsqrt_rn(s);
                }
                __syncwarp();
                const double nrm = sh->nrm;
                for (int i = lane; i < n; i += 32) v[i] = __ddiv_rn(v[i], nrm);
            }
            __syncthreads();
            for (int kk = warp; kk < 2 * n; kk += W) {
                const bool keep = poll_point(kk, n, x, v, rho, delta, gran, stage);
                __syncwarp();
                double fk = __longlong_as_double(0x7ff8000000000000ll); // dropped
                if (keep) fk = eval(stage);
                if (lane == 0) f[kk] = fk;
                __syncwarp();
            }
            __syncthreads();
            if (tid == 0) {
                double best = __longlong_as_double(0x7ff0000000000000ll);
                int kb = -1;
                for (int kk = 0; kk < 2 * n; ++kk) {
                    const double fk = f[kk];
                    if (fk != fk) continue;
                    ++evaluations;
                    if (fk < best) {
                        best = fk;
                        kb = kk;
                    }
                }
                const bool success = kb >= 0 && (best < sh->fx || (!sh->feasible_found && isfinite(best)));
                sh->kb = success ? kb : -1;
                if (success) {
                    sh->fx = best;
                    sh->feasible_found = 1;
                    ++successes;
                }
            }
            __syncthreads();
            const int kb = sh->kb;
            if (kb >= 0) {
                if (warp == 0) poll_point(kb, n, x, v, rho, delta, gran, x); // the winner, re-built in place
                for (int i = tid; i < n; i += nthr) { // enlarge
                    if (am[i] == 1.0) am[i] = 2.0;
                    else if (am[i] == 2.0) am[i] = 5.0;
                    else {
                        am[i] = 1.0;
                        ++bm[i];
                    }
                }
                __syncthreads(); // x, rho and delta are read by the rebuild and rewritten by the next iteration
            } else { // refine; stop when every poll size sits at its granularity
                bool moved = false;
                for (int i = tid; i < n; i += nthr) {
                    if (gran > 0 && __dmul_rn(am[i], pow10_of(a, bm[i])) <= gran) continue;
                    if (am[i] == 1.0) {
                        am[i] = 5.0;
                        --bm[i];
                    } else if (am[i] == 2.0) am[i] = 1.0;
                    else am[i] = 2.0;
                    moved = true;
                }
                if (!__syncthreads_or(moved)) {
                    converged = 1;
                    break;
                }
            }
        }
        __syncthreads();
        const bool found = sh->feasible_found != 0;
        for (int i = tid; i < n; i += nthr) a.X_out[(long long)k * n + i] = found ? x[i] : x0[i];
        if (tid == 0) {
            a.obj_out[k] = sh->fx;
            long long *st = a.stats + 4 * (long long)k;
            st[0] = iterations;
            st[1] = evaluations;
            st[2] = successes;
            st[3] = converged;
        }
        __syncthreads(); // the state and the dispenser slot are rewritten by the next solve
    }
}

template <bool MULTI, bool PLANES_SMEM, int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS)
mads_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o, const __grid_constant__ MadsArgs a,
            unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int W = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N, n = 3 * N;
    const int planes_bytes = PLANES_SMEM ? g.n_planes * g.plane_words * 4 : 0;
    const int warp_bytes = mads_warp_bytes(g, N);
    uint32_t *planes_s = reinterpret_cast<uint32_t *>(smem_raw);
    unsigned char *sbase = smem_raw + planes_bytes;
    unsigned char *wbase = sbase + mads_state_bytes(n) + (size_t)warp * warp_bytes;
    double *stage = reinterpret_cast<double *>(wbase);
    SDisc *sd = reinterpret_cast<SDisc *>(wbase + round_up(3 * N * 8, 16));
    int *pre = reinterpret_cast<int *>(wbase + round_up(3 * N * 8, 16) + N * 32);
    uint32_t *fb = reinterpret_cast<uint32_t *>(wbase + round_up(3 * N * 8, 16) + N * 32 + round_up(N * 4, 16));
    uint64_t *bar = reinterpret_cast<uint64_t *>(sbase + mads_state_bytes(n) + (size_t)W * warp_bytes);

    if (PLANES_SMEM) stage_planes(g, planes_s, bar, planes_bytes); // TMA bulk copy, once per CTA (syncs)
    const uint32_t *planes = PLANES_SMEM ? planes_s : g.planes;
    for (int t = lane; t < mads_fb_bytes(g, N) / 16; t += 32) reinterpret_cast<uint4 *>(fb)[t] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    mads_solves(a, n, sbase, stage, counter, [&](unsigned long long k) { return a.seed + k; }, [&](const double *p) {
        return mads_eval<MULTI, PLANES_SMEM>(g, o, p, sd, pre, fb, planes, a.force_exact, a.ordered);
    });
}

// The solves of E scenarios (launch_scenario_mads): mads_kernel's shared-memory layout without the staged planes.
// Solve k belongs to scenario k / S, whose plane set is read through L2 (E stores rarely fit one SM's shared memory,
// and consecutive solves of a persistent CTA belong to different scenarios).
template <bool MULTI>
__global__ void __launch_bounds__(kMadsThreads, kMadsCtas)
scenario_solve_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
                      const __grid_constant__ MadsArgs a, long long S, unsigned long long key_stride,
                      unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N, n = 3 * N;
    const int warp_bytes = mads_warp_bytes(g, N);
    unsigned char *wbase = smem_raw + mads_state_bytes(n) + (size_t)warp * warp_bytes;
    double *stage = reinterpret_cast<double *>(wbase);
    SDisc *sd = reinterpret_cast<SDisc *>(wbase + round_up(3 * N * 8, 16));
    int *pre = reinterpret_cast<int *>(wbase + round_up(3 * N * 8, 16) + N * 32);
    uint32_t *fb = reinterpret_cast<uint32_t *>(wbase + round_up(3 * N * 8, 16) + N * 32 + round_up(N * 4, 16));
    for (int t = lane; t < mads_fb_bytes(g, N) / 16; t += 32) reinterpret_cast<uint4 *>(fb)[t] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    const long long pstride = (long long)g.n_planes * g.plane_words;
    long long e = 0; // the scenario of the current solve
    mads_solves(
        a, n, smem_raw, stage, counter,
        [&](unsigned long long k) {
            e = (long long)(k / (unsigned long long)S);
            return a.seed + (unsigned long long)e * key_stride + (k - (unsigned long long)e * S);
        },
        [&](const double *p) {
            return mads_eval<MULTI, false>(g, o, p, sd, pre, fb, g.planes + e * pstride, a.force_exact, 0, e * 5 * N);
        });
}

// AreaMaxObjective of E swarms, one warp per swarm (launch_scenario_eval).  Shared memory: W x mads_warp_bytes.
template <bool MULTI>
__global__ void __launch_bounds__(kMadsThreads)
scenario_eval_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
                     const double *__restrict__ X, long long E, int force_exact, double *__restrict__ obj)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int W = blockDim.x >> 5, warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N, n = 3 * N;
    const long long e = (long long)blockIdx.x * W + warp;
    if (e >= E) return;
    unsigned char *wbase = smem_raw + (size_t)warp * mads_warp_bytes(g, N);
    double *stage = reinterpret_cast<double *>(wbase);
    SDisc *sd = reinterpret_cast<SDisc *>(wbase + round_up(3 * N * 8, 16));
    int *pre = reinterpret_cast<int *>(wbase + round_up(3 * N * 8, 16) + N * 32);
    uint32_t *fb = reinterpret_cast<uint32_t *>(wbase + round_up(3 * N * 8, 16) + N * 32 + round_up(N * 4, 16));
    for (int t = lane; t < mads_fb_bytes(g, N) / 16; t += 32) reinterpret_cast<uint4 *>(fb)[t] = make_uint4(0, 0, 0, 0);
    for (int i = lane; i < n; i += 32) stage[i] = X[e * n + i];
    __syncwarp();
    const double f = mads_eval<MULTI, false>(g, o, stage, sd, pre, fb, g.planes + e * g.n_planes * (long long)g.plane_words,
                                             force_exact, 0, e * 5 * N, false);
    if (lane == 0) obj[e] = f;
}

bool mads_plan(const GridDesc &g, int N, const LaunchCfg &cfg, int *warps, int *smem, int *planes_smem)
{
    if (N < 1 || N > kMadsMaxUavs) return false;
    const int planes_bytes = g.n_planes * g.plane_words * 4;
    const int fixed = mads_state_bytes(3 * N) + 16, per_warp = mads_warp_bytes(g, N);
    int w = kMadsThreads / 32;
    while (w > 1 && fixed + w * per_warp > cfg.max_smem_optin) w /= 2;
    if (fixed + w * per_warp > cfg.max_smem_optin) return false;
    const bool ps = planes_bytes + fixed + w * per_warp <= cfg.max_smem_optin;
    *warps = w;
    *smem = (ps ? planes_bytes : 0) + fixed + w * per_warp;
    *planes_smem = ps;
    return true;
}

template <bool M, bool P>
static cudaError_t launch_mads_variant(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                                       unsigned long long *counter, cudaStream_t stream, int warps, int smem)
{
    auto kern = mads_kernel<M, P, kMadsThreads, kMadsCtas>;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem);
    if (err != cudaSuccess) return err;
    const int grid = (int)std::min<long long>(a.S, (long long)cfg.num_sms * std::max(per_sm, 1));
    kern<<<grid, warps * 32, smem, stream>>>(g, o, a, counter);
    return cudaGetLastError();
}

static bool plane_multi(const GridDesc &g) { return !(g.n_planes == 1 && g.n_classes == 1 && g.plane_mult[0] == 1); }

cudaError_t launch_mads(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                        unsigned long long *counter, cudaStream_t stream)
{
    if (a.S <= 0) return cudaSuccess;
    int warps = 0, smem = 0, ps = 0;
    if (!mads_plan(g, o.N, cfg, &warps, &smem, &ps)) return cudaErrorInvalidConfiguration;
    if (plane_multi(g)) return ps ? launch_mads_variant<true, true>(g, o, cfg, a, counter, stream, warps, smem)
                                  : launch_mads_variant<true, false>(g, o, cfg, a, counter, stream, warps, smem);
    return ps ? launch_mads_variant<false, true>(g, o, cfg, a, counter, stream, warps, smem)
              : launch_mads_variant<false, false>(g, o, cfg, a, counter, stream, warps, smem);
}

// Persistent CTAs of kern with smem bytes, at most `work` of them.
template <class K>
static cudaError_t persistent_grid(K kern, int threads, int smem, long long work, const LaunchCfg &cfg, int *grid)
{
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    if (err != cudaSuccess) return err;
    *grid = (int)std::min<long long>(work, (long long)cfg.num_sms * std::max(per_sm, 1));
    return cudaSuccess;
}

cudaError_t launch_scenario_mads(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                                 long long S, unsigned long long key_stride, unsigned long long *counter,
                                 cudaStream_t stream)
{
    if (a.S <= 0) return cudaSuccess;
    int warps = 0, smem = 0, ps = 0;
    if (!mads_plan(g, o.N, cfg, &warps, &smem, &ps)) return cudaErrorInvalidConfiguration;
    if (ps) smem -= g.n_planes * g.plane_words * 4; // the planes stay in global memory
    auto kern = plane_multi(g) ? scenario_solve_kernel<true> : scenario_solve_kernel<false>;
    int grid = 0;
    cudaError_t err = persistent_grid(kern, warps * 32, smem, a.S, cfg, &grid);
    if (err != cudaSuccess) return err;
    kern<<<grid, warps * 32, smem, stream>>>(g, o, a, S, key_stride, counter);
    return cudaGetLastError();
}

cudaError_t launch_scenario_eval(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *X,
                                 long long E, double *obj, cudaStream_t stream)
{
    if (E <= 0) return cudaSuccess;
    int warps = 0, smem = 0, ps = 0;
    if (!mads_plan(g, o.N, cfg, &warps, &smem, &ps)) return cudaErrorInvalidConfiguration;
    smem = warps * mads_warp_bytes(g, o.N);
    auto kern = plane_multi(g) ? scenario_eval_kernel<true> : scenario_eval_kernel<false>;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    kern<<<(unsigned)((E + warps - 1) / warps), warps * 32, smem, stream>>>(g, o, X, E, cfg.force_exact, obj);
    return cudaGetLastError();
}

// The solves of cov_mads_solve_batch with the region objective.  Shared memory: [solve state] [region] [W x (stage,
// interval lists)].
template <int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS)
region_solve_kernel(const __grid_constant__ RegionDesc r, const __grid_constant__ ObjParams o,
                    const __grid_constant__ MadsArgs a, unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = o.N, n = 3 * N, warp = threadIdx.x >> 5;
    unsigned char *rbase = smem_raw + mads_state_bytes(n);
    const RegionView v = region_stage(r, rbase);
    unsigned char *wbase = rbase + region_smem_bytes(r.M, r.K) + (size_t)warp * region_warp_bytes(N, r.M);
    double *stage = reinterpret_cast<double *>(wbase);
    double *ia = reinterpret_cast<double *>(wbase + round_up(3 * N * 8, 16)), *ib = ia + region_list_cap(N, r.M);
    __syncthreads();
    mads_solves(a, n, smem_raw, stage, counter, [&](unsigned long long k) { return a.seed + k; },
                [&](const double *p) { // region_objective with the extreme barrier
        const CandScalars cs = candidate_prologue<false>(GridDesc{}, o, p, nullptr, false);
        if (!cs.feasible) return __longlong_as_double(0x7ff0000000000000ll);
        const double obj = objective_from_area(region_area(v, p, N, ia, ib), cs.violation, o);
        return (obj == obj) ? obj : __longlong_as_double(0x7ff0000000000000ll);
    });
}

cudaError_t launch_mads_region(const RegionDesc &r, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                               unsigned long long *counter, cudaStream_t stream)
{
    if (a.S <= 0) return cudaSuccess;
    int warps = 0, smem = 0;
    if (o.N > kRegionMaxUavs ||
        !region_plan(o.N, r.M, r.K, mads_state_bytes(3 * o.N), cfg.max_smem_optin - 1024 /* the kernel's static shared memory */, &warps, &smem))
        return cudaErrorInvalidConfiguration;
    auto kern = region_solve_kernel<kRegionThreads, kRegionCtas>;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem);
    if (err != cudaSuccess) return err;
    const int grid = (int)std::min<long long>(a.S, (long long)cfg.num_sms * std::max(per_sm, 1));
    kern<<<grid, warps * 32, smem, stream>>>(r, o, a, counter);
    return cudaGetLastError();
}

// region_solve_kernel on cov_run_horizon_region's covered set: M and K read from c.ctl, the discs staged from their
// pitch.  The shared-memory plan is the call's worst case (c.pitch discs, kRegionMaxArcs arcs), fixed for every
// timestep; a candidate's area does not depend on the lists' capacity or on the warps per CTA, so the solves give
// region_solve_kernel's bits.
__global__ void __launch_bounds__(kRegionThreads, kRegionCtas)
cover_solve_kernel(const __grid_constant__ CoverSet c, const __grid_constant__ ObjParams o,
                   const __grid_constant__ MadsArgs a, unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (c.ctl[2]) return; // the same word for every thread: the whole grid returns
    const int N = o.N, n = 3 * N, warp = threadIdx.x >> 5;
    unsigned char *rbase = smem_raw + mads_state_bytes(n);
    const RegionDesc r{c.x_lo, c.y_lo, c.x_hi, c.y_hi, 0, 0, c.discs, c.arcs};
    const RegionView v = cover_stage(r, c.pitch, c.ctl[0], min(c.ctl[1], kRegionMaxArcs), rbase);
    unsigned char *wbase = rbase + region_smem_bytes(c.pitch, kRegionMaxArcs) + (size_t)warp * region_warp_bytes(N, c.pitch);
    double *stage = reinterpret_cast<double *>(wbase);
    double *ia = reinterpret_cast<double *>(wbase + round_up(3 * N * 8, 16)), *ib = ia + region_list_cap(N, c.pitch);
    __syncthreads();
    mads_solves(a, n, smem_raw, stage, counter, [&](unsigned long long k) { return a.seed + k; },
                [&](const double *p) { // region_objective with the extreme barrier, as region_solve_kernel
        const CandScalars cs = candidate_prologue<false>(GridDesc{}, o, p, nullptr, false);
        if (!cs.feasible) return __longlong_as_double(0x7ff0000000000000ll);
        const double obj = objective_from_area(region_area(v, p, N, ia, ib), cs.violation, o);
        return (obj == obj) ? obj : __longlong_as_double(0x7ff0000000000000ll);
    });
}

cudaError_t launch_cover_mads(const CoverSet &c, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                              unsigned long long *counter, cudaStream_t stream)
{
    if (a.S <= 0) return cudaSuccess;
    int warps = 0, smem = 0;
    if (o.N > kRegionMaxUavs ||
        !region_plan(o.N, c.pitch, kRegionMaxArcs, mads_state_bytes(3 * o.N), cfg.max_smem_optin - 1024 /* the kernel's static shared memory */, &warps, &smem))
        return cudaErrorInvalidConfiguration;
    int grid = 0;
    cudaError_t err = persistent_grid(cover_solve_kernel, warps * 32, smem, a.S, cfg, &grid);
    if (err != cudaSuccess) return err;
    cover_solve_kernel<<<grid, warps * 32, smem, stream>>>(c, o, a, counter);
    return cudaGetLastError();
}

// ---- the horizons on a list-order store (launch_list_mads, launch_list_eval) ----
// Scenario e's list at timestep w.t (ListWalk): the base list, then its schedule's entries up to the timestep, each
// live iff no removal since its append reached its cell.  The walk skips dead entries, so the sum is the one over the
// compacted list the single calls keep, in the same order.
struct HorizonList {
    const ListWalk &w;
    const int *stamp;
    long long q0, n;
    __device__ __forceinline__ HorizonList(const ListWalk &w_, long long e)
        : w(w_), stamp(w_.stamps + e * w_.ncell), q0(0), n(w_.n_base)
    {
        if (w.off) {
            const long long l = w.list_of ? w.list_of[e] : 0;
            q0 = w.off[l * w.T];
            n += w.off[l * w.T + w.t] - q0;
        }
    }
    __device__ __forceinline__ long long size() const { return n; }
    __device__ __forceinline__ bool get(long long p, int &cell, int &k) const
    {
        if (p < w.n_base) {
            cell = w.base_cell[p];
            k = w.base_cls[p] & (kMaxClasses - 1);
            return stamp[cell] < 1;
        }
        const long long q = q0 + (p - w.n_base);
        cell = w.cell[q];
        k = w.cls[q] & (kMaxClasses - 1);
        return stamp[cell] < w.ta[q];
    }
};

__host__ __device__ inline int list_warp_bytes(int N) { return round_up(3 * N * 8, 16) + round_up(N * 8, 16); }

// mads_eval's list-order branch over scenario e's list: the same FP64 operations in the same order.  Ts: the warp's N
// thresholds; poff: the parameter block's offset.
__device__ __forceinline__ double list_eval(const GridDesc &g, const ObjParams &o, const double *stage, double *Ts,
                                            const HorizonList &list, long long poff, bool barrier)
{
    const int N = o.N;
    const uint32_t lane = lane_id();
    const CandScalars cs = candidate_prologue<false>(g, o, stage, nullptr, false, poff);
    if (barrier && !cs.feasible) return __longlong_as_double(0x7ff0000000000000ll);
    for (int c = lane; c < N; c += 32) Ts[c] = threshold(stage[2 * N + c]);
    __syncwarp();
    long long cls[kMaxClasses];
    const double area = ordered_area(g, N, stage, Ts, cls, list);
    __syncwarp();
    const double obj = __dadd_rn(-area, __dmul_rn(cs.violation, o.penalty_scale));
    return (obj == obj || !barrier) ? obj : __longlong_as_double(0x7ff0000000000000ll);
}

// The solves of E scenarios (launch_list_mads): solve k of scenario k / S, keyed as in scenario_solve_kernel.  Shared
// memory: [solve state] [W x (stage, thresholds)], no framebuffer and no planes.
__global__ void __launch_bounds__(kMadsThreads, kMadsCtas)
list_solve_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
                  const __grid_constant__ MadsArgs a, const __grid_constant__ ListWalk w, long long S,
                  unsigned long long key_stride, unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const int N = o.N, n = 3 * N;
    unsigned char *wbase = smem_raw + mads_state_bytes(n) + (size_t)warp * list_warp_bytes(N);
    double *stage = reinterpret_cast<double *>(wbase);
    double *Ts = reinterpret_cast<double *>(wbase + round_up(3 * N * 8, 16));
    long long e = 0; // the scenario of the current solve
    mads_solves(
        a, n, smem_raw, stage, counter,
        [&](unsigned long long k) {
            e = (long long)(k / (unsigned long long)S);
            return a.seed + (unsigned long long)e * key_stride + (k - (unsigned long long)e * S);
        },
        [&](const double *p) { return list_eval(g, o, p, Ts, HorizonList(w, e), e * 5 * N, true); });
}

// AreaMaxObjective of E swarms on their lists, one warp per swarm (launch_list_eval).
__global__ void __launch_bounds__(kMadsThreads)
list_eval_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
                 const __grid_constant__ ListWalk w, const double *__restrict__ X, long long E,
                 double *__restrict__ obj)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int W = blockDim.x >> 5, warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N, n = 3 * N;
    const long long e = (long long)blockIdx.x * W + warp;
    if (e >= E) return;
    unsigned char *wbase = smem_raw + (size_t)warp * list_warp_bytes(N);
    double *stage = reinterpret_cast<double *>(wbase);
    double *Ts = reinterpret_cast<double *>(wbase + round_up(3 * N * 8, 16));
    for (int i = lane; i < n; i += 32) stage[i] = X[e * n + i];
    __syncwarp();
    const double f = list_eval(g, o, stage, Ts, HorizonList(w, e), e * 5 * N, false);
    if (lane == 0) obj[e] = f;
}

cudaError_t launch_list_mads(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                             long long S, unsigned long long key_stride, const ListWalk &w,
                             unsigned long long *counter, cudaStream_t stream)
{
    if (a.S <= 0) return cudaSuccess;
    if (o.N < 1 || o.N > kMadsMaxUavs) return cudaErrorInvalidConfiguration;
    const int warps = kMadsThreads / 32, smem = mads_state_bytes(3 * o.N) + warps * list_warp_bytes(o.N);
    int grid = 0;
    cudaError_t err = persistent_grid(list_solve_kernel, kMadsThreads, smem, a.S, cfg, &grid);
    if (err != cudaSuccess) return err;
    list_solve_kernel<<<grid, kMadsThreads, smem, stream>>>(g, o, a, w, S, key_stride, counter);
    return cudaGetLastError();
}

cudaError_t launch_list_eval(const GridDesc &g, const ObjParams &o, const ListWalk &w, const double *X, long long E,
                             double *obj, cudaStream_t stream)
{
    if (E <= 0) return cudaSuccess;
    const int warps = kMadsThreads / 32, smem = warps * list_warp_bytes(o.N);
    list_eval_kernel<<<(unsigned)((E + warps - 1) / warps), kMadsThreads, smem, stream>>>(g, o, w, X, E, obj);
    return cudaGetLastError();
}

} // namespace cov
