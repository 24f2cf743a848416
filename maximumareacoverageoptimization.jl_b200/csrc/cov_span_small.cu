// cov_span_small.cu -- the small-swarm span kernel of libcoverage_cuda (sm_100a): N <= 8 UAVs and a
// grid whose union framebuffer fits a warp's share of shared memory (the reference's own
// configurations: N = 5 on 100 x 100, and BASELINE's 5 x 1M on 256 x 256).
//
// Same result as the general span kernel (cov_span_cta.cu) -- the count of list entries inside the
// union of the discs, src/AreaCoverageCalculation.jl:63-110 of /root/reference, plus the objective
// and constraint outputs -- organised for short candidates.  Persistent CTAs (one per SM, 15-16
// warps); the fire planes (TMA bulk copy) and the closure parameters sit in shared memory; every
// warp works on UNITS of CHUNK candidates taken from an atomic dispenser one unit ahead (the next
// unit's candidates are prefetched into L2 meanwhile):
//   phase 1  the unit's candidates are staged in shared memory (in the idle framebuffer region) and
//            lane k owns candidate k: it forms the penalty sums and constraint verdicts serially in
//            FP64 (the reference's own order), flags the discs whose bounding boxes touch another
//            disc, and writes one 32-byte record per disc plus the prefix sums of the discs' row
//            counts.  CHUNK candidates are set up at once instead of one candidate on N of 32 lanes.
//   phase 2  per candidate, the (disc, row) pairs are FLATTENED over the lanes, two per lane and
//            pass (one for the last short stretch).  A lane computes the covered columns [lo, hi] of
//            its row in FP32, in coordinates relative to the disc's nearest cell (so the FP32 error
//            is ~2^-23 R instead of ~2^-21 * 500 m), certifies both ends against an error band, and
//            falls back to the exact FP64 walk only when the band cannot decide.  A disc that touches
//            no other disc is counted directly (popcount of span & fire words); the others OR their
//            spans into the warp's shared-memory framebuffer with atomicOr and count the bits they
//            were first to set: a union count, whatever the order.
//   phase 3  lane k assembles candidate k's objective; CHUNK results leave as coalesced stores.
// CHUNK in {32, 16, 8, 4} is chosen per launch (launch_span_small) so that batches too small to give
// every warp several 32-candidate units still fill the machine.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <type_traits>
#include "cov_device.cuh"
#include "cov_kernel_common.cuh"
#include "cov_span_common.cuh"
#include "cov_kernels.cuh"
#include "../../include/coverage_cuda.h"

namespace cov {

constexpr int kSmallMaxN = 8;

// The framebuffer region doubles as the staging area of a unit's candidates during phase 1 (it is
// all-zero between candidates and idle until phase 2), so it is at least chunk * 24 N bytes.
__host__ __device__ inline int small_fb_bytes(const GridDesc &g, int N, int chunk)
{
    const int fb = round_up(g.ny * (fb_can_swizzle(g) ? g.wpr : g.stride) * 4, 16), stage = round_up(chunk * 3 * N * 8, 16);
    return fb > stage ? fb : stage;
}
__host__ __device__ inline int small_warp_bytes(const GridDesc &g, int N, int chunk)
{
    const int dp = chunk * N * 32;
    const int pre = chunk * 16; // 8 x u16 item prefixes per candidate
    const int clr = chunk * 4;  // first | last row << 16 of the discs that go through the framebuffer
    return small_fb_bytes(g, N, chunk) + dp + pre + clr;
}
__host__ __device__ inline int small_param_bytes(int N) { return round_up(5 * N * 8, 16); }

// MAXW: the most warps a CTA of this instantiation may have (20: <= 102 registers per thread, no spills;
// 24: <= 85, a few spilled bytes -- worth it when the per-warp shared memory is small enough for 24 warps)
// FEW: N <= 5 -- the disc index of an item needs 4 prefixes at most, half of the packed compare
template <bool MULTI, int CHUNK, int MAXW, bool FEW>
__global__ void __launch_bounds__(MAXW * 32, 1)
span_small_kernel(const __grid_constant__ GridDesc g, const __grid_constant__ ObjParams o,
                  const double *__restrict__ X, long long B, EvalOut out, unsigned long long *counter,
                  int force_exact)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const int N = o.N;
    const int planes_bytes = g.n_planes * g.plane_words * 4;
    const int param_bytes = small_param_bytes(N);
    const int warp_bytes = small_warp_bytes(g, N, CHUNK);
    const int fb_bytes = small_fb_bytes(g, N, CHUNK);
    uint32_t *planes_s = reinterpret_cast<uint32_t *>(smem_raw);
    double *par = reinterpret_cast<double *>(smem_raw + planes_bytes); // r_max, prev_x, prev_y, prev_z, cons3_G
    unsigned char *wbase = smem_raw + planes_bytes + param_bytes + (size_t)warp * warp_bytes;
    uint32_t *fb = reinterpret_cast<uint32_t *>(wbase);
    const double *stage = reinterpret_cast<const double *>(wbase);
    SDisc *dp = reinterpret_cast<SDisc *>(wbase + fb_bytes);
    uint4 *prefix = reinterpret_cast<uint4 *>(wbase + fb_bytes + CHUNK * N * 32);
    uint32_t *clear_rows = reinterpret_cast<uint32_t *>(wbase + fb_bytes + CHUNK * N * 32 + CHUNK * 16);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + planes_bytes + param_bytes + (size_t)warps * warp_bytes);

    // the closure parameters once per CTA (with the shared-memory carve-out at its maximum there is next
    // to no L1 left: every repeated global read would be an L2 round trip)
    for (int t2 = threadIdx.x; t2 < N; t2 += blockDim.x) {
        par[t2] = o.r_max[t2];
        par[N + t2] = o.use_cons3 ? o.prev_x[t2] : 0.0;
        par[2 * N + t2] = o.use_cons3 ? o.prev_y[t2] : 0.0;
        par[3 * N + t2] = o.use_cons3 ? o.prev_z[t2] : 0.0;
        par[4 * N + t2] = o.use_cons3 ? o.cons3_G[t2] : 0.0;
    }
    stage_planes(g, planes_s, bar, planes_bytes); // TMA bulk copy of the fire planes, once per CTA (syncs)
    for (int t2 = lane; t2 < fb_bytes / 16; t2 += 32) reinterpret_cast<uint4 *>(fb)[t2] = make_uint4(0, 0, 0, 0);
    __syncwarp();

    FbLayout fl;
    fl.swz = fb_can_swizzle(g) ? 7 : 0;
    fl.stride = fl.swz ? g.wpr : g.stride;
    const long long n_chunks = (B + CHUNK - 1) / CHUNK;
    const int cstride = 3 * N;

    // units: the first one of a warp is static (warp w of CTA c takes unit c + gridDim.x * w, so a batch of
    // fewer units than warps spreads over all SMs and nobody holds two while another has none); further
    // units come from the global dispenser and are taken one ahead: while unit u is processed the
    // candidates of unit u+1 are already on their way into L2
    const unsigned long long total_warps = (unsigned long long)gridDim.x * (unsigned long long)warps;
    const bool dynamic_units = (unsigned long long)n_chunks > total_warps; // uniform over the grid
    unsigned long long next = (unsigned long long)blockIdx.x + (unsigned long long)gridDim.x * (unsigned long long)warp;
    const bool x_aligned = (reinterpret_cast<unsigned long long>(X) & 15ull) == 0;
    for (;;) {
        const unsigned long long chunk = next;
        if ((long long)chunk >= n_chunks) break;
        next = (unsigned long long)n_chunks;
        if (dynamic_units) {
            if (lane == 0) next = total_warps + atomicAdd(counter, 1ull);
            next = __shfl_sync(0xffffffffu, next, 0);
        }
        const long long base = (long long)chunk * CHUNK;
        const int in_chunk = (int)min((long long)CHUNK, B - base);
        if ((long long)next < n_chunks) {
            const char *nx_ptr = reinterpret_cast<const char *>(X + next * CHUNK * cstride);
            const int nbytes = (int)min((long long)CHUNK, B - (long long)next * CHUNK) * cstride * 8;
            for (int off = lane * 128; off < nbytes; off += 32 * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(nx_ptr + off));
        }
        // stage the unit's candidates (contiguous in_chunk * 24 N bytes) in the framebuffer region
        {
            const int ndbl = in_chunk * cstride;
            const double *src = X + base * cstride;
            double *dst = reinterpret_cast<double *>(fb);
            if (x_aligned && (ndbl & 1) == 0 && ((base * cstride) & 1) == 0) {
                for (int t2 = lane; t2 < ndbl / 2; t2 += 32)
                    reinterpret_cast<double2 *>(dst)[t2] = __ldg(reinterpret_cast<const double2 *>(src) + t2);
            } else {
                for (int t2 = lane; t2 < ndbl; t2 += 32) dst[t2] = __ldg(src + t2);
            }
        }
        __syncwarp();

        // ---------------- phase 1: lane k sets up candidate k ----------------
        // With CHUNK < 32 the other lanes help: lane = cand + CHUNK * part, and the parts share out the discs
        // (the heavy per-disc record, thresholds included) and the rows of the pair loop; the order-dependent
        // FP64 sums stay on part 0, the lane that also assembles the candidate in phase 3.
        constexpr int kParts = 32 / CHUNK;
        const int cand = (int)lane & (CHUNK - 1), part = (int)lane / CHUNK;
        double my_viol = 0.0, my_prog = 0.0;
        int my_feas = 1;
        {
            // Rolled loops over the discs (operands re-read from shared memory): phase 1 runs once per CHUNK
            // candidates, so compact code matters more here than a few extra loads.
            const bool live = cand < in_chunk;
            const double *xr = stage + (live ? cand : 0) * cstride; // shared memory
            const double *yr = xr + N, *rr = xr + 2 * N;
            bool bad = false;
            if (live && part == 0) {
                // penalty: sequential FP64 sum in index order (src/TDM_STATIC_opt.jl:89-93)
#pragma unroll 1
                for (int i = 0; i < N; ++i) {
                    const double diff = __dsub_rn(rr[i], par[i]);
                    my_viol = __dadd_rn(my_viol, fabs(diff));
                    if (out.progressive && prog_takes(o, i)) my_prog = __dadd_rn(my_prog, julia_max0(diff));
                }
                if (o.use_cons3) {
#pragma unroll 1
                    for (int i = 0; i < N; ++i) {
                        const double ax = __dsub_rn(par[N + i], xr[i]);
                        const double ay = __dsub_rn(par[2 * N + i], yr[i]);
                        const double az = __dsub_rn(par[3 * N + i], __ddiv_rn(rr[i], o.tan_half_fov));
                        const double s = __dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az));
                        bad |= (s >= par[4 * N + i]);
                    }
                }
                if (o.use_cons7) {
#pragma unroll 1
                    for (int i = 0; i < N; ++i) bad |= (yr[i] < 200.0) && (rr[i] > o.cons7_R);
                }
            }
            // pairs: cons8 (src/TDM_Constraints.jl:157-172; unordered pairs decide the ordered loop) and the
            // discs that may share cells with another disc of the candidate (bounding boxes, two cells of
            // margin; NaN compares false -> "may share"); first discs a = part, part + kParts, ...
            uint32_t shared_mask = 0;
            if (live) {
#pragma unroll 1
                for (int a = part; a < N - 1; a += kParts) {
                    const double xa = xr[a], ya = yr[a], ra = rr[a];
#pragma unroll 1
                    for (int b2 = a + 1; b2 < N; ++b2) {
                        const double ax = __dsub_rn(xa, xr[b2]), ay = __dsub_rn(ya, yr[b2]);
                        if (o.use_cons8) bad |= (__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)) < o.sep_T);
                        const double sr = ra + rr[b2];
                        const bool apart = (fabs(ax) >= sr + 2.0 * g.dx) || (fabs(ay) >= sr + 2.0 * g.dy);
                        if (!apart) shared_mask |= (1u << a) | (1u << b2);
                    }
                }
                // the per-disc records, without the fields that need the whole candidate (patched below)
#pragma unroll 1
                for (int c = part; c < N; c += kParts) {
                    SDisc d;
                    make_sdisc(g, xr[c], yr[c], rr[c], d);
                    dp[cand * N + c] = d;
                }
            }
            uint32_t bad_bits = bad ? 1u : 0u;
#pragma unroll
            for (int off = CHUNK; off < 32; off <<= 1) { // combine the parts of a candidate
                shared_mask |= __shfl_xor_sync(0xffffffffu, shared_mask, off);
                bad_bits |= __shfl_xor_sync(0xffffffffu, bad_bits, off);
            }
            my_feas = !bad_bits;
            __syncwarp(); // dp[] of the other parts
            if (live && part == 0) {
                uint32_t run = 0;
                int rmin = 0xffff, rmax = 0; // rows of the discs that paint the framebuffer (what phase 2 clears)
                // 8 x u16 inclusive prefixes; unused slots 0x7fff (above every item index, and small enough for the
                // packed compare of phase 2)
                unsigned long long plo = 0x7fff7fff7fff7fffull, phi = 0x7fff7fff7fff7fffull;
#pragma unroll 1
                for (int c = 0; c < N; ++c) {
                    SDisc *q = dp + cand * N + c;
                    const uint32_t rws = q->rows;
                    const int r0 = (int)(rws & 0xffffu), r1 = (int)(rws >> 16);
                    const int rows = r1 - r0 + 1 > 0 ? r1 - r0 + 1 : 0;
                    if (((shared_mask >> c) & 1u) && rows > 0) {
                        rmin = min(rmin, r0);
                        rmax = max(rmax, r1);
                    }
                    // bit 1: may share cells; bits 16..31: (first row) - (items before this disc) + 32768, so that
                    // item t is row base + t
                    q->flags |= (((shared_mask >> c) & 1u) << 1) | ((uint32_t)(r0 - (int)run + 32768) << 16);
                    run += (uint32_t)rows;
                    const unsigned long long v = run; // ny <= 4095 and N <= 8 keep it below 0x8000
                    const int sh = (c & 3) * 16;
                    if (c < 4) plo = (plo & ~(0xffffull << sh)) | (v << sh);
                    else phi = (phi & ~(0xffffull << sh)) | (v << sh);
                }
                // slot 7 is never compared against (a disc index needs N - 1 <= 7 prefixes): it carries the total
                // (N == 8: slot 7 is the last inclusive prefix, which is the total as well); bit 15 of the slot,
                // free because totals stay below 0x8000: some disc of the candidate goes through the framebuffer
                phi = (phi & 0x0000ffffffffffffull) | ((unsigned long long)(run | (shared_mask ? 0x8000u : 0u)) << 48);
                prefix[cand] = make_uint4((uint32_t)plo, (uint32_t)(plo >> 32), (uint32_t)phi, (uint32_t)(phi >> 32));
                clear_rows[cand] = (uint32_t)rmin | ((uint32_t)rmax << 16);
            }
        }
        __syncwarp();
        // the staging bytes go back to all-zero framebuffer
        for (int t2 = lane; t2 < (in_chunk * cstride * 8 + 15) / 16; t2 += 32)
            reinterpret_cast<uint4 *>(fb)[t2] = make_uint4(0, 0, 0, 0);
        __syncwarp();

        // ---------------- phase 2: one candidate at a time, (disc, row) items over the lanes ----------------
        long long my_cnt = 0;
        long long my_cls[kMaxClasses];
#pragma unroll
        for (int k = 0; k < kMaxClasses; ++k) my_cls[k] = 0;

        for (int kc = 0; kc < in_chunk; ++kc) {
            const uint4 pq = prefix[kc];
            const uint32_t total = (pq.w >> 16) & 0x7fffu; // number of items (slot 7, see phase 1)
            const bool any_shared = (pq.w >> 31) != 0;
            const SDisc *cdp = dp + kc * N;
            uint32_t cnt[MULTI ? kMaxClasses : 1];
#pragma unroll
            for (int k = 0; k < (MULTI ? kMaxClasses : 1); ++k) cnt[k] = 0;

            {
                // K items per lane in one pass over 32 K consecutive items: independent instruction streams hide
                // the FP32 and shared-memory latencies
                auto pass = [&](auto K_, const uint32_t tb) {
                    constexpr int kItems = decltype(K_)::value;
                    bool has[kItems];
                    int c[kItems], j[kItems], lo[kItems], hi[kItems], st[kItems];
                    uint32_t tt[kItems];
                    SDisc d[kItems];
#pragma unroll
                    for (int k = 0; k < kItems; ++k) {
                        const uint32_t t = tb + 32 * k + lane;
                        has[k] = t < total;
                        tt[k] = has[k] ? t : tb; // an idle slot shadows item tb, result discarded
                        // disc index = number of inclusive prefixes <= t among slots 0..6, all seven compared at
                        // once: every 16-bit field of (0x8000 | t) - prefix stays within its field (both sides
                        // are below 0x8000) and keeps bit 15 exactly when t >= prefix.  Slot 7 (total | flag) may
                        // borrow out of the top of its word, which harms nothing, and is masked out.
                        const uint32_t rep = tt[k] * 0x10001u + 0x80008000u;
                        const uint32_t x0 = rep - pq.x, x1 = rep - pq.y;
                        uint32_t hits = (x0 & 0x80008000u) | ((x1 & 0x80008000u) >> 1);
                        if (!FEW) {
                            const uint32_t x2 = rep - pq.z, x3 = rep - pq.w;
                            hits |= ((x2 & 0x80008000u) >> 2) | ((x3 & 0x00008000u) >> 3);
                        }
                        c[k] = __popc(hits);
                    }
#pragma unroll
                    for (int k = 0; k < kItems; ++k) {
                        COV_ASSERT(c[k] < N);
                        d[k] = cdp[c[k]];
                        j[k] = (int)(d[k].flags >> 16) - 32768 + (int)tt[k];
                        COV_ASSERT(j[k] >= 1 && j[k] <= (int)(d[k].rows >> 16) && j[k] <= g.ny);
                    }
#pragma unroll
                    for (int k = 0; k < kItems; ++k) {
                        st[k] = fast_span(g, d[k], j[k], force_exact, lo[k], hi[k]);
                        if (!has[k]) st[k] = kEmpty;
                    }
#pragma unroll
                    for (int k = 0; k < kItems; ++k)
                        if (st[k] == kSlow) {
                            int l2 = lo[k], h2 = hi[k]; // temporaries: the arrays stay in registers
                            // (the candidate's doubles are only needed here: no address arithmetic per candidate)
                            slow_item_of(g, X, base, kc, N, c[k], j[k], (d[k].flags & 1u) || force_exact, l2, h2);
                            if (l2 <= h2) st[k] = kSpan;
                            else { st[k] = kEmpty; l2 = h2 = 1; }
                            lo[k] = l2;
                            hi[k] = h2;
                        }
#pragma unroll
                    for (int k = 0; k < kItems; ++k) {
                        const bool sh = (d[k].flags & 2u) != 0;
                        paint_span<MULTI>(g, fb, planes_s, j[k], lo[k], hi[k], st[k] == kSpan, sh, cnt, 1, fl);
                    }
                };
                // two items per lane while more than 32 remain, one for the last short stretch (the trip
                // count is warp-uniform)
#pragma unroll 1
                for (uint32_t tb = 0; tb < total;) {
                    if (total - tb > 32u) {
                        pass(std::integral_constant<int, 2>{}, tb);
                        tb += 64;
                    } else {
                        pass(std::integral_constant<int, 1>{}, tb);
                        tb += 32;
                    }
                }
                // clear what the shared discs painted
                if (any_shared) { // warp-uniform
                    __syncwarp();
                    if (fl.stride <= 16) {
                        // narrow grids: whole rows from the first to the last row of any shared disc -- one contiguous
                        // stretch of the framebuffer (the swizzle permutes words within a row only), 128-bit stores
                        // when rows are 16-byte multiples
                        const uint32_t cr = clear_rows[kc]; // set up in phase 1
                        const int rmin = (int)(cr & 0xffffu), rmax = (int)(cr >> 16);
                        if (rmax >= rmin) {
                            const int w0 = (rmin - 1) * fl.stride, w1 = rmax * fl.stride; // words [w0, w1)
                            if ((fl.stride & 3) == 0) {
                                for (int t = (w0 >> 2) + (int)lane; t < (w1 >> 2); t += 32)
                                    reinterpret_cast<uint4 *>(fb)[t] = make_uint4(0, 0, 0, 0);
                            } else {
                                for (int t = w0 + (int)lane; t < w1; t += 32) fb[t] = 0u;
                            }
                        }
                    } else {
                        // wide grids: every word of the shared discs' bounding boxes
#pragma unroll 1
                        for (int c = 0; c < N; ++c) {
                            const SDisc d = cdp[c];
                            if (!(d.flags & 2u)) continue;
                            const int r0 = d.rows & 0xffffu, r1 = d.rows >> 16;
                            int wa = 0, wb = g.wpr - 1;
                            if (!(d.flags & 1u)) {
                                // columns within sqrt(Tf + delta) of the centre, one cell of margin
                                const float hw = ceilf(sqrtf(d.Tf + d.delta) * g.inv_dxf) + 2.0f;
                                const float nxf = int_to_float_small(g.nx);
                                const int ca = (int)fminf(fmaxf(d.icf - hw, 1.0f), nxf);
                                const int cb = (int)fminf(fmaxf(d.icf + hw, 1.0f), nxf);
                                wa = (ca - 1) >> 5;
                                wb = (cb - 1) >> 5;
                            }
                            for (int j = r0 + (int)lane; j <= r1; j += 32) {
                                for (int w = wa; w <= wb; ++w) fb[fl.at(j - 1, w)] = 0u;
                            }
                        }
                    }
                }
            }
            __syncwarp();

            long long total_cnt = 0;
#pragma unroll
            for (int k = 0; k < (MULTI ? kMaxClasses : 1); ++k) {
                const long long v = (long long)__reduce_add_sync(0xffffffffu, cnt[k]);
                total_cnt += v;
                if ((int)lane == kc) my_cls[k] = v;
            }
            if ((int)lane == kc) my_cnt = total_cnt;
        }

        // ---------------- phase 3: lane k finishes candidate k; coalesced stores ----------------
        if ((int)lane < in_chunk) {
            const long long bidx = base + lane;
            const double my_obj = assemble_objective(g, o, my_cls, my_viol);
            out.obj[bidx] = my_obj;
            store_mirrors(out, bidx, my_obj, my_feas);
            if (out.count) out.count[bidx] = my_cnt;
            if (out.feasible) out.feasible[bidx] = (unsigned char)my_feas;
            if (out.progressive) out.progressive[bidx] = my_prog;
            if (out.class_count)
                for (int k = 0; k < g.n_classes; ++k) out.class_count[bidx * g.n_classes + k] = my_cls[k];
        }
        __syncwarp(); // dp / prefix are rewritten by the next chunk
    }
}

// ------------------------------------------------------------------------------------------
// launcher: returns false when this kernel does not apply (the general span kernel takes over)
// ------------------------------------------------------------------------------------------
template <typename K>
static cudaError_t set_smem_small(K kernel, int bytes)
{
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

// B: batch size (0: unknown / large).  A unit of work is CHUNK candidates processed by one warp, one
// after the other, so a batch with fewer units than resident warps would leave the machine idle and
// stretch the kernel to the latency of one unit: smaller batches take smaller chunks, and tiny ones
// (a MADS poll set) go to the CTA-per-candidate kernel.
bool span_small_applies(const GridDesc &g, int N, const LaunchCfg &cfg, long long B, int *warps_out, int *chunk_out)
{
    if (N > kSmallMaxN || g.stride > 255 || g.ny > 4095) return false; // 8 x ny items fit 15 bits (row base in 16)
    if (B > 0 && B < 128) return false;
    const int planes_bytes = g.n_planes * g.plane_words * 4;
    int best_w = 0, best_chunk = 0;
    for (int chunk : {32, 16}) {
        const int per = small_warp_bytes(g, N, chunk);
        int w = (cfg.max_smem_optin - planes_bytes - small_param_bytes(N) - 16) / per;
        // the 24-warp instantiation (launch_small_variant picks 20 or 24 by this count) -- except 32-candidate
        // units of 6 to 8 UAVs: >= 11 392 bytes per warp, so 21 warps would take more than the 227 KB a CTA can
        // have on sm_100, and that instantiation is not built
        w = std::min(w, (chunk == 32 && N > 5) ? 20 : 24);
        if (cfg.warps_per_cta > 0) w = std::min(w, cfg.warps_per_cta);
        // prefer the 32-candidate chunk unless the 16-candidate one buys >= 25 % more warps
        if (w >= 4 && (best_w == 0 || w * 4 >= best_w * 5)) {
            best_w = w;
            best_chunk = chunk;
        }
    }
    if (best_w < 4) return false;
    if (B > 0) {
        // cost model (measured on B200): a unit costs ~2.65 us per candidate plus ~2.5 us of setup, and the
        // kernel lasts as long as the busiest warp: pick the chunk that minimises ceil(units / warps) * unit
        const double W = (double)best_w * cfg.num_sms;
        double best_t = 0;
        int pick = best_chunk;
        for (int c = best_chunk; c >= 4; c /= 2) {
            const double rounds = ceil((double)((B + c - 1) / c) / W);
            const double tcost = rounds * (2.65 * c + 2.5);
            if (c == best_chunk || tcost < best_t * 0.97) {
                best_t = tcost;
                pick = c;
            }
        }
        best_chunk = pick;
    }
    if (warps_out) *warps_out = best_w;
    if (chunk_out) *chunk_out = best_chunk;
    return true;
}

template <bool M, int C, int MAXW, bool FEW>
static cudaError_t launch_small_variant(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                                        long long B, const EvalOut &out, unsigned long long *counter,
                                        cudaStream_t stream, int grid, int warps, int smem)
{
    // the attribute is per function and per device: raise it only when it has to grow
    static int configured_smem[64] = {0};
    int dev = 0;
    (void)cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || smem > configured_smem[dev]) {
        cudaError_t err = cudaFuncSetAttribute(span_small_kernel<M, C, MAXW, FEW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (err != cudaSuccess) return err;
        if (dev >= 0 && dev < 64) configured_smem[dev] = smem;
    }
    span_small_kernel<M, C, MAXW, FEW><<<grid, warps * 32, smem, stream>>>(g, o, dX, B, out, counter, cfg.force_exact);
    return cudaGetLastError();
}

cudaError_t launch_span_small(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                              long long B, const EvalOut &out, unsigned long long *counter, cudaStream_t stream,
                              LaunchInfo *info)
{
    int warps = 0, chunk = 0;
    if (!span_small_applies(g, o.N, cfg, B, &warps, &chunk)) return cudaErrorInvalidConfiguration;
    const bool multi = !(g.n_planes == 1 && g.n_classes == 1 && g.plane_mult[0] == 1);
    const int smem = g.n_planes * g.plane_words * 4 + small_param_bytes(o.N) + warps * small_warp_bytes(g, o.N, chunk) + 16;
    const long long chunks = (B + chunk - 1) / chunk;
    // a batch of fewer units than warps is spread over all SMs with fewer warps each (they run faster alone)
    const int grid = (int)std::min<long long>(chunks, (long long)cfg.num_sms);
    warps = (int)std::min<long long>(warps, (chunks + grid - 1) / grid);
    if (info) {
        info->grid = grid;
        info->block = warps * 32;
        info->smem_bytes = smem;
        info->band_rows = g.ny;
        info->planes_in_smem = 1;
        info->kernel = COV_KERNEL_SPAN;
        info->multi = multi;
        info->chunk = chunk;
        info->max_warps = warps > 20 ? 24 : 20;
        info->plane_mode = -1;
    }
#define COV_SMALL_ARGS g, o, cfg, dX, B, out, counter, stream, grid, warps, smem
#define COV_SMALL_CASE(M, C)                                                                                     \
    case C:                                                                                                      \
        if (o.N <= 5)                                                                                            \
            return warps > 20 ? launch_small_variant<M, C, 24, true>(COV_SMALL_ARGS)                             \
                              : launch_small_variant<M, C, 20, true>(COV_SMALL_ARGS);                            \
        return warps > 20 && C != 32 ? launch_small_variant<M, C, C == 32 ? 20 : 24, false>(COV_SMALL_ARGS)      \
                                     : launch_small_variant<M, C, 20, false>(COV_SMALL_ARGS)
    if (multi) {
        switch (chunk) {
            COV_SMALL_CASE(true, 32);
            COV_SMALL_CASE(true, 16);
            COV_SMALL_CASE(true, 8);
            COV_SMALL_CASE(true, 4);
        }
    } else {
        switch (chunk) {
            COV_SMALL_CASE(false, 32);
            COV_SMALL_CASE(false, 16);
            COV_SMALL_CASE(false, 8);
            COV_SMALL_CASE(false, 4);
        }
    }
#undef COV_SMALL_CASE
#undef COV_SMALL_ARGS
    return cudaErrorInvalidConfiguration;
}

} // namespace cov
