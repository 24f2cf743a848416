// cov_grid_kernels.cu -- device-side cell store of libcoverage_cuda and the small utility kernels
// around the objective (all citations relative to /root/reference/):
//   cell store         CellFunctions.Cells.points_of_interest        src/CellFunctions.jl:5-16
//   fill_full          createPOI                                      src/AreaCoverageCalculation.jl:11-21
//   add_points         update_POI's push!                             src/CellFunctions.jl:59-79
//   remove_covered     rmvCoveredPOI                                  src/CellFunctions.jl:81-108
// The canonical store is one multiplicity byte and one class byte per cell; the bit planes the
// objective kernels sweep are derived from it by pack_planes.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "cov_device.cuh"
#include "cov_kernels.cuh"

namespace cov {

__global__ void grid_stats_kernel(const unsigned char *__restrict__ mult, const unsigned char *__restrict__ cls,
                                  long long ncell, unsigned long long *stats)
{
    unsigned long long entries = 0, cells = 0;
    unsigned int orm[kMaxClasses] = {0, 0, 0, 0};
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
         t += (long long)gridDim.x * blockDim.x) {
        const unsigned m = mult[t];
        if (m) {
            entries += m;
            cells += 1;
            const int k = cls[t] & (kMaxClasses - 1);
#pragma unroll
            for (int q = 0; q < kMaxClasses; ++q) orm[q] |= (q == k) ? m : 0u;
        }
    }
    for (int off = 16; off; off >>= 1) {
        entries += __shfl_xor_sync(0xffffffffu, entries, off);
        cells += __shfl_xor_sync(0xffffffffu, cells, off);
#pragma unroll
        for (int q = 0; q < kMaxClasses; ++q) orm[q] |= __shfl_xor_sync(0xffffffffu, orm[q], off);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&stats[0], entries);
        atomicAdd(&stats[1], cells);
#pragma unroll
        for (int q = 0; q < kMaxClasses; ++q)
            if (orm[q]) atomicOr(&stats[2 + q], (unsigned long long)orm[q]);
    }
}

cudaError_t launch_grid_stats(const unsigned char *mult, const unsigned char *cls, long long ncell,
                              unsigned long long *stats, cudaStream_t s)
{
    cudaError_t e = cudaMemsetAsync(stats, 0, (2 + kMaxClasses) * sizeof(unsigned long long), s);
    if (e != cudaSuccess) return e;
    const int block = 256;
    const int grid = (int)std::min<long long>((ncell + block - 1) / block, 148 * 8);
    grid_stats_kernel<<<max(grid, 1), block, 0, s>>>(mult, cls, ncell, stats);
    return cudaGetLastError();
}

// The grid of a launch over E stores side by side: blockIdx.y strides over the stores, and the blocks of one store
// shrink so that the whole launch stays near `cap` blocks (E = 1: the single-store grid).
static dim3 store_grid(long long work, int block, int cap, long long E)
{
    const int gy = (int)std::min<long long>(E, 65535);
    const long long gx = std::min<long long>((work + block - 1) / block, std::max(cap / gy, 1));
    return dim3((unsigned)std::max<long long>(gx, 1), (unsigned)gy);
}

// one warp per (row, word): lane b reads cell i = 32w + b + 1 and the ballot is the plane word
__global__ void pack_planes_kernel(const unsigned char *__restrict__ mult, const unsigned char *__restrict__ cls,
                                   const __grid_constant__ GridDesc g, uint32_t *__restrict__ planes, long long E)
{
    const long long warp_global = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const long long n_words = (long long)g.ny * g.stride, ncell = (long long)g.nx * g.ny;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long e = blockIdx.y; e < E; e += gridDim.y) {
        const unsigned char *me = mult + e * ncell, *ce = cls + e * ncell;
        uint32_t *pe = planes + e * g.n_planes * (long long)g.plane_words;
        for (long long t = warp_global; t < n_words; t += n_warps) {
            const int row = (int)(t / g.stride), w = (int)(t % g.stride);
            const int i = 32 * w + lane; // 0-based column
            unsigned m = 0, k = 0;
            if (w < g.wpr && i < g.nx) {
                const long long cell = (long long)i + (long long)g.nx * row;
                m = me[cell];
                k = ce[cell];
            }
            for (int l = 0; l < g.n_planes; ++l) {
                const bool bit = (m & (unsigned)g.plane_mult[l]) && ((int)k == g.plane_class[l]);
                const uint32_t word = __ballot_sync(0xffffffffu, bit);
                if (lane == 0) pe[(size_t)l * g.plane_words + t] = word;
            }
        }
    }
}

cudaError_t launch_pack_planes(const unsigned char *mult, const unsigned char *cls, const GridDesc &g,
                               uint32_t *planes, cudaStream_t s, long long E)
{
    cudaError_t e = cudaMemsetAsync(planes, 0, (size_t)E * g.n_planes * g.plane_words * 4, s);
    if (e != cudaSuccess) return e;
    const long long n_words = (long long)g.ny * g.stride;
    pack_planes_kernel<<<store_grid(n_words * 32, 256, 148 * 16, E), 256, 0, s>>>(mult, cls, g, planes, E);
    return cudaGetLastError();
}

__global__ void requad_plane_kernel(const __grid_constant__ GridDesc g, uint32_t *__restrict__ q)
{
    const long long n = (long long)g.ny * g.qstride;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
        const int row = (int)(t / g.qstride), w = (int)(t % g.qstride);
        const int src = w ^ ((row >> 4) & 1); // row = j - 1; the swizzle is an involution within a word pair
        q[t] = src < g.wpr ? g.planes[(size_t)row * g.stride + src] : 0u;
    }
}
cudaError_t launch_requad_plane(const GridDesc &g, uint32_t *planes_q, cudaStream_t s)
{
    const long long n = (long long)g.ny * g.qstride;
    const int block = 256;
    const int grid = (int)std::min<long long>((n + block - 1) / block, 148 * 8);
    requad_plane_kernel<<<max(grid, 1), block, 0, s>>>(g, planes_q);
    return cudaGetLastError();
}

__global__ void fill_full_kernel(unsigned char *mult, unsigned char *cls, long long ncell)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
         t += (long long)gridDim.x * blockDim.x) {
        mult[t] = 1;
        cls[t] = 0;
    }
}
cudaError_t launch_fill_full(unsigned char *mult, unsigned char *cls, long long ncell, cudaStream_t s)
{
    const int block = 256;
    const int grid = (int)std::min<long long>((ncell + block - 1) / block, 148 * 8);
    fill_full_kernel<<<max(grid, 1), block, 0, s>>>(mult, cls, ncell);
    return cudaGetLastError();
}

__global__ void bits_to_cells_kernel(const uint32_t *__restrict__ bits, int nx, int ny, unsigned char *mult,
                                     unsigned char *cls)
{
    const int wpr = (nx + 31) / 32;
    const long long ncell = (long long)nx * ny;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
         t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t % nx), j = (int)(t / nx);
        const uint32_t w = bits[(size_t)j * wpr + (i >> 5)];
        const unsigned bit = (w >> (i & 31)) & 1u;
        mult[t] = (unsigned char)bit;
        cls[t] = bit ? 0 : 0xffu;
    }
}
cudaError_t launch_bits_to_cells(const uint32_t *bits, int nx, int ny, unsigned char *mult,
                                 unsigned char *cls, cudaStream_t s)
{
    const long long ncell = (long long)nx * ny;
    const int block = 256;
    const int grid = (int)std::min<long long>((ncell + block - 1) / block, 148 * 8);
    bits_to_cells_kernel<<<max(grid, 1), block, 0, s>>>(bits, nx, ny, mult, cls);
    return cudaGetLastError();
}

__global__ void thresholds_kernel(const double *xyR, int N, double *xyT, long long E)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    for (long long e = blockIdx.y; e < E && c < N; e += gridDim.y) {
        const double *in = xyR + e * 3 * N;
        double *out = xyT + e * 3 * N;
        out[c] = in[c];
        out[N + c] = in[N + c];
        out[2 * N + c] = threshold(in[2 * N + c]);
    }
}
cudaError_t launch_thresholds(const double *xyR, int N, double *xyT, cudaStream_t s, long long E)
{
    thresholds_kernel<<<dim3((N + 127) / 128, (unsigned)std::min<long long>(E, 65535)), 128, 0, s>>>(xyR, N, xyT, E);
    return cudaGetLastError();
}

// exact FP64 test of one cell against N discs (same predicate as calculateArea)
__device__ __forceinline__ bool cell_covered(const GridDesc &g, int i1, int j1, const double *xyT, int N)
{
    const double px = cell_centre(i1, g.dx, g.hdx);
    const double py = cell_centre(j1, g.dy, g.hdy);
    for (int c = 0; c < N; ++c)
        if (radicand(px, py, xyT[c], xyT[N + c]) < xyT[2 * N + c]) return true;
    return false;
}

// stamp (nullable): stamp[e * ncell + cell] = t for every cell of store e that loses entries (cov_run_horizon_points'
// last_removed)
__global__ void remove_covered_kernel(unsigned char *mult, unsigned char *cls, const __grid_constant__ GridDesc g,
                                      const double *__restrict__ xyT, int N, unsigned long long *removed, int *stamp,
                                      int t_stamp, long long E, long long removed_stride)
{
    const long long ncell = (long long)g.nx * g.ny;
    for (long long e = blockIdx.y; e < E; e += gridDim.y) {
        unsigned char *me = mult + e * ncell, *ce = cls + e * ncell;
        int *se = stamp ? stamp + e * ncell : nullptr;
        const double *xe = xyT + e * 3 * N;
        unsigned long long mine = 0;
        for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
             t += (long long)gridDim.x * blockDim.x) {
            const unsigned m = me[t];
            if (m) {
                const int i1 = (int)(t % g.nx) + 1, j1 = (int)(t / g.nx) + 1;
                if (cell_covered(g, i1, j1, xe, N)) {
                    mine += m;
                    me[t] = 0;
                    ce[t] = 0xffu;
                    if (se) se[t] = t_stamp;
                }
            }
        }
        for (int off = 16; off; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
        if ((threadIdx.x & 31) == 0 && mine) atomicAdd(removed + e * removed_stride, mine);
    }
}
cudaError_t launch_remove_covered(unsigned char *mult, unsigned char *cls, const GridDesc &g, const double *xyT, int N,
                                  unsigned long long *removed, cudaStream_t s, int *stamp, int t_stamp, long long E,
                                  long long removed_stride)
{
    // the counters of the E stores only: what lies between them (a fire step's push counts) stays
    cudaError_t e = E == 1 ? cudaMemsetAsync(removed, 0, sizeof(unsigned long long), s)
                           : cudaMemset2DAsync(removed, (size_t)removed_stride * sizeof(unsigned long long), 0,
                                               sizeof(unsigned long long), (size_t)E, s);
    if (e != cudaSuccess) return e;
    const long long ncell = (long long)g.nx * g.ny;
    remove_covered_kernel<<<store_grid(ncell, 256, 148 * 8, E), 256, 0, s>>>(mult, cls, g, xyT, N, removed, stamp,
                                                                             t_stamp, E, removed_stride);
    return cudaGetLastError();
}

__global__ void covered_mask_kernel(unsigned char *mask, const __grid_constant__ GridDesc g,
                                    const double *__restrict__ xyT, int N)
{
    const long long ncell = (long long)g.nx * g.ny;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
         t += (long long)gridDim.x * blockDim.x) {
        const int i1 = (int)(t % g.nx) + 1, j1 = (int)(t / g.nx) + 1;
        mask[t] = cell_covered(g, i1, j1, xyT, N) ? 1 : 0;
    }
}
cudaError_t launch_covered_mask(unsigned char *mask, const GridDesc &g, const double *xyT, int N,
                                cudaStream_t s)
{
    const long long ncell = (long long)g.nx * g.ny;
    const int block = 256;
    const int grid = (int)std::min<long long>((ncell + block - 1) / block, 148 * 8);
    covered_mask_kernel<<<max(grid, 1), block, 0, s>>>(mask, g, xyT, N);
    return cudaGetLastError();
}

// append list entries: multiplicities add up (saturation / mixed weights reported through *overflow).
// An empty cell carries class kNoClass; the first entry to arrive claims the cell's class with a
// byte-wide compare-and-swap, so concurrent entries on one cell cannot misread each other.
constexpr unsigned kNoClass = 0xffu;
__device__ __forceinline__ unsigned byte_cas(unsigned char *base, long long idx, unsigned expect, unsigned desired)
{
    unsigned int *word = reinterpret_cast<unsigned int *>(base + (idx & ~3ll));
    const int sh = (int)(idx & 3) * 8;
    unsigned int old = *word, assumed;
    do {
        assumed = old;
        const unsigned cur = (assumed >> sh) & 0xffu;
        if (cur != expect) return cur;
        old = atomicCAS(word, assumed, (assumed & ~(0xffu << sh)) | (desired << sh));
    } while (old != assumed);
    return expect;
}
// blockIdx.y strides over E stores side by side (launch_add_points); list_of NULL: entries 0 .. P-1 into store 0.
// Store e's bytes start at e * ncell, which need not be a word boundary: the words are formed from the absolute byte
// index on the 4-byte aligned bases, and two stores sharing a word is safe under the compare-and-swap.
__global__ void add_points_kernel(unsigned char *mult, unsigned char *cls, const int *__restrict__ cell_idx,
                                  const unsigned char *__restrict__ cell_cls, long long P, int *overflow, long long E,
                                  const long long *__restrict__ offsets, long long offsets_stride,
                                  const long long *__restrict__ list_of, long long ncell)
{
    for (long long e = blockIdx.y; e < E; e += gridDim.y) {
        long long q0 = 0, q1 = P;
        if (list_of) {
            const long long *o = offsets + list_of[e] * offsets_stride;
            q0 = o[0];
            q1 = o[1];
        }
        for (long long t = q0 + blockIdx.x * (long long)blockDim.x + threadIdx.x; t < q1;
             t += (long long)gridDim.x * blockDim.x) {
            const long long idx = e * ncell + cell_idx[t];
            const unsigned k = cell_cls[t];
            const unsigned seen = byte_cas(cls, idx, kNoClass, k);
            if (seen != kNoClass && seen != k) {
                atomicExch(overflow, 2); // entries of different weights on one cell
                continue;
            }
            unsigned int *word = reinterpret_cast<unsigned int *>(mult + (idx & ~3ll));
            const int sh = (int)(idx & 3) * 8;
            unsigned int old = *word, assumed;
            do {
                assumed = old;
                if (((assumed >> sh) & 0xffu) >= 255u) {
                    atomicExch(overflow, 1);
                    break;
                }
                old = atomicCAS(word, assumed, assumed + (1u << sh));
            } while (old != assumed);
        }
    }
}
// cells without entries carry kNoClass (after uploads and removals)
__global__ void normalize_cls_kernel(const unsigned char *__restrict__ mult, unsigned char *cls, long long ncell)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
         t += (long long)gridDim.x * blockDim.x)
        if (mult[t] == 0) cls[t] = (unsigned char)kNoClass;
}
cudaError_t launch_normalize_cls(const unsigned char *mult, unsigned char *cls, long long ncell, cudaStream_t s)
{
    const int block = 256;
    const int grid = (int)std::min<long long>((ncell + block - 1) / block, 148 * 8);
    normalize_cls_kernel<<<max(grid, 1), block, 0, s>>>(mult, cls, ncell);
    return cudaGetLastError();
}
cudaError_t launch_add_points(unsigned char *mult, unsigned char *cls, const int *cell_idx,
                              const unsigned char *cell_cls, long long P, int *overflow, cudaStream_t s, long long E,
                              const long long *offsets, long long offsets_stride, const long long *list_of,
                              long long ncell)
{
    if (P <= 0) return cudaSuccess;
    add_points_kernel<<<store_grid(P, 256, 148 * 8, E), 256, 0, s>>>(mult, cls, cell_idx, cell_cls, P, overflow, E,
                                                                     offsets, offsets_stride, list_of, ncell);
    return cudaGetLastError();
}

// ---- poll winner: (min objective, smallest index among ties); NaN objectives never win -----
__device__ __forceinline__ bool better(double a, long long ia, double b, long long ib)
{
    return (a < b) || (a == b && ia < ib);
}
__global__ void argmin_stage1(const double *__restrict__ obj, const unsigned char *__restrict__ feasible,
                              long long B, int barrier, double *so, long long *si)
{
    double best = __longlong_as_double(0x7ff0000000000000ll);
    long long bi = -1;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < B;
         t += (long long)gridDim.x * blockDim.x) {
        double v = obj[t];
        if (barrier && feasible && !feasible[t]) continue;
        if (v != v) continue;
        if (bi < 0 || better(v, t, best, bi)) {
            best = v;
            bi = t;
        }
    }
    __shared__ double sb[32];
    __shared__ long long sbi[32];
    for (int off = 16; off; off >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, off);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, off);
        if (oi >= 0 && (bi < 0 || better(ob, oi, best, bi))) {
            best = ob;
            bi = oi;
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        sb[warp] = best;
        sbi[warp] = bi;
    }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        best = lane < nw ? sb[lane] : __longlong_as_double(0x7ff0000000000000ll);
        bi = lane < nw ? sbi[lane] : -1;
        for (int off = 16; off; off >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, off);
            const long long oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (oi >= 0 && (bi < 0 || better(ob, oi, best, bi))) {
                best = ob;
                bi = oi;
            }
        }
        if (lane == 0) {
            so[blockIdx.x] = best;
            si[blockIdx.x] = bi;
        }
    }
}
__global__ void argmin_stage2(double *so, long long *si, int n)
{
    // one warp folds the per-block partials into slot 0
    const int lane = threadIdx.x;
    double best = __longlong_as_double(0x7ff0000000000000ll);
    long long bi = -1;
    for (int t = lane; t < n; t += 32) {
        const double v = so[t];
        const long long i = si[t];
        if (i >= 0 && (bi < 0 || better(v, i, best, bi))) {
            best = v;
            bi = i;
        }
    }
    for (int off = 16; off; off >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, off);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, off);
        if (oi >= 0 && (bi < 0 || better(ob, oi, best, bi))) {
            best = ob;
            bi = oi;
        }
    }
    if (lane == 0) {
        so[0] = best;
        si[0] = bi;
    }
}
cudaError_t launch_argmin(const double *obj, const unsigned char *feasible, long long B, int barrier,
                          double *scratch_obj, long long *scratch_idx, int scratch_n, cudaStream_t s)
{
    const int block = 256;
    int grid = (int)std::min<long long>((B + block - 1) / block, (long long)scratch_n);
    grid = max(grid, 1);
    argmin_stage1<<<grid, block, 0, s>>>(obj, feasible, B, barrier, scratch_obj, scratch_idx);
    argmin_stage2<<<1, 32, 0, s>>>(scratch_obj, scratch_idx, grid);
    return cudaGetLastError();
}

// ---- synthetic candidates on the device: Philox4x32-10, counter = (index lo, index hi, uav, draw),
//      key = (seed lo, seed hi). The host reproduces the same stream (synth.py); philox4x32_10 is in
//      cov_device.cuh. ----
__device__ __forceinline__ double u01_53(uint32_t a, uint32_t b)
{
    // 53 random bits -> [0, 1)
    const unsigned long long v = ((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6);
    return __dmul_rn((double)v, 1.1102230246251565e-16); // 2^-53
}
// ---- forest-fire cellular automaton on the device (src/DynamicArea.jl:52-72 of /root/reference) ----
// One thread per interior cell.  A TREE cell with burning Moore neighbours draws once PER burning
// neighbour, window index (a, b) iterated column-major like findall; a success sets FIRE and pushes
// one list entry (so a cell can be pushed several times in a step: the duplicates of FirePoints.xlsx).
// rand() is replaced by a counter-based uniform: Philox4x32-10 with counter
// (cell index, step, neighbour index k = (a-1) + 3(b-1), 0) and key = seed.
// blockIdx.y strides over E automata side by side (launch_fire_step); E = 1 with zero strides is the single automaton.
__global__ void fire_step_kernel(const unsigned char *__restrict__ cur, unsigned char *__restrict__ nxt,
                                 unsigned char *mult, unsigned char *cls, int nx, int ny, unsigned long long seed,
                                 unsigned int step, const double *__restrict__ p_dir, int append,
                                 unsigned long long *pushed, int *overflow, long long E, unsigned long long seed_stride,
                                 long long pushed_stride)
{
    const long long ncell = (long long)nx * ny;
    for (long long e = blockIdx.y; e < E; e += gridDim.y) {
        const unsigned char *ce = cur + e * ncell;
        unsigned char *ne = nxt + e * ncell, *me = mult + e * ncell, *ke = cls + e * ncell;
        const double *pe = p_dir + 9 * e;
        const unsigned long long key = seed + (unsigned long long)e * seed_stride;
        unsigned long long mine = 0;
        for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
             t += (long long)gridDim.x * blockDim.x) {
            const int i = (int)(t % nx) + 1, j = (int)(t / nx) + 1; // 1-based grid[i, j]
            unsigned char st = ce[t];
            unsigned pushes = 0;
            if (st == 1 && i >= 2 && i <= nx - 1 && j >= 2 && j <= ny - 1) {
                for (int b = 1; b <= 3; ++b)
                    for (int a = 1; a <= 3; ++a) {
                        const long long nb = (long long)(i - 2 + a - 1) + (long long)nx * (j - 2 + b - 1);
                        if (ce[nb] != 2) continue;
                        const int k = (a - 1) + 3 * (b - 1);
                        uint32_t r[4];
                        philox4x32_10((uint32_t)t, step, (uint32_t)k, (uint32_t)((unsigned long long)t >> 32),
                                      (uint32_t)key, (uint32_t)(key >> 32), r);
                        if (pe[k] > u01_53(r[0], r[1])) ++pushes;
                    }
                if (pushes) st = 2;
            }
            ne[t] = st;
            if (pushes && append) {
                const unsigned m = me[t] + pushes; // one thread per cell: no race
                if (m > 255u) atomicExch(overflow, 1);
                me[t] = (unsigned char)(m > 255u ? 255u : m);
                ke[t] = 0;
            }
            mine += pushes;
        }
        for (int off = 16; off; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
        if ((threadIdx.x & 31) == 0 && mine) atomicAdd(pushed + e * pushed_stride, mine);
    }
}

// initial state -> the list entries of the ignition cells (src/DynamicArea.jl:37-43)
__global__ void fire_seed_kernel(const unsigned char *__restrict__ state, unsigned char *mult, unsigned char *cls,
                                 long long ncell, int push_initial)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < ncell;
         t += (long long)gridDim.x * blockDim.x) {
        const bool burning = push_initial && state[t] == 2;
        mult[t] = burning ? 1 : 0;
        cls[t] = burning ? 0 : 0xffu;
    }
}

__global__ void generate_kernel(double *X, long long B, int N, unsigned long long seed, long long first, double lx,
                                double ly, double h_min, double h_max, double tan_half_fov)
{
    const long long total = B * N;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const long long b = t / N;
        const int u = (int)(t % N);
        const unsigned long long idx = (unsigned long long)(first + b);
        uint32_t r[4], q[4];
        philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
        philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)u, 1u, (uint32_t)seed, (uint32_t)(seed >> 32), q);
        const double x = __dmul_rn(u01_53(r[0], r[1]), lx);
        const double y = __dmul_rn(u01_53(r[2], r[3]), ly);
        const double h = __dadd_rn(h_min, __dmul_rn(u01_53(q[0], q[1]), __dsub_rn(h_max, h_min)));
        double *row = X + b * 3 * N;
        row[u] = x;
        row[N + u] = y;
        row[2 * N + u] = __dmul_rn(h, tan_half_fov);
    }
}
cudaError_t launch_generate(double *dX, long long B, int N, unsigned long long seed, long long first,
                            double lx, double ly, double h_min, double h_max, double tan_half_fov,
                            cudaStream_t s)
{
    if (B <= 0) return cudaSuccess;
    const int block = 256;
    const int grid = (int)std::min<long long>((B * N + block - 1) / block, 148 * 16);
    generate_kernel<<<grid, block, 0, s>>>(dX, B, N, seed, first, lx, ly, h_min, h_max, tan_half_fov);
    return cudaGetLastError();
}

// ---- packed candidates (cov_eval_batch_packed): mesh indices or FP32 values widened to the Float64 matrix the
// objective kernels read.  MADS trial points sit on a granular mesh (granularity 1.0 on every variable in the
// reference, src/TDM_STATIC_opt.jl:131-137), so a candidate is q * granularity with small integers q: 2 or 4 bytes per
// variable cross PCIe instead of 8 and the value the kernels see is the same double (one exact conversion, one
// correctly rounded multiply -- exact itself when granularity is a power of two or the product fits 53 bits).
// HBM-bound and tiny beside the objective kernel: 4 elements per thread when both sides are 16-byte aligned.
template <typename T>
__device__ __forceinline__ double unpack_one(T v, double g)
{
    return __dmul_rn((double)v, g);
}
template <>
__device__ __forceinline__ double unpack_one<float>(float v, double)
{
    return (double)v;
}
template <typename T, typename V4, bool VEC>
__global__ void unpack_kernel(const T *__restrict__ in, double *__restrict__ out, long long n, double g)
{
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (VEC) {
        const long long n4 = n >> 2;
        for (long long i = tid; i < n4; i += stride) {
            const V4 v = reinterpret_cast<const V4 *>(in)[i];
            double2 a, b;
            a.x = unpack_one<T>(v.x, g);
            a.y = unpack_one<T>(v.y, g);
            b.x = unpack_one<T>(v.z, g);
            b.y = unpack_one<T>(v.w, g);
            reinterpret_cast<double2 *>(out)[2 * i] = a;
            reinterpret_cast<double2 *>(out)[2 * i + 1] = b;
        }
        const long long t = (n4 << 2) + tid; // the last n % 4 elements
        if (t < n) out[t] = unpack_one<T>(in[t], g);
    } else {
        for (long long i = tid; i < n; i += stride) out[i] = unpack_one<T>(in[i], g);
    }
}
template <typename T, typename V4>
static cudaError_t launch_unpack_t(const void *raw, double g, double *out, long long n, cudaStream_t s)
{
    const bool vec = (((uintptr_t)raw | (uintptr_t)out) & 15u) == 0;
    const int block = 256;
    const long long items = vec ? (n + 3) / 4 : n;
    const int grid = (int)std::max<long long>(1, std::min<long long>((items + block - 1) / block, 148 * 16));
    if (vec) unpack_kernel<T, V4, true><<<grid, block, 0, s>>>((const T *)raw, out, n, g);
    else unpack_kernel<T, V4, false><<<grid, block, 0, s>>>((const T *)raw, out, n, g);
    return cudaGetLastError();
}
cudaError_t launch_unpack(const void *raw, int pack, double g, double *out, long long n, cudaStream_t s)
{
    if (n <= 0) return cudaSuccess;
    switch (pack) {
    case 1: return launch_unpack_t<float, float4>(raw, g, out, n, s);
    case 2: return launch_unpack_t<int, int4>(raw, g, out, n, s);
    case 3: return launch_unpack_t<short, short4>(raw, g, out, n, s);
    default: return cudaErrorInvalidValue;
    }
}


// ---- continuous variant: exact area of the union of the discs of a candidate (SURVEY.md 8f-4) ----
// Boundary integration (Green's theorem): for every circle, the arcs that lie inside no other disc
// contribute 1/2 * integral (x dy - y dx) = 1/2 [R^2 (t2 - t1) + R (cx (sin t2 - sin t1) - cy (cos t2 - cos t1))].
// The reference ships only the pair primitives of this method (src/Base_Functions.jl:230-355: distance,
// contained, intersection) and no driver; containment / tangency are decided like `contained` (<=) and
// identical discs keep the lower index.  One warp per candidate, lanes over its circles (N <= 64), FP64;
// the per-circle terms are summed in a fixed order, so the result is deterministic.
constexpr int kUnionMaxN = 64;
__global__ void union_area_kernel(const double *__restrict__ X, long long B, int N, double *__restrict__ area)
{
    const long long warp_global = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    const double two_pi = 6.283185307179586;
    for (long long b = warp_global; b < B; b += n_warps) {
        const double *x = X + b * 3 * N;
        double mine = 0.0;
        for (int i = lane; i < N; i += 32) {
            const double cxi = x[i], cyi = x[N + i], Ri = x[2 * N + i];
            if (!(Ri > 0.0)) continue;
            double ia[2 * kUnionMaxN], ib[2 * kUnionMaxN]; // covered angular intervals (local memory)
            int n = 0;
            bool whole = false;
            for (int j = 0; j < N && !whole; ++j) {
                const double Rj = x[2 * N + j];
                if (j == i || !(Rj > 0.0)) continue;
                const double dx = x[j] - cxi, dy = x[N + j] - cyi;
                const double d = hypot(dx, dy);
                if (d >= Ri + Rj) continue;
                if (d + Ri <= Rj) { // circle i inside disc j (identical discs: the lower index survives)
                    if (d + Rj <= Ri && i < j) continue;
                    whole = true;
                    break;
                }
                if (d + Rj <= Ri) continue; // disc j inside disc i: does not touch i's boundary
                const double phi = atan2(dy, dx);
                const double c = (Ri * Ri + d * d - Rj * Rj) / (2.0 * Ri * d);
                const double alpha = acos(fmax(-1.0, fmin(1.0, c)));
                double a = fmod(phi - alpha, two_pi);
                if (a < 0.0) a += two_pi;
                const double e = a + 2.0 * alpha;
                if (e > two_pi) {
                    ia[n] = a; ib[n++] = two_pi;
                    ia[n] = 0.0; ib[n++] = e - two_pi;
                } else {
                    ia[n] = a; ib[n++] = e;
                }
            }
            if (whole) continue;
            for (int p = 1; p < n; ++p) { // insertion sort by interval start
                const double ka = ia[p], kb = ib[p];
                int q = p - 1;
                while (q >= 0 && ia[q] > ka) {
                    ia[q + 1] = ia[q];
                    ib[q + 1] = ib[q];
                    --q;
                }
                ia[q + 1] = ka;
                ib[q + 1] = kb;
            }
            double pos = 0.0, acc = 0.0;
            for (int p = 0; p <= n; ++p) {
                const double a = p < n ? ia[p] : two_pi;
                if (a > pos) { // exposed arc [pos, a]
                    double s1, c1, s2, c2;
                    sincos(pos, &s1, &c1);
                    sincos(a, &s2, &c2);
                    acc += 0.5 * (Ri * Ri * (a - pos) + Ri * (cxi * (s2 - s1) - cyi * (c2 - c1)));
                }
                if (p < n) pos = fmax(pos, ib[p]);
            }
            mine += acc;
        }
        // fixed-order reduction over the lanes
        for (int off = 16; off; off >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, off);
        if (lane == 0) area[b] = mine;
    }
}
// Large swarms (64 < N <= kMaxUavs): one CTA per candidate, one warp per circle i, lanes over the other
// circles j.  The covered angular intervals of circle i go to the warp's list in shared memory (warp-
// aggregated appends); instead of sorting them, every interval END that no other interval covers opens an
// exposed arc, which runs to the nearest interval START at or after it (plus the arc that starts at angle 0
// when 0 is uncovered).  Among intervals with the same end the lowest list position speaks for all, and angle 0
// speaks for every end at 0.  Same formulas and tie rules as union_area_kernel; sums in a fixed order (deterministic).
constexpr int kUnionBigWarps = 4;
__global__ void __launch_bounds__(kUnionBigWarps * 32)
union_area_big_kernel(const double *__restrict__ X, long long B, int N, double *__restrict__ area)
{
    extern __shared__ __align__(16) unsigned char union_smem[];
    double *xs = reinterpret_cast<double *>(union_smem);                        // 3N staged doubles
    double *lists = xs + 3 * N;                                                 // per warp: 2N starts, 2N ends
    __shared__ double s_part[kUnionBigWarps];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double *ia = lists + (size_t)warp * 4 * N, *ib = ia + 2 * N;
    const double two_pi = 6.283185307179586;
    for (long long b = blockIdx.x; b < B; b += gridDim.x) {
        __syncthreads(); // previous candidate retired
        for (int t = tid; t < 3 * N; t += blockDim.x) xs[t] = __ldg(X + b * 3 * N + t);
        __syncthreads();
        double mine = 0.0; // lane-partial sum of this warp's circles
        for (int i = warp; i < N; i += kUnionBigWarps) {
            const double cxi = xs[i], cyi = xs[N + i], Ri = xs[2 * N + i];
            if (!(Ri > 0.0)) continue; // warp-uniform
            int n = 0;                 // list length, the same in every lane
            bool whole = false;
            for (int j0 = 0; j0 < N && !whole; j0 += 32) {
                const int j = j0 + lane;
                int k = 0; // intervals this lane appends (0, 1 or 2)
                double a0 = 0, b0 = 0, a1 = 0, b1 = 0;
                bool inside = false;
                if (j < N && j != i) {
                    const double Rj = xs[2 * N + j];
                    if (Rj > 0.0) {
                        const double dx = xs[j] - cxi, dy = xs[N + j] - cyi;
                        const double d = hypot(dx, dy);
                        if (d < Ri + Rj) {
                            if (d + Ri <= Rj) {
                                inside = !(d + Rj <= Ri && i < j); // identical discs: the lower index survives
                            } else if (!(d + Rj <= Ri)) {
                                const double phi = atan2(dy, dx);
                                const double c = (Ri * Ri + d * d - Rj * Rj) / (2.0 * Ri * d);
                                const double alpha = acos(fmax(-1.0, fmin(1.0, c)));
                                double a = fmod(phi - alpha, two_pi);
                                if (a < 0.0) a += two_pi;
                                const double e = a + 2.0 * alpha;
                                if (e > two_pi) {
                                    a0 = a; b0 = two_pi; a1 = 0.0; b1 = e - two_pi; k = 2;
                                } else {
                                    a0 = a; b0 = e; k = 1;
                                }
                            }
                        }
                    }
                }
                whole = __any_sync(0xffffffffu, inside);
                // exclusive prefix of k over the lanes: list positions in (j, first/second) order
                int incl = k;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, off);
                    if (lane >= off) incl += v;
                }
                const int at = n + incl - k;
                if (k >= 1) { ia[at] = a0; ib[at] = b0; }
                if (k == 2) { ia[at + 1] = a1; ib[at + 1] = b1; }
                n += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (whole) continue;
            __syncwarp();
            // candidates for the start of an exposed arc: angle 0 (p == -1) and every interval end
            double acc = 0.0;
            for (int p = lane - 1; p < n; p += 32) {
                const double pos = p < 0 ? 0.0 : ib[p];
                // an end at angle 0 (a zero-length interval there, when alpha rounds to 0) is angle 0's own candidate
                bool covered = !(pos < two_pi) || (p >= 0 && pos == 0.0);
                double nxt = two_pi;
                for (int q = 0; q < n && !covered; ++q) {
                    const double aq = ia[q], bq = ib[q];
                    if (q != p && aq <= pos && (pos < bq || (pos == bq && q < p))) covered = true;
                    if (aq > pos && aq < nxt) nxt = aq; // (a start AT pos either covers it or is a zero-length interval)
                }
                if (!covered && nxt > pos) {
                    double s1, c1, s2, c2;
                    sincos(pos, &s1, &c1);
                    sincos(nxt, &s2, &c2);
                    acc += 0.5 * (Ri * Ri * (nxt - pos) + Ri * (cxi * (s2 - s1) - cyi * (c2 - c1)));
                }
            }
            mine += acc;
            __syncwarp(); // the list is rewritten for the warp's next circle
        }
        for (int off = 16; off; off >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, off);
        if (lane == 0) s_part[warp] = mine;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int w = 0; w < kUnionBigWarps; ++w) tot += s_part[w];
            area[b] = tot;
        }
    }
}

cudaError_t launch_union_area(const double *dX, long long B, int N, double *d_area, cudaStream_t s)
{
    if (B <= 0) return cudaSuccess;
    if (N > kUnionMaxN) {
        const int smem = (3 * N + kUnionBigWarps * 4 * N) * 8;
        cudaError_t err = cudaFuncSetAttribute(union_area_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (err != cudaSuccess) return err;
        const int grid = (int)std::min<long long>(B, 148 * 4);
        union_area_big_kernel<<<grid, kUnionBigWarps * 32, smem, s>>>(dX, B, N, d_area);
        return cudaGetLastError();
    }
    const int block = 128;
    const int grid = (int)std::min<long long>((B * 32 + block - 1) / block, 148 * 16);
    union_area_kernel<<<grid, block, 0, s>>>(dX, B, N, d_area);
    return cudaGetLastError();
}

cudaError_t launch_fire_step(const unsigned char *cur, unsigned char *nxt, unsigned char *mult, unsigned char *cls,
                             int nx, int ny, unsigned long long seed, unsigned int step, const double *p_dir,
                             int append, unsigned long long *pushed, int *overflow, cudaStream_t s, long long E,
                             unsigned long long seed_stride, long long pushed_stride)
{
    const long long ncell = (long long)nx * ny;
    fire_step_kernel<<<store_grid(ncell, 256, 148 * 8, E), 256, 0, s>>>(cur, nxt, mult, cls, nx, ny, seed, step, p_dir,
                                                                        append, pushed, overflow, E, seed_stride,
                                                                        pushed_stride);
    return cudaGetLastError();
}
cudaError_t launch_fire_seed(const unsigned char *state, unsigned char *mult, unsigned char *cls, long long ncell,
                             int push_initial, cudaStream_t s)
{
    const int block = 256;
    const int grid = (int)std::min<long long>((ncell + block - 1) / block, 148 * 8);
    fire_seed_kernel<<<max(grid, 1), block, 0, s>>>(state, mult, cls, ncell, push_initial);
    return cudaGetLastError();
}

} // namespace cov
