// cov_kernels.cuh -- launch interface between the C ABI (cov_api.cu) and the kernels
// (cov_kernels.cu, cov_grid_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include "cov_types.h"

namespace cov {

struct LaunchCfg {
    int kernel;          // COV_KERNEL_*
    int warps_per_cta;   // 0 = auto
    int ctas_per_sm;     // 0 = auto
    int band_rows;       // 0 = auto
    int force_exact;
    int num_sms;
    int max_smem_optin;  // bytes
    int plane_mode;      // CTA kernel: -1 auto, 0 lazy global, 1 early global, 2 staged per band (TMA), 3 sweep with
                         // a staged plane band, 4 sweep with the plane read through L2
    int ordered;         // 1: the store's area depends on the order of the Float64 additions -> ordered kernel
};

struct LaunchInfo {
    int grid, block, smem_bytes, band_rows, planes_in_smem;
    int kernel; // cov_kernel of the kernel that ran (SPAN = small-swarm, SPAN_GENERAL = CTA per candidate)
    // template instantiation that ran (names the ncu profile the issue roofline is computed from)
    int multi;      // 1: several planes / classes / multiplicities
    int chunk;      // small-swarm kernel: candidates per unit (CHUNK); else 0
    int max_warps;  // small-swarm kernel: MAXW of the instantiation (20 or 24); else 0
    int plane_mode; // CTA kernel: 0 lazy, 1 early, 2 staged, 3 sweep, 4 sweep through L2 (PLANES); else -1
};

// Coverage objective over B candidates (device pointers). counter: one ZEROED unsigned long long
// per launch (work dispenser; the caller hands out fresh slots of a ring it zeroes in bulk, so no
// memset sits between consecutive launches). Returns cudaError_t.
cudaError_t launch_eval(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                        long long B, const EvalOut &out, unsigned long long *counter,
                        cudaStream_t stream, LaunchInfo *info);

// The small-swarm span kernel (cov_span_small.cu): N <= 8 and a framebuffer that fits shared memory.
bool span_small_applies(const GridDesc &g, int N, const LaunchCfg &cfg, long long B, int *warps_out, int *chunk_out);
cudaError_t launch_span_small(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                              long long B, const EvalOut &out, unsigned long long *counter, cudaStream_t stream,
                              LaunchInfo *info);

// The general span kernel (cov_span_cta.cu): one CTA per candidate, banded framebuffer.
cudaError_t launch_span_cta(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                            long long B, const EvalOut &out, unsigned long long *counter, cudaStream_t stream,
                            LaunchInfo *info);

// ---- the device MADS solver (cov_mads.cu): S independent solves, one persistent CTA per solve at a time ----
constexpr int kMadsMaxUavs = 64;    // N of the launch plan (2 * 3N = 384 poll points per iteration)
constexpr int kMadsPow10Min = -400; // pow10 holds 10^b for b in [kMadsPow10Min, -kMadsPow10Min]; clamped outside
struct MadsArgs {
    const double *X0;        // S x n start points (n = 3N)
    const double *a0;        // S x n initial poll-size mantissas (1, 2 or 5)
    const int *b0;           // S x n initial poll-size exponents
    const double *pow10;     // 10^b as the host's libm computes it, b = kMadsPow10Min .. -kMadsPow10Min
    double *X_out;           // S x n
    double *obj_out;         // S
    long long *stats;        // S x 4: iterations, evaluations, successes, converged
    long long S, n_iter;
    double granularity;
    unsigned long long seed; // solve k uses the Philox key seed + k
    int force_exact;
    int ordered;             // 1: the list-order Float64 sum (cov_grid_info.area_exact == 0)
};
// Shared-memory plan of the solver for this store and swarm size: warps per CTA and dynamic bytes; false when
// not even one warp's framebuffer fits (or N > kMadsMaxUavs).
bool mads_plan(const GridDesc &g, int N, const LaunchCfg &cfg, int *warps, int *smem, int *planes_smem);
cudaError_t launch_mads(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                        unsigned long long *counter, cudaStream_t stream);
// The solves of E scenarios in one launch (cov_run_horizon_ensemble): a.S = E * S solves, solve j of scenario j / S.
// Scenario e reads plane set e (g.planes + e * n_planes * plane_words, read through L2) and parameter block e (o's
// five arrays shifted by e * 5N); solve k of scenario e is keyed by a.seed + e * key_stride + k.
cudaError_t launch_scenario_mads(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                                 long long S, unsigned long long key_stride, unsigned long long *counter,
                                 cudaStream_t stream);
// AreaMaxObjective without the barrier of E swarms (X: E x 3N, device), swarm e on plane set e and parameter block e
// as above, one warp per swarm: obj[e].
cudaError_t launch_scenario_eval(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const double *X,
                                 long long E, double *obj, cudaStream_t stream);

// ---- the horizons on a list-order store (COV_OPT_LIST_ORDER_HORIZON; cov_mads.cu) ----
// Scenario e's point list after timestep t's removal, as liveness over one fixed sequence: the base list (the handle's
// at the call's start, append time 1), then the entries of schedule l = list_of[e] (list_of NULL: l = 0) up to
// off[l * T + t], appended at ta[q].  An entry is live iff stamps[e * ncell + cell] < its append time (stamps: the
// removal stamps of launch_remove_covered, zero before the call).  off NULL: the base list alone.
struct ListWalk {
    const int *base_cell;
    const unsigned char *base_cls;
    long long n_base;
    const int *cell;         // the schedules' entries (device)
    const unsigned char *cls;
    const int *ta;           // their append timesteps
    const long long *off;    // L T + 1 offsets (device, nullable)
    const long long *list_of; // E schedule numbers (device, nullable)
    long long T, t, ncell;
    const int *stamps;       // E x ncell
};
// The solves of E scenarios with the list-order sum (launch_scenario_mads' numbering and keys; E = 1: launch_mads'),
// scenario e on parameter block e and on its list; a.ordered and the plane sets are unused.
cudaError_t launch_list_mads(const GridDesc &g, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                             long long S, unsigned long long key_stride, const ListWalk &w,
                             unsigned long long *counter, cudaStream_t stream);
// AreaMaxObjective without the barrier of E swarms (X: E x 3N) on their lists, one warp per swarm: obj[e].
cudaError_t launch_list_eval(const GridDesc &g, const ObjParams &o, const ListWalk &w, const double *X, long long E,
                             double *obj, cudaStream_t stream);

// ---- cov_run_horizon (cov_horizon.cu): the kernels between the launchers above, per timestep t (1-based) ----
// A launch covers E scenarios side by side (cov_run_horizon_ensemble; E = 1: cov_run_horizon): scenario e's cur,
// parameter block and starts at e * 3N, e * 5N and e * S * 3N doubles.
struct HorizonStep {
    int N, n_boxes;
    long long t, S, E;
    double spread, granularity;
    unsigned long long seed;        // Philox key of scenario 0's perturbations
    unsigned long long seed_stride; // scenario e's key: seed + e * seed_stride
    const double *pow10;      // the solver's table (MadsArgs::pow10)
    const double *boxes;      // n_boxes x 4: x_LB, x_UB, y_LB, y_UB (device)
    double h_focus, h_max, tan_half_fov;
};
// The r_max rule (t >= 2, n_boxes > 0) and cons3's previous swarm := cur into params (cov_handle's 5N doubles:
// r_max, prev_x, prev_y, prev_z, cons3_G), and S starts with their initial meshes (start 0 = cur).
cudaError_t launch_horizon_start(const HorizonStep &s, const double *cur, double *params, double *X0, double *a0,
                                 int *b0, cudaStream_t stream);
// One CTA per scenario: the winner of S solves (Xs S x 3N, objs S, mstats S x 4) to cur, stats_row[0..2], and xyT of
// cur.  Scenario e's arrays are at e times their size, its stats row at e * row_stride.
cudaError_t launch_horizon_commit(long long S, int N, const double *Xs, const double *objs, const long long *mstats,
                                  double *cur, long long *stats_row, double *xyT, cudaStream_t stream, long long E = 1,
                                  long long row_stride = 0);

// ---- the grid-free static objective (cov_region.cu, cov_mads.cu; geometry and limits in cov_region.cuh) ----
// The arcs of the covered set's boundary inside the domain (r.arcs / r.K unused): at most cap of them to out, the
// count of all of them to *count (device).
cudaError_t launch_region_arcs(const RegionDesc &r, RegionArc *out, int cap, int *count, cudaStream_t s);
// obj / area / feasible (device, each nullable) of B candidates; cudaErrorInvalidConfiguration when N or the region
// exceed the shared-memory plan.
cudaError_t launch_region_eval(const RegionDesc &r, const ObjParams &o, const LaunchCfg &cfg, const double *dX,
                               long long B, double *obj, double *area, unsigned char *feasible, cudaStream_t s);
// cov_mads_solve_batch's solves with the region objective (a.force_exact and a.ordered unused).
cudaError_t launch_mads_region(const RegionDesc &r, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                               unsigned long long *counter, cudaStream_t stream);

// ---- cov_run_horizon_region (cov_region.cu, cov_mads.cu): the covered set grows on the device ----
// The discs sit at a fixed pitch (the call's M0 + T N), so appending never moves them; M and K live in ctl, because
// the R <= 0 filter and the arc count are known only on the device.  Once ctl[2] is set every kernel below returns at
// once, touching nothing.
constexpr int kCoverBadDisc = 1, kCoverManyArcs = 2; // ctl[2]
struct CoverSet {
    double x_lo, y_lo, x_hi, y_hi;
    double *discs;   // [x_1..x_pitch | y | R]: the first ctl[0] of each are the covered discs
    RegionArc *arcs; // the arcs of their boundary (capacity kRegionMaxArcs)
    int pitch;
    int *ctl;        // {M, K, failure (0: none), the timestep that failed}
};
// Step 1 of timestep t: cur's discs with R > 0 appended, the arcs recomputed, K to stats_row[3].
cudaError_t launch_cover_arcs(const CoverSet &c, const double *cur, int N, long long t, long long *stats_row,
                              cudaStream_t s);
// cov_mads_solve_batch_region's solves on the covered set as ctl gives it, with the shared-memory plan of pitch discs
// and kRegionMaxArcs arcs (cudaErrorInvalidConfiguration when even that plan's one warp does not fit).
cudaError_t launch_cover_mads(const CoverSet &c, const ObjParams &o, const LaunchCfg &cfg, const MadsArgs &a,
                              unsigned long long *counter, cudaStream_t stream);
// The region objective without the barrier of one swarm x (device, 3N) to *obj (device).
cudaError_t launch_cover_eval(const CoverSet &c, const ObjParams &o, const double *x, double *obj, cudaStream_t s);

// ---- cell-store kernels (cov_grid_kernels.cu) ----
// stats[0] = entries, stats[1] = cells, stats[2 + k] = OR of the multiplicities of class k
cudaError_t launch_grid_stats(const unsigned char *mult, const unsigned char *cls, long long ncell,
                              unsigned long long *stats, cudaStream_t s);
// The launchers below that take E work on E stores side by side (cov_run_horizon_ensemble): store e's mult / cls at
// e * nx*ny bytes, its plane set at e * n_planes * plane_words words, its xyT at e * 3N doubles.
cudaError_t launch_pack_planes(const unsigned char *mult, const unsigned char *cls, const GridDesc &g,
                               uint32_t *planes, cudaStream_t s, long long E = 1);
// plane 0 in the pair-aligned, swizzled layout of the CTA kernel's sweep mode (GridDesc::planes_q)
cudaError_t launch_requad_plane(const GridDesc &g, uint32_t *planes_q, cudaStream_t s);
cudaError_t launch_fill_full(unsigned char *mult, unsigned char *cls, long long ncell, cudaStream_t s);
cudaError_t launch_bits_to_cells(const uint32_t *bits, int nx, int ny, unsigned char *mult,
                                 unsigned char *cls, cudaStream_t s);
// xyT: 3N doubles on the device: cx[N], cy[N], T[N]. removed: one unsigned long long (store e's at e *
// removed_stride).  stamp (nullable, E x nx*ny ints): stamp[e * nx*ny + cell] = t_stamp for every cell of store e whose
// entries are removed.
cudaError_t launch_remove_covered(unsigned char *mult, unsigned char *cls, const GridDesc &g, const double *xyT, int N,
                                  unsigned long long *removed, cudaStream_t s, int *stamp = nullptr, int t_stamp = 0,
                                  long long E = 1, long long removed_stride = 0);
cudaError_t launch_normalize_cls(const unsigned char *mult, unsigned char *cls, long long ncell, cudaStream_t s);
cudaError_t launch_covered_mask(unsigned char *mask, const GridDesc &g, const double *xyT, int N,
                                cudaStream_t s);
cudaError_t launch_thresholds(const double *xyR, int N, double *xyT, cudaStream_t s, long long E = 1); // E swarms
// E stores side by side (cov_run_horizon_points_ensemble): store e's mult / cls at e * ncell bytes from 4-byte aligned
// bases; it appends entries offsets[list_of[e] * offsets_stride] .. offsets[list_of[e] * offsets_stride + 1] - 1 of
// (cell_idx, cell_cls), and P bounds the length of every such slice.  list_of NULL (E = 1): entries 0 .. P-1.
cudaError_t launch_add_points(unsigned char *mult, unsigned char *cls, const int *cell_idx,
                              const unsigned char *cell_cls, long long P, int *overflow, cudaStream_t s,
                              long long E = 1, const long long *offsets = nullptr, long long offsets_stride = 0,
                              const long long *list_of = nullptr, long long ncell = 0);
cudaError_t launch_argmin(const double *obj, const unsigned char *feasible, long long B, int barrier,
                          double *scratch_obj, long long *scratch_idx, int scratch_n, cudaStream_t s);
cudaError_t launch_union_area(const double *dX, long long B, int N, double *d_area, cudaStream_t s);
// E automata side by side (cov_run_horizon_fire_ensemble): automaton e's cur / nxt / mult / cls at e * nx*ny bytes, its
// 9 direction probabilities at p_dir + 9e, its key seed + e * seed_stride (mod 2^64), its push counter at
// pushed + e * pushed_stride; overflow is shared.
cudaError_t launch_fire_step(const unsigned char *cur, unsigned char *nxt, unsigned char *mult, unsigned char *cls,
                             int nx, int ny, unsigned long long seed, unsigned int step, const double *p_dir,
                             int append, unsigned long long *pushed, int *overflow, cudaStream_t s, long long E = 1,
                             unsigned long long seed_stride = 0, long long pushed_stride = 0);
cudaError_t launch_fire_seed(const unsigned char *state, unsigned char *mult, unsigned char *cls, long long ncell,
                             int push_initial, cudaStream_t s);
cudaError_t launch_generate(double *dX, long long B, int N, unsigned long long seed, long long first,
                            double lx, double ly, double h_min, double h_max, double tan_half_fov,
                            cudaStream_t s);
// n packed candidate values (pack: COV_PACK_F32 / _I32 / _I16 of coverage_cuda.h) -> doubles: value * g (FP32: value)
cudaError_t launch_unpack(const void *raw, int pack, double g, double *out, long long n, cudaStream_t s);

} // namespace cov
