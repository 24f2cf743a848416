/*
 * coverage_cuda.h -- C ABI of libcoverage_cuda, the B200 (sm_100a) batched coverage objective.
 *
 * The reference (Gabisanth/MaximumAreaCoverageOptimization.jl) is pure Julia and has NO FFI
 * boundary; its de-facto operator interface is what DirectSearch.jl accepts:
 *   SetObjective(p, f)            f(x::Vector{Float64})::Float64   src/TDM_STATIC_opt.jl:125
 *   AddExtremeConstraint(p, c)    c(x)::Bool                       src/TDM_STATIC_opt.jl:151-153
 *   createObjective(cells, N, r_max) -> f                          src/TDM_STATIC_opt.jl:82-100
 *   create_cons3(pre, FOV, d_lim)    -> c                          src/TDM_Constraints.jl:54-75
 * Each entry point below names the reference lines it replaces.  Julia binds them with `ccall`
 * (see INTEGRATION.md and maximumareacoverageoptimization.jl_b200/julia/CoverageCUDA.jl); the
 * tests bind them with Python ctypes.
 *
 * Conventions
 *  - plain C, no C++ types; sizes int64_t, reals double; every call returns COV_OK (0) or a
 *    negative cov_status, never throws; the message is at cov_last_error().
 *  - The library owns device buffers and streams.  Host pointers are caller-owned and borrowed
 *    only for the duration of the call; every call that takes host outputs is synchronous on
 *    return.  A handle is not thread-safe; distinct handles may be used from distinct threads
 *    (covers DirectSearch's SetMaxEvals threaded evaluation, src/TDM_STATIC_opt.jl:129).
 *  - Candidate layout: B x 3N doubles, candidate-major, each row [x_1..x_N, y_1..y_N, R_1..R_N]
 *    (src/AreaCoverageCalculation.jl:31,38-40).
 *  - Cell (i, j), i = 1..nx, j = 1..ny, has its centre at (i*dx - dx/2, j*dy - dy/2)
 *    (src/AreaCoverageCalculation.jl:16, src/DynamicArea.jl:65).  Per-cell arrays are indexed
 *    (i-1) + nx*(j-1), i.e. Julia's column-major grid[i, j].
 *  - There is no CPU fallback: without a CUDA device cov_create fails with COV_ERR_CUDA.
 */
#ifndef COVERAGE_CUDA_H
#define COVERAGE_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COV_ABI_VERSION 3 /* 2: COV_OPT_PROGRESSIVE_INDEX, COV_KERNEL_ORDERED, cov_get_class_weights, cov_eval_batch_best;
                             3: cov_eval_batch_packed (COV_PACK_*); later, with no existing symbol changed:
                                cov_mads_solve_batch; cov_set_region, cov_eval_region_batch,
                                cov_mads_solve_batch_region (the grid-free static objective); cov_run_horizon;
                                cov_run_horizon_points, cov_run_horizon_fire (the dynamic horizon);
                                cov_run_horizon_ensemble, cov_multi_run_horizon_ensemble;
                                cov_run_horizon_fire_ensemble, cov_multi_run_horizon_fire_ensemble;
                                cov_run_horizon_points_ensemble, cov_multi_run_horizon_points_ensemble;
                                COV_OPT_LIST_ORDER_HORIZON; cov_run_horizon_region (the grid-free horizon) */

#if defined(__GNUC__)
#define COV_API __attribute__((visibility("default")))
#else
#define COV_API
#endif

typedef enum cov_status {
    COV_OK = 0,
    COV_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, N mismatch ...) */
    COV_ERR_STATE = -2,     /* grid or parameters not set yet */
    COV_ERR_CUDA = -3,      /* CUDA runtime error (message has the CUDA error string) */
    COV_ERR_OFF_LATTICE = -4, /* cov_set_points: a point is not a cell centre of the lattice */
    COV_ERR_LIMIT = -5,     /* a size exceeds what the kernels support (see cov_limits) */
    COV_ERR_NOMEM = -6
} cov_status;

/* Kernel selection for cov_set_option(COV_OPT_KERNEL). */
enum {
    COV_KERNEL_AUTO = 0,    /* row-span kernels (default): the small-swarm variant (N <= 8, framebuffer in shared
                               memory) for batches of a thousand or two candidates and more, else the general one */
    COV_KERNEL_SPAN = 1,    /* row-span kernels, small-swarm variant whenever it applies (from 128 candidates on) */
    COV_KERNEL_BRUTE = 2,   /* every cell against every disc, FP32 band + FP64 exact band cells */
    COV_KERNEL_EXACT = 3,   /* every cell against every disc in FP64 only (slow cross-check) */
    COV_KERNEL_SPAN_GENERAL = 4, /* force the general span kernel (one CTA per candidate, any N) */
    COV_KERNEL_ORDERED = 5  /* the reference's own loop over the point list in list order, FP64 only: the Float64 area is
                               the reference's whatever the weights. Chosen automatically (whatever this option says)
                               when cov_grid_info.area_exact == 0; selectable as a cross-check otherwise */
};

enum {
    COV_OPT_KERNEL = 1,         /* one of COV_KERNEL_* */
    COV_OPT_WARPS_PER_CTA = 2,  /* 0 = auto */
    COV_OPT_CTAS_PER_SM = 3,    /* 0 = auto */
    COV_OPT_BAND_ROWS = 4,      /* span kernel framebuffer band height in rows; 0 = auto */
    COV_OPT_FORCE_EXACT = 5,    /* 1: span/brute kernels skip the FP32 band and decide every edge in FP64 */
    COV_OPT_CHUNK = 6,          /* host-path pipeline chunk (candidates per H2D/launch/D2H slice); 0 = auto */
    COV_OPT_TRACE = 7,          /* 1: record a per-slice device timeline of every host-path call (cov_get_trace) */
    COV_OPT_PLANE_MODE = 9,     /* CTA kernel, how fire words are read: -1 auto (default), 0 through L2 only when
                                   the framebuffer atomic left new bits, 1 through L2 ahead of the atomics,
                                   2 staged in shared memory band by band with TMA bulk copies, 3 paint-then-sweep
                                   (spans only painted, then popc(framebuffer & staged plane) over the band), 4 the
                                   same with the plane read through L2 in the sweep (no staging: taller bands or a
                                   fourth CTA per SM; what auto picks unless the swarm is tiny for its grid) */
    COV_OPT_ZEROCOPY_OUT = 8,   /* 1 (default): the host path's kernels write their results straight into pinned host
                                   memory; 0: into device buffers, copied back slice by slice */
    COV_OPT_PROGRESSIVE_INDEX = 10, /* which progressive constraint the `progressive` output of cov_eval_batch_ex is:
                                   0 (default) cons1_progressive = sum over every UAV of max(R_i - r_max_i, 0.0)
                                   (src/TDM_Constraints.jl:182-195); k >= 1 the single-UAV forms, 1-based index as in
                                   the reference: 2 = cons2_progressive (:197-208), 3 = cons3_progressive (:210-221).
                                   k > N is rejected by the evaluation calls with COV_ERR_INVALID */
    COV_OPT_LIST_ORDER_HORIZON = 11 /* 0 (default): the horizons refuse a store whose area depends on the list order
                                   (cov_grid_info.area_exact == 0) with COV_ERR_STATE; 1: cov_run_horizon,
                                   cov_run_horizon_points and their ensembles (cov_multi_* through their member
                                   handles) accept it and replay the reference's list-order sum on the device, every
                                   candidate walking the whole point list (the cost of COV_KERNEL_ORDERED).  Dyadic
                                   stores run as with 0, and the automaton horizons refuse such stores either way.
                                   Other values: COV_ERR_INVALID */
};

typedef struct cov_handle cov_handle;
typedef struct cov_multi cov_multi;

/* ---- lifecycle ------------------------------------------------------------------------- */
COV_API int cov_abi_version(void);
COV_API int cov_device_count(void);                       /* 0 when no CUDA device is usable */
COV_API int cov_create(int device, cov_handle **out);
COV_API void cov_destroy(cov_handle *h);
/* Message of the last failing call on this handle (h == NULL: last failing call of this thread
 * that had no handle, e.g. cov_create). Never NULL. */
COV_API const char *cov_last_error(const cov_handle *h);
COV_API int cov_set_option(cov_handle *h, int option, int64_t value);
COV_API int cov_get_option(const cov_handle *h, int option, int64_t *value);

/* ---- the cell store (replaces CellFunctions.Cells.points_of_interest as the kernel's input;
 *      src/CellFunctions.jl:5-16, producers src/AreaCoverageCalculation.jl:11-21,
 *      src/CellFunctions.jl:20-79) -----------------------------------------------------------
 * The store also stands for a point LIST, whose order decides the Float64 area when the weights are not
 * dyadic (cov_grid_info.area_exact == 0, COV_KERNEL_ORDERED):
 *  - cov_set_points: the order given;
 *  - cov_set_grid_bits, cov_set_grid_cells, cov_set_grid_full, cov_fire_init and cov_fire_step: createPOI's order
 *    (i outer, j inner, src/AreaCoverageCalculation.jl:14-15), the entries of a cell next to each other (these
 *    stores hold one weight class, or several given per cell by cov_set_grid_cells);
 *  - cov_add_points: the new entries after all the others, in the order given (push!, src/CellFunctions.jl:74);
 *  - cov_remove_covered: the remaining entries keep their order (src/CellFunctions.jl:81-108). */

/* 1 bit per cell, every set cell is one list entry of weight `weight`.
 * bits: ny rows of ceil(nx/32) uint32 words; bit b of word w of row j-1 is cell i = 32*w + b + 1. */
COV_API int cov_set_grid_bits(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy,
                      const uint32_t *bits, double weight);

/* Per-cell multiplicity (how many list entries sit on the cell; the fire list repeats cells,
 * src/DynamicArea.jl:61-67) and optional per-cell weight class.
 * mult: nx*ny bytes; cls: nx*ny bytes or NULL (all class 0); class_weight: n_classes doubles. */
COV_API int cov_set_grid_cells(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy,
                       const uint8_t *mult, const uint8_t *cls, int64_t n_classes,
                       const double *class_weight);

/* The reference's own list: P entries [x, y, area, weight, covered] (P*5 doubles). Every point
 * must be a cell centre of the nx x ny lattice (bit-exactly i*dx - dx/2), else
 * COV_ERR_OFF_LATTICE; all entries on one cell must carry the same weight; distinct weights
 * become weight classes in order of first appearance. Entry 5 (the covered flag) is ignored as
 * in calculateArea (src/AreaCoverageCalculation.jl:69 is commented out). */
COV_API int cov_set_points(cov_handle *h, const double *pts5, int64_t P, int64_t nx, int64_t ny, double dx,
                   double dy);

/* createPOI(dx, dy, nx, ny) built on the device (src/AreaCoverageCalculation.jl:11-21). */
COV_API int cov_set_grid_full(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy);

/* Append list entries (update_POI, src/CellFunctions.jl:59-79): same rules as cov_set_points,
 * multiplicities add up. Limits of the store (also of cov_set_points): at most 4 distinct weights (weight classes),
 * one weight per cell, at most 255 entries per cell, at most 8 bit planes (the set bits of the multiplicities of
 * each class, summed over the classes) (COV_ERR_LIMIT / COV_ERR_INVALID otherwise). A failing append leaves the
 * store exactly as it was. */
COV_API int cov_add_points(cov_handle *h, const double *pts5, int64_t P);

typedef struct cov_grid_info {
    int64_t nx, ny;
    double dx, dy;
    int64_t n_entries;      /* list entries = sum of multiplicities */
    int64_t n_cells;        /* cells with multiplicity > 0 */
    int64_t n_planes;       /* bit planes the kernels sweep */
    int64_t n_classes;
    int32_t area_exact;     /* 1: weight*count is exactly representable for every reachable count,
                               so the returned Float64 area equals the reference's list-order sum */
    int32_t planes_in_smem; /* 1: the span kernel stages the planes in shared memory */
} cov_grid_info;
COV_API int cov_get_grid_info(const cov_handle *h, cov_grid_info *info);
/* The weight of every class as the device numbers them (class k of `class_count`, the order fixed when the
 * store was created; it does NOT follow later removals). Writes min(cap, n_classes) doubles. */
COV_API int cov_get_class_weights(const cov_handle *h, double *class_weight, int64_t cap);
/* Read the device-resident multiplicity plane back (nx*ny bytes). */
COV_API int cov_get_grid_cells(cov_handle *h, uint8_t *mult);

/* rmvCoveredPOI (src/CellFunctions.jl:81-108): delete every entry covered by the discs xyR
 * ([x;y;R], 3N doubles) from the device-resident cell store. removed (nullable) = entries deleted. */
COV_API int cov_remove_covered(cov_handle *h, const double *xyR, int64_t N, int64_t *removed);

/* ---- forest-fire cellular automaton on the device (replaces the offline generator
 *      src/DynamicArea.jl:17-86 and its xlsx hand-off :100-108 to CellFunctions.update_POI) ----------
 * state: nx*ny bytes indexed (i-1) + nx*(j-1) like grid[i, j]: 0 = EMPTY, 1 = TREE, 2 = FIRE.
 * cov_fire_init uploads it and re-creates the cell store on the same lattice (weight dx*dy); with
 * push_initial != 0 every burning cell becomes one list entry (the reference's initial_points).
 * cov_fire_step is one update_grid(): each interior TREE cell draws once per burning Moore
 * neighbour, `wind_speed*cos(wind_direction - atan(2-b, 2-a))*prob_spread > u`, u from
 * Philox4x32-10 keyed by seed with counter (cell, step, neighbour); every success pushes one list
 * entry (append != 0: straight into the device-resident store; multiplicities add up like the
 * duplicates of FirePoints.xlsx). n_pushed (nullable) = entries pushed by this step. The pushed entries weigh
 * dx*dy, so the store must hold a single weight class of weight dx*dy (else COV_ERR_STATE, nothing changes); with one
 * class the order of the entries does not change the area. */
COV_API int cov_fire_init(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy, const uint8_t *state,
                          int32_t push_initial);
COV_API int cov_fire_step(cov_handle *h, double wind_speed, double wind_direction, double prob_spread,
                          uint64_t seed, int64_t step, int32_t append, int64_t *n_pushed);
COV_API int cov_fire_get_state(cov_handle *h, uint8_t *state);

/* ---- objective and constraint parameters (the closures' captured variables:
 *      createObjective(cells, N, r_max) src/TDM_STATIC_opt.jl:82, create_cons3(pre, FOV, d_lim)
 *      src/TDM_Constraints.jl:54, cons8's 15.0 :163, cons7 :142-154) --------------------------- */
COV_API int cov_set_params(cov_handle *h, int64_t N,
                   const double *r_max,        /* N */
                   double penalty_scale,       /* 1e5 in the reference */
                   const double *prev_xyR,     /* 3N [x;y;R] of the previous timestep, NULL: cons3 off */
                   const double *d_lim,        /* N (ignored when prev_xyR is NULL) */
                   double tan_half_fov,        /* tan(FOV/2) as the caller's libm computes it */
                   double sep_min,             /* cons8 threshold (15.0); <= 0: cons8 off */
                   int32_t use_cons7);         /* != 0: cons7 on */

/* ---- evaluation (replaces the per-trial-point loop of a MADS poll step, each iteration of which
 *      is cons_k(x) then AreaMaxObjective(x); SURVEY.md 3.1) -------------------------------- */

/* Host buffers. obj[b] = -area + penalty_scale * sum|R_i - r_max_i| (src/TDM_STATIC_opt.jl:89-97);
 * count[b] (nullable) = covered list entries; feasible[b] (nullable) = 1 iff every enabled
 * extreme constraint holds. The objective is computed for infeasible candidates too; applying
 * the extreme barrier is the caller's choice (cov_argmin applies it). */
COV_API int cov_eval_batch(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count,
                   uint8_t *feasible);

/* Extra per-candidate outputs (all nullable): class_count B x n_classes covered entries per
 * weight class; progressive B values of cons1_progressive (src/TDM_Constraints.jl:182-195). */
COV_API int cov_eval_batch_ex(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count,
                      uint8_t *feasible, int64_t *class_count, double *progressive);

/* Device buffers, asynchronous on the handle's stream (no host copies, no synchronisation). */
COV_API int cov_eval_batch_device(cov_handle *h, const double *dX, int64_t B, double *d_obj,
                          int64_t *d_count, uint8_t *d_feasible);

/* The scalar closure: AreaMaxObjective(x) for one candidate (src/TDM_STATIC_opt.jl:83-98). */
COV_API int cov_eval_one(cov_handle *h, const double *x, double *obj);

/* Poll winner: smallest objective and its 0-based index; among equal objectives the smallest index wins (MADS's
 * first strict minimum), however the candidates are split over threads, slices and devices. barrier != 0:
 * infeasible candidates are skipped (extreme barrier); if none is feasible best_idx = -1, best_obj = +Inf. A
 * feasible candidate whose objective is +Inf still counts: best_obj = +Inf with best_idx >= 0. The same rule holds
 * for cov_eval_batch_best, cov_eval_batch_packed and cov_multi_argmin. */
COV_API int cov_argmin(cov_handle *h, const double *X, int64_t B, int32_t barrier, double *best_obj,
               int64_t *best_idx);

/* cov_eval_batch and the poll winner in one call: the per-candidate outputs as above (obj nullable here) plus
 * (best_obj, best_idx) reduced on the device -- the 16 bytes a rank contributes to the (min, index) exchange
 * when the candidates of one poll are sharded over several GPUs (SURVEY.md 8e). */
COV_API int cov_eval_batch_best(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count,
                        uint8_t *feasible, int32_t barrier, double *best_obj, int64_t *best_idx);

/* The same evaluation for candidates that sit on a mesh, sent PACKED: the trial points of a MADS poll / search step
 * are x = q * granularity with integer q (granularity 1.0 on every variable in the reference,
 * src/TDM_STATIC_opt.jl:131-137), so 2 or 4 bytes per variable can cross PCIe instead of 8 -- the end-to-end rate
 * of cov_eval_batch is the PCIe rate (DESIGN.md 5). Q: B x 3N values in the candidate layout above, of type
 *   COV_PACK_I16  int16_t,  value = (double)q * granularity   (one correctly rounded FP64 multiply; exact
 *   COV_PACK_I32  int32_t,  value = (double)q * granularity    whenever granularity is a power of two)
 *   COV_PACK_F32  float,    value = (double)q                  (granularity ignored)
 * The device widens every slice into the Float64 matrix the kernels read, so the results are bit for bit those of
 * cov_eval_batch on the widened matrix. The caller vouches that its Float64 trial points ARE these values (integers
 * and FP32-representable numbers always are); nothing is rounded on the way in. obj / count / feasible as in
 * cov_eval_batch (obj may be NULL when a winner is asked for); best_obj and best_idx both NULL, or both given:
 * the poll winner as in cov_eval_batch_best. Pinned Q (cov_host_alloc) is DMA'd in place. */
enum { COV_PACK_F32 = 1, COV_PACK_I32 = 2, COV_PACK_I16 = 3 };
COV_API int cov_eval_batch_packed(cov_handle *h, const void *Q, int32_t pack, double granularity, int64_t B,
                          double *obj, int64_t *count, uint8_t *feasible, int32_t barrier, double *best_obj,
                          int64_t *best_idx);

/* A whole MADS solve in native code: the batch producer the reference lacks (DirectSearch.jl evaluates one
 * trial point per call). Settings of TDM_STATIC_opt.optimize (src/TDM_STATIC_opt.jl:118-222): start point x0
 * (3N), iteration limit n_iter (100 there), the same granularity on every variable (1.0 there), the enabled
 * constraints of cov_set_params as extreme barrier; x_out = the feasible incumbent if one was found, else x0.
 * Algorithm: granular-mesh MADS (Audet, Le Digabel & Tribes 2019), 2n Householder poll directions, complete
 * polling, one launch per poll set. stats (nullable): iterations, evaluations, batches, successes. */
COV_API int cov_mads_solve(cov_handle *h, const double *x0, int64_t n_iter, double granularity, uint64_t seed,
                           double *x_out, double *obj_out, int64_t *stats);

/* S independent MADS solves on the device, one kernel launch for all of them (multi-start: MADS is a local method).
 * Each CTA owns one solve from its first evaluation to its result; the host uploads the starts once, downloads the
 * results once and synchronises once.  X0, X_out: S x 3N in the candidate layout; obj_out (nullable): S values;
 * stats (nullable): S x 4 values [iterations, evaluations, successes, converged] -- converged = 1 when the solve
 * stopped because the mesh could not refine any further, 0 when it reached n_iter.  S == 0 does nothing.
 * Settings and results as cov_mads_solve: the constraints of cov_set_params as extreme barrier, one granularity on
 * every variable (0: continuous), X_out[k] = the feasible incumbent if one was found, else X0[k], obj_out[k] = its
 * barrier value (+Inf when no feasible point was found).  The loop is cov_mads_solve's in the same FP64 operations,
 * with two differences:
 *  - directions: solve k uses Philox4x32-10 keyed by (low, high 32 bits of seed + k mod 2^64).  At iteration t
 *    (0-based), variable i takes the 12 words of the blocks with counter (t low 32, t high 32, i, g), g = 0, 1, 2,
 *    summed as a uint64 s; v_i = s * 2^-32 - 6.0 (an Irwin-Hall(12) normal, mean 0, variance 1, exact in binary64);
 *    v /= sqrt(sum of v_i^2 summed in index order).  Powers of ten and the initial mesh are computed by the host's
 *    libm, so every iterate can be replayed on a host.  A start component that is +Inf or -Inf gets the poll size
 *    5 x 10^400 (b clamped to the table's 400), a NaN one 5 x 10^0; n_iter = 0 evaluates the start alone and
 *    returns it;
 *  - no cache and no duplicate removal: every kept poll point is evaluated (the winner, the first strict minimum in
 *    generation order -- sign + for columns 0..n-1, then sign -, is the same); evaluations counts them and x0.
 * Limits: N <= 64 (384 poll points per iteration) and a grid whose framebuffer (ny x stride words) fits one warp's
 * share of shared memory, else COV_ERR_LIMIT.  COV_OPT_FORCE_EXACT is honoured, COV_OPT_KERNEL does not apply
 * (stores with area_exact == 0 use the list-order sum, as every evaluation does).  cov_launch_count counts the
 * launch; cov_last_launch and the kernel timers are left unchanged. */
COV_API int cov_mads_solve_batch(cov_handle *h, const double *X0, int64_t S, int64_t n_iter, double granularity,
                                 uint64_t seed, double *X_out, double *obj_out, int64_t *stats);

/* The receding-horizon simulation on the device (FullSimulation.run_simulation, src/FullSimulation.jl:42-107, static
 * environment): T timesteps of rmvCoveredPOI and multi-start MADS, all enqueued before ONE synchronise at the end.
 * Needs a cell store with area_exact == 1 (or COV_OPT_LIST_ORDER_HORIZON at 1, below) and cov_set_params with
 * prev_xyR (cons3 on); the penalty, cons3's d_lim, cons7 and cons8 are the ones set there.  Let cur = x_start (3N).
 * For t = 1 .. T:
 *  1. rmvCoveredPOI(cur), as cov_remove_covered;
 *  2. for t >= 2 and n_boxes > 0 the r_max rule of FullSimulation.py:80-87 in its FP64 operations: for each UAV i with
 *     fabs(h_focus - R_i / tan_half_fov) < 1 and m = h_max * tan_half_fov, r_max[i] = h_focus * tan_half_fov if some
 *     box k has x_i < xu_k + m && x_i > xl_k - m && y_i < yu_k + m && y_i > yl_k - m, else m.  boxes: n_boxes x 4
 *     doubles x_LB, x_UB, y_LB, y_UB; tan_half_fov: cov_set_params's;
 *  3. cons3's previous swarm := cur (prev_z = R / tan_half_fov, as cov_set_params forms it);
 *  4. S starts: start 0 is cur; start k >= 1 moves x_i and y_i (never R) to v = cur + spread * z, snapped to
 *     nearbyint(v / g) * g when granularity g > 0.  z = s * 2^-32 - 6.0 with s the sum of the 12 words of the
 *     Philox4x32-10 blocks keyed by (low, high 32 bits of seed) with counter (t, k, j, 3 + q), q = 0, 1, 2 (t and k
 *     taken mod 2^32; j = i for x_i, N + i for y_i).  The direction stream of cov_mads_solve_batch only uses 0 .. 2 in
 *     that word.  The initial mesh of every start is cov_mads_solve_batch's, with floor(log10(target)) taken as the
 *     largest b >= 0 whose host-libm 10^b is <= target: the same b except for targets a few ulps below a power of
 *     ten, which mesh points are not (checked for every point |x| <= 10^4 of granularity 1, 0.5 and 0.25);
 *  5. the S solves of cov_mads_solve_batch (n_iter, granularity), solve k keyed by seed + (t - 1) S + k (mod 2^64);
 *  6. cur := X of the solve with the smallest barrier value (NaN counts as +Inf, ties to the smallest k; k = 0, whose
 *     X is cur itself, when none is finite); X_out row t-1 = cur;
 *  7. obj_out[t-1] (nullable) = AreaMaxObjective(cur) without the barrier, on step t's store and r_max.
 * stats (nullable): T x 4 [winner k, evaluations summed over the S solves, solves that found a feasible point,
 * entries removed in step 1]; step_ms (nullable): T device times between CUDA events recorded between the steps.
 * Afterwards the store holds every removal and the parameters are step T's (r_max, previous swarm), exactly as the
 * same sequence of existing calls leaves them.  T == 0 does nothing.  COV_ERR_STATE: no grid or parameters, cons3 off,
 * or area_exact == 0 unless COV_OPT_LIST_ORDER_HORIZON is 1; COV_ERR_LIMIT: cov_mads_solve_batch's limits;
 * COV_ERR_INVALID: T < 0, S < 1, n_iter < 0, NULL x_start or X_out when T > 0, spread not finite or < 0,
 * granularity < 0 or NaN, n_boxes < 0 or n_boxes > 0 with NULL boxes.  A refused call changes nothing.  cov_last_launch and the kernel
 * timers are left unchanged.
 *
 * List-order stores (COV_OPT_LIST_ORDER_HORIZON at 1; cov_run_horizon, cov_run_horizon_points and their ensembles).
 * A store whose area depends on the order of the list (non-dyadic weights such as update_POI's high-interest weight
 * (h_max tan(FOV/2))^2 pi) is accepted, and the call still equals its sequence of single calls bit for bit: those
 * calls already sum in list order, and so does the horizon.  Inside one call the list only loses every entry of a
 * covered cell (rmvCoveredPOI, order kept) and gains appends at its end (update_POI), so scenario e's list at timestep
 * t is a filter of one fixed sequence -- the handle's list at the call (its pending removals applied; createPOI's order
 * when no list is known), then the schedule's entries in timestep order -- in which an entry appended at timestep ta
 * (ta = 1 for the handle's) is live iff ta <= t and no timestep >= ta removed entries from its cell.  Every candidate
 * walks that sequence, skipping dead entries, with the warp-wide left fold of the list-order evaluation, so each
 * objective is the one the single calls compute on their compacted list.  Each scenario keeps its removal stamps on the
 * device (E x nx*ny ints, allocated for the call whether or not last_removed is asked for), and the bit planes are not
 * repacked inside the loop (nothing reads them).  Every other check is unchanged, in the same order.  Afterwards the
 * handle's ordered list is the single calls' (the ensembles leave it unchanged, as always); a CUDA failure inside the
 * loop of cov_run_horizon_points leaves the store unusable (cov_grid_info's calls fail until a setter rebuilds it),
 * because its list is not known then.  Dyadic stores run exactly as with the option at 0.  The automaton horizons
 * (cov_run_horizon_fire and its ensemble) refuse list-order stores whatever the option: after an automaton push the
 * list order becomes createPOI's, another replay. */
COV_API int cov_run_horizon(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                            int64_t n_iter, double granularity, uint64_t seed,
                            const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                            double *X_out, double *obj_out, int64_t *stats, double *step_ms);

/* The dynamic receding horizon (FullSimulation.run_simulation with environment_type = "dynamic"): cov_run_horizon
 * with an append step that opens every timestep, before step 1 (update_POI before rmvCoveredPOI, as the reference
 * orders them).  Arguments, outputs and errors are cov_run_horizon's, except that stats is T x 5: [winner k,
 * evaluations, solves with a feasible point, entries removed, entries appended].
 *
 * The store's envelope.  The plane set stays fixed inside the loop, so before anything is enqueued the call reads the
 * cell store (one download) and bounds every cell's multiplicity over the whole call, ignoring removals:
 *  - classes: the store's, then the new weights in order of first appearance in the schedule (cov_add_points'
 *    numbering; a store without entries starts afresh, as there).  More than 4: COV_ERR_LIMIT;
 *  - planes: for class k, bits 0 .. floor(log2(the largest bound of its cells)).  More than 8, or a bound over 255:
 *    COV_ERR_LIMIT;
 *  - area_exact of the store with n_entries replaced by n_entries plus every entry the call can add: 0 gives
 *    COV_ERR_STATE unless COV_OPT_LIST_ORDER_HORIZON is 1 (list-order stores, as for cov_run_horizon; never for the
 *    automaton);
 *  - cov_mads_solve_batch's limits on that plane set: COV_ERR_LIMIT.
 * An empty plane adds nothing to any count, so every objective, iterate and winner is the one the sequence of single
 * calls computes on its smaller plane sets; one rebuild at the end leaves the minimal plane set and the statistics.
 * Because removals are ignored, the checks are conservative: a call can be refused that the sequence of single calls
 * would accept (e.g. a cell whose bound passes 255 although a removal would have emptied it first).
 *
 * Afterwards the handle is exactly as the sequence of single calls leaves it (per timestep: the appends, then
 * cov_remove_covered, cov_set_params, cov_mads_solve_batch on the documented starts, the argmin and the evaluation):
 * cell store, cov_get_grid_info, cov_get_class_weights, the parameters of step T, the automaton's state and the
 * ordered point list.  The one exception: when the store empties completely inside the loop, cov_add_points would
 * restart its class numbering and this call does not (counts and objectives are the same).  A refused call changes
 * nothing: every check runs before the first enqueue.  A CUDA failure inside the loop leaves what was enqueued, the
 * store rebuilt, and the list order forgotten (createPOI's from then on).  T == 0 does nothing.
 *
 * cov_run_horizon_points: the reference's fire list (update_POI's push!).  Timestep t appends rows offsets[t-1] ..
 * offsets[t] - 1 of pts5 (reference 5-tuples, P = offsets[T] rows).  COV_ERR_INVALID: offsets NULL, offsets[0] != 0,
 * decreasing, or T > 2^31 - 1; pts5 NULL with P > 0; a NaN weight; entries of different weights on one cell, checked
 * against the cell's class at the call and across the whole schedule (conservatively).  COV_ERR_OFF_LATTICE: a point
 * that is not a cell centre.  stats[t][4] = offsets[t+1] - offsets[t].  last_removed (nullable, nx*ny ints indexed
 * (i-1) + nx*(j-1)): the last timestep of this call in which rmvCoveredPOI removed entries from the cell, 0 if none.
 * The ordered list afterwards is the single calls': an entry appended at timestep ta (ta = 1 for the entries listed
 * before the call) survives iff last_removed[cell] < ta; a store without a known list first fixes createPOI's order,
 * as cov_add_points does. */
COV_API int cov_run_horizon_points(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                                   int64_t n_iter, double granularity, uint64_t seed,
                                   const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                   const double *pts5, const int64_t *offsets,
                                   double *X_out, double *obj_out, int64_t *stats, double *step_ms,
                                   int *last_removed);

/* cov_run_horizon_fire: the device automaton (cov_fire_step with append = 1).  Timestep t runs fire_steps[t-1] >= 0
 * steps, numbered consecutively from first_step (the last is first_step + sum(fire_steps) - 1 <= 2^32 - 1), with the
 * direction probabilities cov_fire_step forms from wind_speed, wind_direction and prob_spread, keyed by fire_seed.
 * The envelope bounds a cell by its multiplicity plus 8 for every interior TREE cell (one ignition, at most one entry
 * per burning Moore neighbour).  stats[t][4]: the entries the timestep's steps pushed.  If any entry is pushed, the
 * list order is createPOI's afterwards, as after cov_fire_step.  COV_ERR_STATE: cov_fire_step's preconditions
 * (cov_fire_init called, one weight class of weight dx*dy); COV_ERR_INVALID: fire_steps NULL with T > 0 or negative,
 * first_step < 0 or the step range past 2^32 - 1. */
COV_API int cov_run_horizon_fire(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                                 int64_t n_iter, double granularity, uint64_t seed,
                                 const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                 const int64_t *fire_steps, double wind_speed, double wind_direction,
                                 double prob_spread, uint64_t fire_seed, int64_t first_step,
                                 double *X_out, double *obj_out, int64_t *stats, double *step_ms);

/* E independent static receding horizons in one call, on the device side by side: scenario e (0 <= e < E) is exactly
 * cov_run_horizon(x_starts + e * 3N, T, S, spread, n_iter, granularity, seed + e * T * S (mod 2^64), boxes, ...) run on
 * a private copy of the handle's current cell store and parameters.  Solve k of timestep t of scenario e is keyed by
 * seed + e * T * S + (t - 1) * S + k, so the scenarios' keys are disjoint and a scenario's results do not depend on E
 * or on the other scenarios.  Static environment only (no append step).  Every step of a timestep is one launch for
 * the whole ensemble.
 *
 * x_starts: E x 3N.  X_out: E x T x 3N; obj_out (nullable): E x T; stats (nullable): E x T x 4 with cov_run_horizon's
 * columns [winner k, evaluations, feasible solves, entries removed]; step_ms (nullable): T device times of the whole
 * ensemble per timestep; cells_out (nullable): E x nx*ny bytes, row e the multiplicities scenario e leaves (what
 * cov_get_grid_cells returns after the equivalent cov_run_horizon).
 *
 * The handle is not changed: unlike cov_run_horizon, which consumes the store, the cell store, cov_get_grid_info, the
 * class weights, the parameters (r_max and the previous swarm), the ordered point list and the automaton's state are
 * as before the call.  cov_launch_count counts the launches; cov_last_launch and the kernel timers are left unchanged.
 * Errors: cov_run_horizon's, in its order; COV_ERR_INVALID also for E < 1, E * S > 2^31 - 1 or E * T * S > 2^63 - 1;
 * a failed device allocation as the other calls report it.  T == 0 does nothing, and a refused or failed call changes
 * nothing on the handle. */
COV_API int cov_run_horizon_ensemble(cov_handle *h, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                     double spread, int64_t n_iter, double granularity, uint64_t seed,
                                     const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                     double *X_out, double *obj_out, int64_t *stats, double *step_ms,
                                     uint8_t *cells_out);

/* E independent dynamic receding horizons with the device automaton in one call, on the device side by side: scenario
 * e (0 <= e < E) is exactly cov_run_horizon_fire(x_starts + e * 3N, T, S, spread, n_iter, granularity, seed + e * T * S,
 * boxes, ..., fire_steps, winds[3e], winds[3e + 1], winds[3e + 2], fire_seed + e * fire_seed_stride, first_step, ...)
 * (arithmetic mod 2^64) run on a private copy of the handle's current cell store, parameters and automaton state.  Each
 * scenario has its own fire realisation (its fire seed), its own wind and its own starting swarm; fire_seed_stride = 1
 * gives independent realisations (Monte Carlo), 0 gives every scenario the same fire.  fire_steps (T values) and
 * first_step are shared by every scenario.  Every step of a timestep, each automaton step included, is one launch for
 * the whole ensemble.
 *
 * x_starts: E x 3N; winds: E x 3 doubles (wind_speed, wind_direction, prob_spread).  X_out: E x T x 3N; obj_out
 * (nullable): E x T; stats (nullable): E x T x 5 with cov_run_horizon_fire's columns [winner k, evaluations, feasible
 * solves, entries removed, entries appended]; step_ms (nullable): T device times of the whole ensemble per timestep;
 * cells_out (nullable): E x nx*ny bytes, the multiplicities each scenario leaves; states_out (nullable): E x nx*ny
 * bytes, the automaton state each scenario leaves, laid out as cov_fire_get_state returns it.
 *
 * Every scenario starts from the same store and state, so one envelope (cov_run_horizon_fire's) serves all of them.
 * The handle is not changed: the cell store, cov_get_grid_info, the class weights, the parameters, the ordered point
 * list, the automaton's state and its current buffer are as before the call, so the next cov_fire_step gives what it
 * would have given without it.  Errors: cov_run_horizon_fire's, in its order, with cov_run_horizon_ensemble's E checks
 * after cov_run_horizon's; COV_ERR_INVALID also for winds NULL with T > 0.  T == 0 does nothing, and a refused or
 * failed call changes nothing on the handle. */
COV_API int cov_run_horizon_fire_ensemble(cov_handle *h, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                          double spread, int64_t n_iter, double granularity, uint64_t seed,
                                          const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                          const int64_t *fire_steps, const double *winds, uint64_t fire_seed,
                                          uint64_t fire_seed_stride, int64_t first_step,
                                          double *X_out, double *obj_out, int64_t *stats, double *step_ms,
                                          uint8_t *cells_out, uint8_t *states_out);

/* E independent dynamic receding horizons over the reference's fire list in one call, on the device side by side, each
 * scenario with its own starting swarm and one of L fire schedules: scenario e (0 <= e < E) is exactly
 * cov_run_horizon_points(x_starts + e * 3N, T, S, spread, n_iter, granularity, seed + e * T * S (mod 2^64), boxes, ...,
 * schedule list_of[e], ...) run on a private copy of the handle's current cell store and parameters.  A schedule is a
 * forecast of the fire: what it appends to the current store, timestep by timestep.  L = 1 with list_of all zeros is
 * the Monte Carlo over starting swarms and keys.  Every step of a timestep is one launch for the whole ensemble.
 *
 * Schedules: the rows of the L schedules are concatenated in pts5 (reference 5-tuples); offsets holds L * T + 1
 * non-decreasing values from 0, and schedule l appends rows offsets[l * T + t - 1] .. offsets[l * T + t] - 1 at
 * timestep t.  list_of: E values in [0, L).
 *
 * x_starts: E x 3N.  X_out: E x T x 3N; obj_out (nullable): E x T; stats (nullable): E x T x 5 with
 * cov_run_horizon_points' columns (column 4 of scenario e counts its own schedule's rows); step_ms (nullable): T device
 * times of the whole ensemble per timestep; cells_out (nullable): E x nx*ny bytes, the multiplicities each scenario
 * leaves; last_removed (nullable): E x nx*ny ints, row e what cov_run_horizon_points returns for scenario e, from which
 * the caller can rebuild each scenario's point list with the rule documented there.
 *
 * Every scenario starts from the same store, so one envelope serves all of them: cov_run_horizon_points' with a cell's
 * bound the store's multiplicity plus the largest count any one schedule puts on it (a scenario holds only its own
 * schedule); the classes the store's, then the new weights in order of first appearance over the concatenated
 * schedules; mixed weights on one cell checked across all schedules; the entry count the store's plus the longest
 * schedule's.  Every schedule counts, whether a scenario uses it or not, so the checks are conservative.  A scenario's
 * single call may number the classes differently (a weight that schedule 2 brings first); counts and objectives do not
 * change, since the store is dyadic and classes are not returned.
 *
 * The handle is not changed: the cell store, cov_get_grid_info, the class weights, the parameters, the ordered point
 * list with its pending removals and the automaton's state are as before the call.  Errors: cov_run_horizon_points',
 * in its order, with cov_run_horizon_ensemble's E checks after cov_run_horizon's; COV_ERR_INVALID also for L < 1, L * T
 * + 1 past 2^63 - 1, list_of NULL with T > 0 or a value outside [0, L).  T == 0 does nothing, and a refused or failed
 * call changes nothing on the handle. */
COV_API int cov_run_horizon_points_ensemble(cov_handle *h, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                            double spread, int64_t n_iter, double granularity, uint64_t seed,
                                            const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                            const double *pts5, const int64_t *offsets, int64_t L,
                                            const int64_t *list_of, double *X_out, double *obj_out, int64_t *stats,
                                            double *step_ms, uint8_t *cells_out, int *last_removed);

/* Covered-cell mask of ONE candidate: nx*ny bytes, 1 where the cell is inside some disc (whether
 * or not it holds entries). Lets the host replay an ordered Float64 sum over a weighted list. */
COV_API int cov_covered_mask(cov_handle *h, const double *x, uint8_t *mask);

/* ---- continuous variant (SURVEY.md 8f-4): exact area of the union of the N discs of every candidate, by
 *      boundary integration in FP64 (Green's theorem; the reference ships only the pair primitives,
 *      src/Base_Functions.jl:230-355, and no driver, so this is an extension checked against closed forms and
 *      an independent restatement to 1e-9 relative, far inside north_star's 1e-5). No grid is involved.
 *      N <= 1024 (one warp per candidate up to 64 discs, one CTA per candidate above). Host buffers, synchronous. */
COV_API int cov_union_area_batch(cov_handle *h, const double *X, int64_t B, int64_t N, double *area);

/* ---- grid-free static objective (SURVEY.md 8f-4, the continuous limit of the static environment): the exact area
 *      A(x) = |(D_1 u ... u D_N) n Omega \ C| newly covered inside the domain, where Omega is the rectangle
 *      [x_lo, x_hi] x [y_lo, y_hi] (createPOI's [0, nx dx] x [0, ny dy]) and C the union of the discs already covered
 *      (what rmvCoveredPOI removed timestep after timestep).  As dx = dy -> 0 the grid objective's area term of the
 *      static environment converges to A(x).  Computed in FP64 by boundary integration (Green's theorem, DESIGN.md 11);
 *      no cell store is involved and the cell store is not touched: these calls need cov_set_region and
 *      cov_set_params only, and every other entry point behaves as before.
 *      Limits: N <= 64 discs per candidate, M <= 512 covered discs, and at most 2048 arcs of C's boundary inside
 *      Omega (COV_ERR_LIMIT beyond them; 40 timesteps x 5 UAVs are 200 discs). ------------------------------------- */

/* The domain rectangle and the discs already covered (the continuous rmvCoveredPOI).
 * covered_xyR: M discs as [x_1..x_M, y_1..y_M, R_1..R_M] (NULL when M == 0); discs of radius <= 0 cover nothing.
 * Replaces any earlier region; a failing call leaves the earlier region in place.  The arcs of C's boundary inside
 * Omega are computed here, once, on the device.  COV_ERR_INVALID: non-finite values, x_hi <= x_lo, y_hi <= y_lo or
 * M < 0. */
COV_API int cov_set_region(cov_handle *h, double x_lo, double y_lo, double x_hi, double y_hi,
                           const double *covered_xyR, int64_t M);

/* obj[b] = -A(x_b) + penalty_scale * sum_i |R_i - r_max_i| (same FP64 assembly order as the grid objective);
 * area[b] = A(x_b); feasible[b] as cov_eval_batch (the constraints of cov_set_params, fused). All nullable;
 * best_obj / best_idx both NULL or both given: the poll winner with cov_argmin's rule (smallest index among ties,
 * barrier != 0 skips infeasible candidates). Host buffers, synchronous. N <= 64.  A candidate's results have the same
 * bits whatever the batch it is part of.  COV_ERR_STATE without a region or parameters.  cov_last_kernel_ms gives
 * the device time of this call's evaluation kernel(s). */
COV_API int cov_eval_region_batch(cov_handle *h, const double *X, int64_t B, double *obj, double *area,
                                  uint8_t *feasible, int32_t barrier, double *best_obj, int64_t *best_idx);

/* cov_mads_solve_batch (same arguments, loop, direction stream, drop rules, stats and results) with the region
 * objective of cov_eval_region_batch as the function minimised, so every iterate can be replayed through
 * cov_eval_region_batch. No cell store needed. N <= 64. */
COV_API int cov_mads_solve_batch_region(cov_handle *h, const double *X0, int64_t S, int64_t n_iter,
                                        double granularity, uint64_t seed, double *X_out, double *obj_out,
                                        int64_t *stats);

/* The receding horizon on the region objective (FullSimulation.run_simulation_region): cov_run_horizon's loop with
 * the covered set in place of the cell store, all enqueued before ONE synchronise at the end.  Arguments are
 * cov_run_horizon's.  Needs cov_set_region and cov_set_params with prev_xyR (cons3 on); no cell store is touched.
 * Let C be the region's covered set (its M0 discs with R > 0) and cur = x_start.  For t = 1 .. T:
 *  1. cur's discs with R > 0 are appended to C in UAV order (FullSimulation's vstack(covered, swarm), filtered as
 *     cov_set_region filters), and the arcs of C's boundary inside the domain are recomputed as cov_set_region does;
 *  2.-6. cov_run_horizon's steps 2 to 6 (the r_max rule, cons3's previous swarm := cur, the S starts, the solves keyed
 *     seed + (t - 1) S + k, the winner), the solves minimising the region objective as cov_mads_solve_batch_region;
 *  7. obj_out[t-1] (nullable) = the region objective of cur without the barrier, on step t's C and r_max.
 * stats (nullable): T x 4 [winner k, evaluations summed over the S solves, solves that found a feasible point, arcs
 * K_t of C's boundary at step t (at most 2048)]; step_ms (nullable): T device times, as cov_run_horizon's.  Five kernel
 * launches per timestep (cov_launch_count).  Afterwards the region holds C with its M0 + appended discs and their
 * arcs, and the parameters are step T's (r_max, previous swarm), exactly as the sequence cov_set_region,
 * cov_set_params, cov_mads_solve_batch_region, cov_eval_region_batch leaves them, and every value above equals what
 * that sequence gives, bit for bit.  T == 0 does nothing.
 * Refused before anything is enqueued, changing nothing, in this order: COV_ERR_STATE without a region or parameters;
 * COV_ERR_LIMIT for N > 64; COV_ERR_STATE with cons3 off; COV_ERR_LIMIT when M0 + T N > 512 (discs with R <= 0 count,
 * since how many go is known on the device only); cov_run_horizon's COV_ERR_INVALID checks; COV_ERR_INVALID for a
 * non-finite value in x_start.
 * Found inside the loop: when C's boundary has more than 2048 arcs at step t, or a swarm holds a non-finite value,
 * every later step does nothing and the call returns COV_ERR_LIMIT (the arcs) or COV_ERR_INVALID (the value) with a
 * message naming t -- the timestep at which the sequence's cov_set_region fails with the same code.  The region and
 * the parameters are then as before the call (C is built in buffers of the call, the parameters copied back). */
COV_API int cov_run_horizon_region(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                                   int64_t n_iter, double granularity, uint64_t seed,
                                   const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                   double *X_out, double *obj_out, int64_t *stats, double *step_ms);

/* ---- streams, memory, timing (so hosts without a CUDA binding can keep data resident) ------ */
COV_API int cov_sync(cov_handle *h);
COV_API void *cov_stream(cov_handle *h);                 /* the handle's cudaStream_t */
COV_API int cov_set_stream(cov_handle *h, void *stream); /* adopt a caller-owned cudaStream_t (NULL: back to own) */
COV_API int cov_host_alloc(cov_handle *h, int64_t bytes, void **out); /* pinned host memory */
COV_API int cov_host_free(cov_handle *h, void *p);
COV_API int cov_device_alloc(cov_handle *h, int64_t bytes, void **out);
COV_API int cov_device_free(cov_handle *h, void *p);
COV_API int cov_memcpy_h2d(cov_handle *h, void *dst, const void *src, int64_t bytes); /* async on the stream */
COV_API int cov_memcpy_d2h(cov_handle *h, void *dst, const void *src, int64_t bytes); /* async on the stream */
/* Kernel launches issued by this handle since creation (evidence for bench.py's gpu_launches). */
COV_API int64_t cov_launch_count(const cov_handle *h);
/* Timeline of the last host-path call recorded under COV_OPT_TRACE: per slice the device times (ms since
 * the call's first copy was queued) of: H2D done, kernel start, kernel end, D2H done. Returns the number of
 * values available; copies at most cap of them. */
COV_API int64_t cov_get_trace(const cov_handle *h, double *ms, int64_t cap);
/* Device time of the last cov_eval_batch* coverage-kernel launch(es) in milliseconds, measured
 * with CUDA events on the handle's stream (synchronises). */
COV_API int cov_last_kernel_ms(cov_handle *h, double *ms);
/* Shape of the last coverage-kernel launch of this handle (diagnostics; which kernel COV_KERNEL_AUTO and
 * COV_KERNEL_SPAN resolved to). COV_ERR_STATE before the first launch. */
typedef struct cov_launch_info {
    int32_t kernel;         /* cov_kernel: SPAN = small-swarm kernel, SPAN_GENERAL = CTA per candidate, BRUTE, EXACT */
    int32_t grid, block;    /* CTAs, threads per CTA */
    int32_t smem_bytes;     /* dynamic shared memory per CTA */
    int32_t band_rows;      /* framebuffer rows per band (ny: a single band) */
    int32_t planes_in_smem; /* 1: bit planes staged in shared memory */
    /* the template instantiation that ran (ABI 2; names the ncu profile bench.py's issue roofline reads) */
    int32_t multi;          /* 1: several bit planes / weight classes / multiplicities */
    int32_t chunk;          /* small-swarm kernel: candidates per work unit; CTA kernel: co-resident CTAs per SM the
                               instantiation is compiled for (3 or 4); else 0 */
    int32_t max_warps;      /* small-swarm kernel: warps per CTA the instantiation allows (20 or 24); else 0 */
    int32_t plane_mode;     /* CTA kernel: COV_OPT_PLANE_MODE it resolved to (0 to 4); else -1 */
} cov_launch_info;
COV_API int cov_last_launch(const cov_handle *h, cov_launch_info *out);
/* Running totals over every coverage-kernel launch of this handle: summed device time (CUDA
 * events on the launching stream) and number of launches (synchronises). Both nullable. */
COV_API int cov_kernel_time_total(cov_handle *h, double *ms, int64_t *launches);

/* Candidates ~ the benchmark distribution of BASELINE.md generated on the device:
 * x, y ~ U(0, lx/ly), h ~ U(h_min, h_max), R = h * tan_half_fov, Philox4x32-10 keyed by
 * (seed, candidate index, uav index). dX: B x 3N doubles on the device. */
COV_API int cov_generate_candidates(cov_handle *h, double *dX, int64_t B, int64_t N, uint64_t seed,
                            int64_t first_index, double lx, double ly, double h_min, double h_max,
                            double tan_half_fov);

/* ---- several GPUs of one box: candidates sharded contiguously, grid replicated ------------- */
COV_API int cov_multi_create(const int *devices, int n, cov_multi **out);
COV_API void cov_multi_destroy(cov_multi *m);
COV_API const char *cov_multi_last_error(const cov_multi *m);
COV_API int cov_multi_size(const cov_multi *m);
COV_API cov_handle *cov_multi_handle(cov_multi *m, int k); /* borrow shard k's handle (set grid/params on each) */
COV_API int cov_multi_eval_batch(cov_multi *m, const double *X, int64_t B, double *obj, int64_t *count,
                         uint8_t *feasible);
/* cov_run_horizon_ensemble over the devices (without step_ms): contiguous shards of scenarios (ceil(E / G) each),
 * shard k from scenario b0 on with seed + b0 * T * S, so its results equal the single-device call's bit for bit.  Set
 * the same store and parameters on every shard's handle (cov_multi_handle). */
COV_API int cov_multi_run_horizon_ensemble(cov_multi *m, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                           double spread, int64_t n_iter, double granularity, uint64_t seed,
                                           const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                           double *X_out, double *obj_out, int64_t *stats, uint8_t *cells_out);
/* cov_run_horizon_fire_ensemble over the devices (without step_ms): contiguous shards of scenarios, shard k from
 * scenario b0 on with seed + b0 * T * S, fire_seed + b0 * fire_seed_stride and winds + 3 * b0, so its results equal the
 * single-device call's bit for bit.  Set the same store, parameters and automaton state on every shard's handle. */
COV_API int cov_multi_run_horizon_fire_ensemble(cov_multi *m, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                                double spread, int64_t n_iter, double granularity, uint64_t seed,
                                                const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                                const int64_t *fire_steps, const double *winds, uint64_t fire_seed,
                                                uint64_t fire_seed_stride, int64_t first_step,
                                                double *X_out, double *obj_out, int64_t *stats, uint8_t *cells_out,
                                                uint8_t *states_out);
/* cov_run_horizon_points_ensemble over the devices (without step_ms): contiguous shards of scenarios, shard k from
 * scenario b0 on with seed + b0 * T * S and list_of + b0 (every shard gets all of pts5 and offsets), so its results
 * equal the single-device call's bit for bit.  Set the same store and parameters on every shard's handle. */
COV_API int cov_multi_run_horizon_points_ensemble(cov_multi *m, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                                  double spread, int64_t n_iter, double granularity, uint64_t seed,
                                                  const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                                  const double *pts5, const int64_t *offsets, int64_t L,
                                                  const int64_t *list_of, double *X_out, double *obj_out,
                                                  int64_t *stats, uint8_t *cells_out, int *last_removed);
COV_API int cov_multi_argmin(cov_multi *m, const double *X, int64_t B, int32_t barrier, double *best_obj,
                     int64_t *best_idx);

/* ---- limits ---------------------------------------------------------------------------- */
typedef struct cov_limits {
    int64_t max_uavs;     /* N */
    int64_t max_nx, max_ny;
    int64_t max_planes;
    int64_t max_classes;
} cov_limits;
COV_API void cov_get_limits(cov_limits *out);

/* T(R): the smallest double t with sqrt(t) >= R, computed by the same closed form the kernels
 * use (exposed so the tests can check it against the definition). */
COV_API double cov_threshold(double R);

#ifdef __cplusplus
}
#endif
#endif /* COVERAGE_CUDA_H */
