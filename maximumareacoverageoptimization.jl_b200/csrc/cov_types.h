// cov_types.h -- plain structs passed by value from the host side of libcoverage_cuda to its
// kernels (kernel parameter space; no device-side indirection for the small stuff).
#pragma once
#include <cstdint>

namespace cov {

constexpr int kMaxPlanes = 8;   // bit planes (weight class x multiplicity bit)
constexpr int kMaxClasses = 4;  // distinct per-entry weights
constexpr int kMaxUavs = 1024;  // N
constexpr int kMaxDim = 32768;  // nx, ny (row indices travel as 16-bit pairs, see DiscParam)

// The cell store as the kernels see it.
// Cell (i, j), 1-based, centre (i*dx - dx/2, j*dy - dy/2).  A plane is ny rows of `stride` words
// (stride = words per row rounded up to an ODD count, so that 32 lanes working on 32
// consecutive rows at the same word index hit 32 different shared-memory banks); bit b of word w
// of row j-1 is cell i = 32*w + b + 1.  plane_words = ny*stride rounded up to a multiple of 4 so
// a plane is one 16-byte-granular bulk copy.
struct GridDesc {
    int nx, ny;
    int wpr;          // words per row actually holding cells
    int stride;       // padded words per row
    int plane_words;  // words per plane (multiple of 4)
    int n_planes;
    int n_classes;
    int lattice_f32_exact;  // 1: every cell-centre coordinate is exactly representable in FP32
    double dx, dy, hdx, hdy;         // hd = d/2
    double inv_dx, inv_dy;
    float dxf, dyf, hdxf, hdyf, inv_dxf, inv_dyf;
    float extent;                    // max(nx*dx, ny*dy): magnitude bound for the FP32 error band
    float k_ca;                      // 0.75 / dx, rounded up: (band delta) -> (zone half-width * chord), see fast_span
    int plane_class[kMaxPlanes];
    int plane_mult[kMaxPlanes];      // 1, 2, 4, ... entries per set bit
    double class_weight[kMaxClasses];
    const uint32_t *planes;          // device: n_planes * plane_words
    // Plane 0 once more for the paint-then-sweep mode of the CTA kernel (single-plane stores only, else null):
    // rows of `qstride` words, qstride even and qstride/2 odd (rows are 8-byte aligned, 16 consecutive rows start
    // in 16 different bank pairs), and word w of grid row j stored at w ^ (((j-1) >> 4) & 1): 32 lanes on 32
    // consecutive rows at one column hit 32 different banks although the rows are aligned.
    int qstride;
    const uint32_t *planes_q;        // device: ny * qstride words (+ padding), or null
    // The point list in the reference's own order (cell index (i-1) + nx*(j-1) and weight class per entry), for the
    // ordered kernel; null until a launch needs it.
    const int *ent_cell;
    const unsigned char *ent_cls;
    long long n_ent;
};

// Captured variables of the reference's closures (createObjective, create_cons3, cons7, cons8).
struct ObjParams {
    int N;
    int use_cons3, use_cons7, use_cons8;
    int prog_which;         // progressive output: 0 = sum over every UAV (cons1_progressive), k >= 1 = UAV k only
                            // (cons2_progressive: k = 2, cons3_progressive: k = 3; src/TDM_Constraints.jl:182-221)
    double penalty_scale;   // 1e5
    double tan_half_fov;
    double cons7_R;         // fl(19 * tan_half_fov)
    double sep_T;           // T(sep_min): sqrt(s) < sep  <=>  s < sep_T
    const double *r_max;    // device, N
    const double *prev_x;   // device, N   (cons3)
    const double *prev_y;   // device, N
    const double *prev_z;   // device, N: fl(prev_R / tan_half_fov)
    const double *cons3_G;  // device, N: sqrt(s) > d_lim[i]  <=>  s >= cons3_G[i]
};

// The grid-free static objective's region (cov_set_region): the domain rectangle and the covered discs C, with the
// arcs of C's boundary that lie inside the domain (each a piece [a, b] of covered circle m, 0 <= a < b <= 2 pi).
struct RegionArc {
    double a, b;
    int m, pad;
};
struct RegionDesc {
    double x_lo, y_lo, x_hi, y_hi;
    int M, K;               // covered discs (radius > 0), arcs
    const double *discs;    // device: 3M doubles [x_1..x_M, y_1..y_M, R_1..R_M]
    const RegionArc *arcs;  // device: K
};

struct EvalOut {
    double *obj;            // B
    long long *count;       // B or null
    unsigned char *feasible; // B or null
    long long *class_count; // B * n_classes or null
    double *progressive;    // B or null
    // device-resident mirrors of obj / feasible (both or neither; null as a rule): what the winner reduction of
    // cov_eval_batch_best reads when the results themselves go straight to pinned host memory
    double *obj_mirror;
    unsigned char *feasible_mirror;
};

} // namespace cov
