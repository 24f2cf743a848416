// cov_device.cuh -- arithmetic shared by every coverage kernel and by the host side.
//
// The reference predicate (src/AreaCoverageCalculation.jl:70, /root/reference) is
//     sqrt((px - cx)^2 + (py - cy)^2) < R          Float64, strict <, no FMA.
// Correctly rounded sqrt is monotone, so for each R there is one double T(R) with
//     sqrt(s) < R  <=>  s < T(R)            for every double s >= 0,
// namely T(R) = the smallest double strictly above m^2, m = the midpoint between R and the
// double just below it (m^2 is never a double: m has an odd 54/55-bit significand).  The kernels
// therefore evaluate  s = fl(fl(dx*dx) + fl(dy*dy)) < T  with the individually rounded
// __dsub_rn/__dmul_rn/__dadd_rn (which nvcc never contracts into FMA) and never take a sqrt per
// test.  cov_threshold() below is that closed form; tests check it against the definition.
#pragma once
#include <cstdint>
#include <cmath>

#if defined(__CUDACC__)
#define COV_HD __host__ __device__ __forceinline__
#else
#define COV_HD inline
#endif

namespace cov {

COV_HD uint64_t dbl_bits(double v)
{
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t b;
    __builtin_memcpy(&b, &v, 8);
    return b;
#endif
}
COV_HD double bits_dbl(uint64_t b)
{
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)b);
#else
    double v;
    __builtin_memcpy(&v, &b, 8);
    return v;
#endif
}

// Slow definition-following form: used outside the closed form's exponent window.
COV_HD double threshold_by_search(double R)
{
    double t = R * R;
    if (isinf(t)) {
        t = 1.7976931348623157e308;
        if (sqrt(t) < R) return bits_dbl(0x7ff0000000000000ull);
    }
    while (t > 0 && sqrt(t) >= R) t = bits_dbl(dbl_bits(t) - 1);
    while (sqrt(t) < R) t = bits_dbl(dbl_bits(t) + 1);
    return t;
}

// T(R) = min { t double : sqrt_rn(t) >= R }.  R <= 0 or NaN: 0 (no s >= 0 is below it, matching
// `sqrt(s) < R` being false); R = +Inf: +Inf (every finite s is covered).
COV_HD double threshold(double R)
{
    if (!(R > 0)) return 0.0;
    const uint64_t b = dbl_bits(R);
    const int e = (int)((b >> 52) & 0x7ff);
    if (e == 0x7ff) return R; // +Inf
    if (e < 1023 - 400 || e > 1023 + 400) return threshold_by_search(R);
    const uint64_t frac = b & 0x000fffffffffffffull;
    const uint64_t k = frac | 0x0010000000000000ull; // R = k * 2^(e-1075)
    // midpoint m = n * 2^sc between R and its predecessor
    uint64_t n;
    int sc;
    if (frac != 0) {
        n = 2 * k - 1;
        sc = e - 1075 - 1;
    } else { // R is a power of two: the gap below is half as wide
        n = 4 * k - 1;
        sc = e - 1075 - 2;
    }
    // A = n^2 as 128 bits
#if defined(__CUDA_ARCH__)
    const uint64_t hi = __umul64hi(n, n);
    const uint64_t lo = n * n;
    const int nb = 128 - __clzll((long long)hi);
#else
    const unsigned __int128 A = (unsigned __int128)n * n;
    const uint64_t hi = (uint64_t)(A >> 64);
    const uint64_t lo = (uint64_t)A;
    const int nb = 128 - __builtin_clzll(hi);
#endif
    const int shift = nb - 53; // 53..55
    const uint64_t t = (hi << (64 - shift)) | (lo >> shift);
    // A is odd and shift > 0, so the discarded part is non-zero: round up unconditionally.
    const uint64_t t1 = t + 1; // in (2^52, 2^53]
    const int q = 2 * sc + shift;
    const uint64_t eb = (uint64_t)(q + 1075);
    // a carry out of the significand (t1 == 2^53) lands in the exponent field by itself
    return bits_dbl((eb << 52) + (t1 - 0x0010000000000000ull));
}

// G(d): the double with  sqrt(s) > d  <=>  s >= G(d)   (cons3's `sqrt(...) > d_lim[i]`,
// src/TDM_Constraints.jl:67).  sqrt(s) is a double, so sqrt(s) > d <=> !(sqrt(s) < next(d))
// <=> s >= T(next(d)).  d NaN or +Inf: nothing violates (NaN: s >= NaN is false for every s,
// like `> NaN`); d < 0: every non-NaN s violates (s >= 0).
COV_HD double threshold_ge(double d)
{
    if (d != d || (isinf(d) && d > 0)) return bits_dbl(0x7ff8000000000000ull);
    if (d < 0) return 0.0;
    if (d == 0) d = 0.0; // -0.0 -> +0.0 so that bits+1 is the next double up
    return threshold(bits_dbl(dbl_bits(d) + 1));
}

#if defined(__CUDACC__)
// Cell-centre coordinate exactly as the reference forms it: fl(fl(i*d) - d/2)
// (src/AreaCoverageCalculation.jl:16).  i is an exact small integer.
__device__ __forceinline__ double cell_centre(int i, double d, double half_d)
{
    // (double)i without a conversion instruction: 2^52 + i has i in its low significand bits.
    const double di = __hiloint2double(0x43300000, i) - 4503599627370496.0;
    return __dsub_rn(__dmul_rn(di, d), half_d);
}

// s = fl(fl(ddx^2) + fl(ddy^2)) with ddx = fl(px - cx): the reference's radicand.
__device__ __forceinline__ double radicand(double px, double py, double cx, double cy)
{
    const double ddx = __dsub_rn(px, cx);
    const double ddy = __dsub_rn(py, cy);
    return __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
}

// Philox4x32-10 (Salmon et al., SC'11): counter (c0..c3), key (k0, k1) -> 4 words.  The stream of the candidate
// generator, the fire automaton and the device MADS solver's directions; synth._philox restates it in NumPy.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4])
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0;
        c1 = n1;
        c2 = n2;
        c3 = n3;
        k0 += W0;
        k1 += W1;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}
#endif

} // namespace cov
