// sinf_glibc.h -- f32 sine with glibc's results, usable on host and device.
//
// knaster's SinNumeric / PolyBlep call f32::sin (osc.rs:264, polyblep.rs:244), which is the
// platform libm's sinf (num-traits `std`, knaster_primitives/Cargo.toml:12,19): a third-party
// dependency outside /root/reference.  Pinned version here: glibc 2.39 (the image's libm; the
// algorithm is the ARM optimized-routines sinf that glibc adopted in 2.28: sysdeps/ieee754/flt-32/
// s_sinf.c + s_sincosf.h + s_sincosf_data.c).  This is a restatement of that published algorithm:
// fast range reduction by pi/2 in f64 and a degree-7 sine / degree-8 cosine polynomial in f64,
// rounded once to f32; for |y| >= 120 glibc's reduce_large (y times 4/pi in integer arithmetic).  cosf is restated as well.
// tests/test_host_plan.py::test_sinf_restatement_matches_libm checks the sine bit-for-bit against the libm the oracle
// links, and tests/test_sinf_exhaustive.py (tools/sinf_exhaustive.cpp) both functions over EVERY float; the device
// instantiation is checked over every float by tests/test_gpu_devmath.py (tools/devmath_exhaustive.cu).
// The fused multiply-adds are glibc's too: on a CPU with FMA its ifunc selects __sinf_fma, the same source
// compiled with contraction (12 of the 2.2e9 results differ from the un-fused build).
//
// Why it matters: an FM carrier integrates its modulator's output, so 1-ulp differences between the
// device sine and libm's would random-walk the carrier phase past the 1e-5 budget within seconds.
#pragma once
#include <stdint.h>
#include <string.h>
#if defined(__CUDACC__)
#define KN_SINF_HD __host__ __device__ __forceinline__
// glibc's large-argument reduction is a call on the device (as the f64 sin / cos slow-path reduction was), with its quadrant
// returned through memory as in glibc; the rest is inline
#define KN_SINF_CALL __host__ __device__ inline __noinline__
#else
#include <cmath>
#define KN_SINF_HD inline
#define KN_SINF_CALL inline
#endif

namespace kgpu {

KN_SINF_HD double kn_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
    return __fma_rn(a, b, c);
#else
    // a true fused multiply-add, as in glibc's __sinf_fma (the variant its ifunc picks on every CPU with FMA): over ALL floats
    // |y| < 120 the un-fused form differs from it in 12 results (tools/sinf_exhaustive.cpp)
    return __builtin_fma(a, b, c);
#endif
}

// glibc's sinf for |y| < 120 (its reduce_fast domain).
//
// glibc branches three ways (|y| < 2^-12: y itself; |y| < pi/4: sine polynomial without reduction;
// else reduce and pick the sine or cosine polynomial by the quadrant's parity).  On a GPU those
// branches diverge in every warp, so the same arithmetic is laid out straight-line here:
//   * for |y| < pi/4 the reduction yields n = 0 and leaves x untouched, so the general path IS the
//     small-argument path;
//   * both polynomials are evaluated (they share x2) and one is selected -- a diverged warp would
//     execute both anyway;
//   * |y| < 2^-12 still returns y (select), which also keeps the sign of -0.
// Every f64 operation is the one glibc performs for the selected path, in the same order.
KN_SINF_HD float kn_sinf_glibc_inrange(float y) { // requires |y| < 120
    const double HPI_INV = 0x1.45F306DC9C883p+23; // 2^24 / (pi/2)
    const double HPI = 0x1.921FB54442D18p0;       // pi/2
    const double C0 = 0x1p0, C1 = -0x1.ffffffd0c621cp-2, C2 = 0x1.55553e1068f19p-5, C3 = -0x1.6c087e89a359dp-10,
                 C4 = 0x1.99343027bf8c3p-16;
    const double S1 = -0x1.555545995a603p-3, S2 = 0x1.1107605230bc4p-7, S3 = -0x1.994eb3774cf24p-13;
    uint32_t iy;
#if defined(__CUDA_ARCH__)
    iy = __float_as_uint(y);
#else
    memcpy(&iy, &y, 4);
#endif
    const uint32_t top = (iy >> 20) & 0x7ff;          // abstop12
    double x = (double)y;
    // reduce_fast.  glibc skips it for |y| < pi/4 (abstop12 < 0x3f4); there |r| < 2^23, so n = 0 and
    // fma(-0, HPI, x) == x: running it unconditionally changes nothing
    const double r = x * HPI_INV;
#if defined(__CUDA_ARCH__)
    const int n = (__double2int_rz(r) + 0x800000) >> 24;
#else
    const int n = ((int32_t)r + 0x800000) >> 24;
#endif
    x = kn_fma(-(double)n, HPI, x);
    const double x2 = x * x;
    // sine polynomial (odd in x); sign table {1,-1,-1,1}[n & 3]
    const double x3 = x * x2, s1 = kn_fma(x2, S3, S2), x7 = x3 * x2, sp = kn_fma(x3, S1, x);
    const double rs = kn_fma(x7, s1, sp);
    // cosine polynomial (even in x); __sincosf_table[1] (negated coefficients) when n & 2
    const double x4 = x2 * x2, c2 = kn_fma(x2, C4, C3), c1 = kn_fma(x2, C1, C0), x6 = x4 * x2, cp = kn_fma(x4, C2, c1);
    double rc = kn_fma(x6, c2, cp);
    double rs_ = rs;
#if defined(__CUDA_ARCH__)
    // keep both polynomials unconditional: nvcc would otherwise sink each into a branch on the
    // quadrant's parity, and a diverging branch per sine ends the basic block (no overlap of the
    // frames' f64 chains)
    asm volatile("" : "+d"(rs_), "+d"(rc));
#endif
    const bool odd = (n & 1) != 0;
    const bool neg = odd ? (n & 2) != 0 : ((n + 1) & 2) != 0;
    double res = odd ? rc : rs_;
    res = neg ? -res : res;
    return top < 0x398 ? y : (float)res;              // |y| < 2^-12: sin(y) = y to f32 precision
}

// The same function in the form the FM kernels use: fewer instructions on the pipes that bound render_fm2 (DESIGN.md section 3).
//   * n comes from the "magic number" rounding of x * 2/pi (t = u + 1.5 * 2^52 leaves RN(u) in t's low word and t - 1.5 * 2^52 is n as a
//     double): two FP64 additions instead of F2I + shift + add + I2F (two quarter-rate conversions).  glibc's n is
//     floor((trunc(x * 2^24 * 2/pi) + 2^23) / 2^24), round-half-up of the same product for x >= 0: the two disagree for five negative
//     floats in the whole domain (arguments a hair beyond an odd multiple of pi/4), and there both polynomials round to the same f32;
//   * the sign is bit 1 of n for both parities ({+sin, +cos, -sin, -cos}) and is applied to the rounded f32;
//   * no special case below 2^-12: the sine polynomial rounds to y there anyway.
// tools/sinf_exhaustive.cpp compares it with libm's sinf for EVERY float |y| < 120 (2.2e9 arguments, 5 s on 8 cores): bit-identical
// everywhere except sin(-0.0), which is +0.0 here (an oscillator's phase argument is never -0: x + (-x) rounds to +0).
// Every f64 operation of the selected polynomial is still glibc's, in glibc's order.
KN_SINF_HD float kn_sinf_glibc_lean(float y) { // requires |y| < 120
    const double TWO_OVER_PI = 0x1.45F306DC9C883p-1, MAGIC = 0x1.8p52;
    const double HPI = 0x1.921FB54442D18p0;
    const double C0 = 0x1p0, C1 = -0x1.ffffffd0c621cp-2, C2 = 0x1.55553e1068f19p-5, C3 = -0x1.6c087e89a359dp-10,
                 C4 = 0x1.99343027bf8c3p-16;
    const double S1 = -0x1.555545995a603p-3, S2 = 0x1.1107605230bc4p-7, S3 = -0x1.994eb3774cf24p-13;
    double x = (double)y;
#if defined(__CUDA_ARCH__)
    const double t = __dadd_rn(__dmul_rn(x, TWO_OVER_PI), MAGIC); // two roundings (the product, then the sum): never contracted
    const double nd = __dadd_rn(t, -MAGIC);
    const uint32_t n = (uint32_t)__double2loint(t);
#else
    volatile double u = x * TWO_OVER_PI;               // (volatile: keeps a host compiler from fusing the product into the sum)
    const double t = u + MAGIC;
    const double nd = t - MAGIC;
    uint64_t tb;
    memcpy(&tb, &t, 8);
    const uint32_t n = (uint32_t)tb;
#endif
    x = kn_fma(-nd, HPI, x);
    const double x2 = x * x;
    const double x3 = x * x2, s1 = kn_fma(x2, S3, S2), x7 = x3 * x2, sp = kn_fma(x3, S1, x);
    double rs = kn_fma(x7, s1, sp);
    const double x4 = x2 * x2, c2 = kn_fma(x2, C4, C3), c1 = kn_fma(x2, C1, C0), x6 = x4 * x2, cp = kn_fma(x4, C2, c1);
    double rc = kn_fma(x6, c2, cp);
#if defined(__CUDA_ARCH__)
    asm volatile("" : "+d"(rs), "+d"(rc));             // both polynomials stay unconditional (see kn_sinf_glibc_inrange)
#endif
    const float f = (float)((n & 1u) ? rc : rs);
    uint32_t fb;
#if defined(__CUDA_ARCH__)
    fb = __float_as_uint(f) ^ ((n << 30) & 0x80000000u);
    return __uint_as_float(fb);
#else
    memcpy(&fb, &f, 4);
    fb ^= (n << 30) & 0x80000000u;
    float o;
    memcpy(&o, &fb, 4);
    return o;
#endif
}

#if defined(__CUDACC__)
// N independent sines, written stage by stage (every stage over all N arguments before the next one): the order a software-pipelined
// schedule wants; the operations per argument are kn_sinf_glibc_lean's.
template <int N> __device__ __forceinline__ void kn_sinf_glibc_lean_n(const float (&y)[N], float (&o)[N]) {
    const double TWO_OVER_PI = 0x1.45F306DC9C883p-1, MAGIC = 0x1.8p52;
    const double HPI = 0x1.921FB54442D18p0;
    const double C0 = 0x1p0, C1 = -0x1.ffffffd0c621cp-2, C2 = 0x1.55553e1068f19p-5, C3 = -0x1.6c087e89a359dp-10,
                 C4 = 0x1.99343027bf8c3p-16;
    const double S1 = -0x1.555545995a603p-3, S2 = 0x1.1107605230bc4p-7, S3 = -0x1.994eb3774cf24p-13;
    double x[N], t[N], x2[N], a[N], b[N], c[N], d[N];
    uint32_t n[N];
#pragma unroll
    for (int i = 0; i < N; i++) x[i] = (double)y[i];
#pragma unroll
    for (int i = 0; i < N; i++) t[i] = __dmul_rn(x[i], TWO_OVER_PI);
#pragma unroll
    for (int i = 0; i < N; i++) t[i] = __dadd_rn(t[i], MAGIC);
#pragma unroll
    for (int i = 0; i < N; i++) {
        n[i] = (uint32_t)__double2loint(t[i]);
        t[i] = __dadd_rn(t[i], -MAGIC);
    }
#pragma unroll
    for (int i = 0; i < N; i++) x[i] = __fma_rn(-t[i], HPI, x[i]);
#pragma unroll
    for (int i = 0; i < N; i++) x2[i] = __dmul_rn(x[i], x[i]);
#pragma unroll
    for (int i = 0; i < N; i++) {
        a[i] = __dmul_rn(x[i], x2[i]);            // x3
        b[i] = __fma_rn(x2[i], S3, S2);           // s1
        c[i] = __dmul_rn(x2[i], x2[i]);           // x4
        d[i] = __fma_rn(x2[i], C4, C3);           // c2
        t[i] = __fma_rn(x2[i], C1, C0);           // c1
    }
#pragma unroll
    for (int i = 0; i < N; i++) {
        x[i] = __fma_rn(a[i], S1, x[i]);          // sp
        a[i] = __dmul_rn(a[i], x2[i]);            // x7
        t[i] = __fma_rn(c[i], C2, t[i]);          // cp
        c[i] = __dmul_rn(c[i], x2[i]);            // x6
    }
#pragma unroll
    for (int i = 0; i < N; i++) {
        a[i] = __fma_rn(a[i], b[i], x[i]);        // rs
        c[i] = __fma_rn(c[i], d[i], t[i]);        // rc
    }
#pragma unroll
    for (int i = 0; i < N; i++) {
        asm volatile("" : "+d"(a[i]), "+d"(c[i]));
        const float f = (float)((n[i] & 1u) ? c[i] : a[i]);
        o[i] = __uint_as_float(__float_as_uint(f) ^ ((n[i] << 30) & 0x80000000u));
    }
}
#endif

// ---- the rest of glibc's sinf and all of its cosf (s_sinf.c, s_cosf.c) -----------------------------------------------------

KN_SINF_HD uint32_t kn_f32_bits(float y) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(y);
#else
    uint32_t b;
    memcpy(&b, &y, 4);
    return b;
#endif
}

// sinf_poly: n even -> the sine polynomial, n odd -> the cosine polynomial, its coefficients negated when neg
// (__sincosf_table[1]); fused operations as in __sinf_fma
KN_SINF_HD float kn_sincosf_poly(double x, double x2, bool neg, int n) {
    const double S1 = -0x1.555545995a603p-3, S2 = 0x1.1107605230bc4p-7, S3 = -0x1.994eb3774cf24p-13;
    if ((n & 1) == 0) {
        const double x3 = x * x2, s1 = kn_fma(x2, S3, S2), x7 = x3 * x2, s = kn_fma(x3, S1, x);
        return (float)kn_fma(x7, s1, s);
    }
    const double g = neg ? -1.0 : 1.0; // sign changes are exact: the negated table's products and sums are the negated ones
    const double C0 = g * 0x1p0, C1 = g * -0x1.ffffffd0c621cp-2, C2 = g * 0x1.55553e1068f19p-5, C3 = g * -0x1.6c087e89a359dp-10,
                 C4 = g * 0x1.99343027bf8c3p-16;
    const double x4 = x2 * x2, c2 = kn_fma(x2, C4, C3), c1 = kn_fma(x2, C1, C0), x6 = x4 * x2, c = kn_fma(x4, C2, c1);
    return (float)kn_fma(x6, c2, c);
}

// glibc's __inv_pio4: 4/pi in overlapping 32-bit windows, one byte apart.  Constant memory on the device (a local array
// would be stored to every kernel's stack at every call and cost the interpreter registers), a plain array on the host.
#define KN_INV_PIO4                                                                                                              \
    {0xa2,       0xa2f9,     0xa2f983,   0xa2f9836e, 0xf9836e4e, 0x836e4e44, 0x6e4e4415, 0x4e441529,                             \
     0x441529fc, 0x1529fc27, 0x29fc2757, 0xfc2757d1, 0x2757d1f5, 0x57d1f534, 0xd1f534dd, 0xf534ddc0,                             \
     0x34ddc0db, 0xddc0db62, 0xc0db6295, 0xdb629599, 0x6295993c, 0x95993c43, 0x993c4390, 0x3c439041}
#if defined(__CUDACC__)
static __constant__ const uint32_t kn_inv_pio4_dev[24] = KN_INV_PIO4;
#endif
#if !defined(__CUDA_ARCH__)
static const uint32_t kn_inv_pio4_host[24] = KN_INV_PIO4;
#endif
#undef KN_INV_PIO4

// glibc's reduce_large for 120 <= |y| < inf: y * 4/pi from 96 bits of 4/pi chosen by y's exponent, in integer arithmetic;
// returns the reduced argument in radians and the quadrant in *np
KN_SINF_CALL double kn_sincosf_reduce_large(uint32_t xi, int *np) {
#if defined(__CUDA_ARCH__)
    const uint32_t *arr = &kn_inv_pio4_dev[(xi >> 26) & 15];
#else
    const uint32_t *arr = &kn_inv_pio4_host[(xi >> 26) & 15];
#endif
    const double PI63 = 0x1.921FB54442D18p-62; // pi / 2^62
    const int shift = (xi >> 23) & 7;
    xi = ((xi & 0xffffff) | 0x800000) << shift;
    uint64_t res0 = xi * arr[0];               // 32-bit product: only its low word is kept
    const uint64_t res1 = (uint64_t)xi * arr[4], res2 = (uint64_t)xi * arr[8];
    res0 = (res2 >> 32) | (res0 << 32);
    res0 += res1;
    const uint64_t n = (res0 + (1ULL << 61)) >> 62;
    res0 -= n << 62;
    *np = (int)n;
    return (double)(int64_t)res0 * PI63;
}

// glibc's sinf (want_cos = false) or cosf (want_cos = true) for |y| >= 120: the large-argument path, whose sign table includes
// y's sign.  +-inf and NaN give NaN (__math_invalidf).
KN_SINF_HD float kn_sincosf_glibc_large(float y, bool want_cos) {
    const uint32_t xi = kn_f32_bits(y);
    if (((xi >> 20) & 0x7ff) >= 0x7f8) return y - y;
    int n;
    const double x = kn_sincosf_reduce_large(xi, &n);
    const int q = (n + (int)(xi >> 31)) & 3;
    const double s = (q == 1 || q == 2) ? -1.0 : 1.0; // sign[] = {1, -1, -1, 1}
    return kn_sincosf_poly(x * s, x * x, (q & 2) != 0, want_cos ? n ^ 1 : n);
}

// glibc's sinf for every float: bit-identical to it (tools/sinf_exhaustive.cpp checks all 2^32 arguments)
KN_SINF_HD float kn_sinf_glibc(float y) {
    return ((kn_f32_bits(y) >> 20) & 0x7ff) < 0x42f ? kn_sinf_glibc_inrange(y) : kn_sincosf_glibc_large(y, false); // abstop12(120.0f)
}

// glibc's cosf for |y| < 120, straight-line like kn_sinf_glibc_inrange: for |y| < pi/4 the reduction gives n = 0 and leaves x
// as it is, which is glibc's unreduced path; below 2^-12 the polynomial rounds to 1, glibc's special case
KN_SINF_HD float kn_cosf_glibc_inrange(float y) { // requires |y| < 120
    double x = (double)y;
    const double r = x * 0x1.45F306DC9C883p+23;
#if defined(__CUDA_ARCH__)
    const int n = (__double2int_rz(r) + 0x800000) >> 24;
#else
    const int n = ((int32_t)r + 0x800000) >> 24;
#endif
    x = kn_fma(-(double)n, 0x1.921FB54442D18p0, x);
    const int q = n & 3;
    const double s = (q == 1 || q == 2) ? -1.0 : 1.0;
    return kn_sincosf_poly(x * s, x * x, (q & 2) != 0, n ^ 1);
}

// glibc's cosf for every float
KN_SINF_HD float kn_cosf_glibc(float y) {
    return ((kn_f32_bits(y) >> 20) & 0x7ff) < 0x42f ? kn_cosf_glibc_inrange(y) : kn_sincosf_glibc_large(y, true);
}

} // namespace kgpu
