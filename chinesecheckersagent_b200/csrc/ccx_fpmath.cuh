/* ccx_fpmath.cuh — float64 log / exp whose every bit is fixed, for the Gumbel search (ccx_mcts.cu) and its CPU restatement.
 *
 * Device log() / exp() and the C library's differ in their last bits, and a search that takes arg-maxes over softmaxes
 * amplifies a one-ulp difference into a different tree.  These two functions are built only from IEEE float64 + - x /
 * (round to nearest, no contraction: explicit __d*_rn on the device, -ffp-contract=off on the host), integer bit
 * operations and fixed polynomials, so the device and any C compiler produce the same bits.  The algorithms and
 * coefficients are fdlibm's e_log.c and e_exp.c (error below one ulp).
 *
 * C-compatible: a C11 translation unit can include this header as well as a CUDA one. */
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define FM_HD __host__ __device__ __forceinline__
#else
#include <string.h>
#define FM_HD static inline
#endif

#if defined(__CUDA_ARCH__)
#define FM_ADD(a, b) __dadd_rn((a), (b))
#define FM_SUB(a, b) __dsub_rn((a), (b))
#define FM_MUL(a, b) __dmul_rn((a), (b))
#define FM_DIV(a, b) __ddiv_rn((a), (b))
#else
#define FM_ADD(a, b) ((a) + (b))
#define FM_SUB(a, b) ((a) - (b))
#define FM_MUL(a, b) ((a) * (b))
#define FM_DIV(a, b) ((a) / (b))
#endif

FM_HD uint64_t fm_bits(double x)
{
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(x);
#else
    uint64_t u; memcpy(&u, &x, 8); return u;
#endif
}

FM_HD double fm_from_bits(uint64_t u)
{
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double x; memcpy(&x, &u, 8); return x;
#endif
}

/* natural logarithm of a positive finite x (normal or subnormal); 0 -> -inf.  fdlibm e_log.c: x = 2^k (1 + f) with
 * 1 + f in [sqrt(2)/2, sqrt(2)), s = f / (2 + f), log(1 + f) = f - (hfsq - s (hfsq + R(s^2))) */
FM_HD double fm_log(double x)
{
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, two54 = 1.80143985094819840000e+16;
    const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                 Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                 Lg7 = 1.479819860511658591e-01;
    uint64_t u = fm_bits(x);
    int k = 0;
    if (x == 0.0) return fm_from_bits(0xFFF0000000000000ULL);
    if ((u >> 52) == 0) {                                    /* subnormal: scale into the normal range */
        x = FM_MUL(x, two54);
        u = fm_bits(x);
        k = -54;
    }
    int32_t hx = (int32_t)(u >> 32);
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    const int32_t i = (hx + 0x95f64) & 0x100000;             /* 1 + f >= sqrt(2): halve it */
    x = fm_from_bits(((uint64_t)(uint32_t)(hx | (i ^ 0x3ff00000)) << 32) | (u & 0xFFFFFFFFULL));
    k += i >> 20;
    const double f = FM_SUB(x, 1.0);
    const double s = FM_DIV(f, FM_ADD(2.0, f));
    const double dk = (double)k;
    const double z = FM_MUL(s, s), w = FM_MUL(z, z);
    const double t1 = FM_MUL(w, FM_ADD(Lg2, FM_MUL(w, FM_ADD(Lg4, FM_MUL(w, Lg6)))));
    const double t2 = FM_MUL(z, FM_ADD(Lg1, FM_MUL(w, FM_ADD(Lg3, FM_MUL(w, FM_ADD(Lg5, FM_MUL(w, Lg7)))))));
    const double R = FM_ADD(t2, t1);
    const double hfsq = FM_MUL(FM_MUL(0.5, f), f);
    if (k == 0) return FM_SUB(f, FM_SUB(hfsq, FM_MUL(s, FM_ADD(hfsq, R))));
    return FM_SUB(FM_MUL(dk, ln2_hi), FM_SUB(FM_SUB(hfsq, FM_ADD(FM_MUL(s, FM_ADD(hfsq, R)), FM_MUL(dk, ln2_lo))), f));
}

/* e^x for finite x; overflow -> +inf, below the subnormal range -> 0.  fdlibm e_exp.c: x = k ln2 + r, |r| <= ln2 / 2,
 * e^r = 1 + r + r c / (2 - c) with c = r - r^2 P(r^2), scaled by 2^k through the exponent bits */
FM_HD double fm_exp(double x)
{
    const double o_threshold = 7.09782712893383973096e+02, u_threshold = -7.45133219101941108420e+02;
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, invln2 = 1.44269504088896338700e+00;
    const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
                 P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
    const double twom1000 = 9.33263618503218878990e-302;     /* 2^-1000 */
    if (x > o_threshold) return fm_from_bits(0x7FF0000000000000ULL);
    if (x < u_threshold) return 0.0;
    const double ax = x < 0.0 ? -x : x;
    int k = 0;
    double hi = x, lo = 0.0;
    if (ax > 0.5 * 6.93147180559945286227e-01) {
        k = (int)FM_ADD(FM_MUL(invln2, x), x < 0.0 ? -0.5 : 0.5);       /* truncation toward zero: round to nearest */
        const double t = (double)k;
        hi = FM_SUB(x, FM_MUL(t, ln2_hi));                       /* t * ln2_hi is exact (|k| < 2^11, 32 trailing zeros) */
        lo = FM_MUL(t, ln2_lo);
        x = FM_SUB(hi, lo);
    } else if (ax < 3.7252902984e-09) {                          /* |x| < 2^-28 */
        return FM_ADD(1.0, x);
    }
    const double t = FM_MUL(x, x);
    const double c = FM_SUB(x, FM_MUL(t, FM_ADD(P1, FM_MUL(t, FM_ADD(P2, FM_MUL(t, FM_ADD(P3, FM_MUL(t, FM_ADD(P4, FM_MUL(t, P5))))))))));
    if (k == 0) return FM_SUB(1.0, FM_SUB(FM_DIV(FM_MUL(x, c), FM_SUB(c, 2.0)), x));
    const double y = FM_SUB(1.0, FM_SUB(FM_SUB(lo, FM_DIV(FM_MUL(x, c), FM_SUB(2.0, c))), hi));
    const uint64_t yb = fm_bits(y);
    if (k >= -1021) return fm_from_bits(yb + ((uint64_t)(int64_t)k << 52));
    return FM_MUL(fm_from_bits(yb + ((uint64_t)(int64_t)(k + 1000) << 52)), twom1000);
}

/* Gumbel(0, 1) draw from 64 random bits: u = ((x >> 12) + 0.5) 2^-52 lies in (0, 1) exactly (52 bits plus a half need no
 * rounding; with 53 bits the sum rounds and the largest draw becomes u = 1, g = +inf), g = -log(-log(u)) */
FM_HD double fm_gumbel(uint64_t bits)
{
    const double u = FM_MUL(FM_ADD((double)(bits >> 12), 0.5), 2.220446049250313080847e-16);
    return -fm_log(-fm_log(u));
}
