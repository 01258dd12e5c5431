/* mcb_sinf / mcb_cosf — `sin` and `cos` of the function grammar (mcb.h, MCB_GRAMMAR_FUNCTIONS).
 *
 * The equation language has no reference for these functions, so "correct" is defined as what a C program calling
 * sinf / cosf gets from glibc >= 2.28: Szabolcs Nagy's ARM "optimized-routines" single-precision sine and cosine
 * (MIT licence; glibc sysdeps/ieee754/flt-32/s_sinf.c, s_cosf.c, sincosf.h, sincosf_data.c), in the operation order of
 * the x86-64 FMA build that glibc's IFUNC selects on every FMA-capable CPU (each a*b+c of the source contracted to one
 * fused multiply-add, the products that feed other products left alone).  All arithmetic is IEEE-754 binary64
 * (+, *, fma, conversions) plus 64-bit integer arithmetic, so the same source gives the same bits on the host (compiled
 * with -ffp-contract=off and explicit fma()) and on sm_100a (DFMA; nvcc -fmad=false, NVRTC --fmad=false).
 *
 *   |x| < pi/4      odd (sin) or even (cos) polynomial in x, evaluated in fp64
 *   |x| < 120       x - n pi/2 with n = round(x 2/pi) (a 24-bit fixed-point product), then the polynomial of quadrant n
 *   |x| < inf       Payne-Hanek: 96 bits of 4/pi around the exponent of x (table mcb_trig_inv_pio4), a 62-bit fixed-point
 *                   fraction, times pi/2^62
 *   inf, NaN        NaN
 *
 * oracle/trig_exhaustive.c compares the host build against this machine's libm sinf and cosf on all 2^32 inputs (zero
 * mismatches, NaNs compared as a class) and checks that every finite result lies in [-1, 1], which the interval rule of
 * sin / cos (mcb_interval.h) relies on; profiles/trig_exhaustive.txt is its output.
 */
#ifndef MCB_TRIG_H
#define MCB_TRIG_H

#include "mcb_pow.h" /* integer types, MCB_POW_FN, mcb_f2u / mcb_u2d / mcb_d2u */

/* 4/pi to 192 bits, eight new bits per entry (sincosf_data.c __inv_pio4) */
#define MCB_TRIG_INV_PIO4                                                                                    \
    0xa2u, 0xa2f9u, 0xa2f983u, 0xa2f9836eu, 0xf9836e4eu, 0x836e4e44u, 0x6e4e4415u, 0x4e441529u,              \
    0x441529fcu, 0x1529fc27u, 0x29fc2757u, 0xfc2757d1u, 0x2757d1f5u, 0x57d1f534u, 0xd1f534ddu, 0xf534ddc0u,  \
    0x34ddc0dbu, 0xddc0db62u, 0xc0db6295u, 0xdb629599u, 0x6295993cu, 0x95993c43u, 0x993c4390u, 0x3c439041u

static const uint32_t mcb_trig_inv_pio4_h[24] = {MCB_TRIG_INV_PIO4};
#if defined(__CUDACC__)
static __device__ const uint32_t mcb_trig_inv_pio4_d[24] = {MCB_TRIG_INV_PIO4};
#endif

MCB_POW_FN uint32_t mcb_trig_inv_pio4(int i) {
#if defined(__CUDA_ARCH__)
    return mcb_trig_inv_pio4_d[i];
#else
    return mcb_trig_inv_pio4_h[i];
#endif
}

MCB_POW_FN uint32_t mcb_trig_abstop12(float x) { return (mcb_f2u(x) >> 20) & 0x7ffu; }

/* sinf_poly of sincosf.h: the sine polynomial for even n, the cosine polynomial for odd n.  `neg` selects the
 * second coefficient set (__sincosf_table[1]: cosine coefficients negated). */
MCB_POW_FN double mcb_trig_poly(double x, double x2, int neg, int n) {
    if ((n & 1) == 0) {
        const double S1 = -0x1.555545995a603p-3,
                     S2 = 0x1.1107605230bc4p-7,
                     S3 = -0x1.994eb3774cf24p-13;
        const double x3 = x * x2;
        const double s1 = fma(x2, S3, S2);
        const double x7 = x3 * x2;
        const double s = fma(x3, S1, x);
        return fma(x7, s1, s);
    }
    double C0 = 1.0, C1 = -0x1.ffffffd0c621cp-2,
           C2 = 0x1.55553e1068f19p-5,
           C3 = -0x1.6c087e89a359dp-10,
           C4 = 0x1.99343027bf8c3p-16;
    if (neg) { C0 = -C0; C1 = -C1; C2 = -C2; C3 = -C3; C4 = -C4; }
    const double x4 = x2 * x2;
    const double c2 = fma(x2, C4, C3);
    const double c1 = fma(x2, C1, C0);
    const double x6 = x4 * x2;
    const double c = fma(x4, C2, c1);
    return fma(x6, c2, c);
}

/* |x| < 120: n = nearest integer to x 2/pi, computed as a 2^24-scaled product truncated to int; r = x - n pi/2 */
MCB_POW_FN double mcb_trig_reduce_fast(double x, int* np) {
    const double HPI_INV = 0x1.45f306dc9c883p+23,
                 HPI = 0x1.921fb54442d18p0;
    const double r = x * HPI_INV;
    const int n = ((int32_t)r + 0x800000) >> 24;
    *np = n;
    return fma(-(double)n, HPI, x);
}

/* Payne-Hanek reduction of a finite |x| >= 120 (bit pattern xi): fraction of x 4/pi in 2^62 fixed point */
MCB_POW_FN double mcb_trig_reduce_large(uint32_t xi, int* np) {
    const int base = (int)((xi >> 26) & 15u);
    const int shift = (int)((xi >> 23) & 7u);
    xi = (xi & 0xffffffu) | 0x800000u;
    xi <<= shift;
    uint64_t res0 = (uint64_t)(uint32_t)(xi * mcb_trig_inv_pio4(base));
    const uint64_t res1 = (uint64_t)xi * mcb_trig_inv_pio4(base + 4);
    const uint64_t res2 = (uint64_t)xi * mcb_trig_inv_pio4(base + 8);
    res0 = (res2 >> 32) | (res0 << 32);
    res0 += res1;
    const uint64_t n = (res0 + (1ull << 61)) >> 62;
    res0 -= n << 62;
    const double x = (double)(int64_t)res0;
    *np = (int)n;
    return x * 0x1.921fb54442d18p-62 /* pi / 2^62 */;
}

/* cos = 0: sinf, 1: cosf */
MCB_POW_FN float mcb_trigf(float y, int cos) {
    const double x = (double)y;
    const uint32_t top = mcb_trig_abstop12(y);
    if (top < 0x3f4u) { /* |y| < pi/4 (abstop12(0x1.921fb6p-1f)) */
        if (top < 0x398u) return cos ? 1.0f : y; /* |y| < 2^-12 */
        return (float)mcb_trig_poly(x, x * x, 0, cos);
    }
    int n;
    double r;
    int q;
    if (top < 0x42fu) { /* |y| < 120 */
        r = mcb_trig_reduce_fast(x, &n);
        q = n;
    } else if (top < 0x7f8u) {
        const uint32_t xi = mcb_f2u(y);
        r = mcb_trig_reduce_large(xi, &n);
        q = n + (int)(xi >> 31);
    } else {
        return y - y; /* inf or NaN: NaN (glibc: __math_invalidf) */
    }
    const double s = (q & 1) != (q & 2 ? 1 : 0) ? -1.0 : 1.0; /* sign[q & 3] = {1, -1, -1, 1} */
    return (float)mcb_trig_poly(r * s, r * r, (q & 2) != 0, cos ? n ^ 1 : n);
}

MCB_POW_FN float mcb_sinf(float x) { return mcb_trigf(x, 0); }
MCB_POW_FN float mcb_cosf(float x) { return mcb_trigf(x, 1); }

#endif /* MCB_TRIG_H */
