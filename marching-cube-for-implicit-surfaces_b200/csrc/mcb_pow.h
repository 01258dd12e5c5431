/* mcb_powf — the `^` operator of the equation language (evaluator.cpp:133 calls pow(float,float) -> libm powf).
 *
 * The reference delegates `^` to the platform C runtime, which is NOT part of /root/reference (MSVC 2015 CRT on
 * the author's machine; glibc 2.39 libm wherever the oracle is built).  Following the rule for third-party
 * arithmetic on the path, this header restates the PUBLISHED algorithm that glibc >= 2.28 uses for powf
 * (Szabolcs Nagy's ARM "optimized-routines" powf, MIT licence: sysdeps/ieee754/flt-32/e_powf.c + e_powf_log2_data.c
 * + e_exp2f_data.c), in the exact operation order of the x86-64 FMA build that glibc's IFUNC selects on every
 * FMA-capable CPU (each a*b+c of the source contracted to one fused multiply-add).  All arithmetic is IEEE-754
 * binary64 (+, *, fma) plus integer bit manipulation, so the same source gives the same bits on the host (oracle,
 * compiled with -ffp-contract=off and explicit fma()) and on sm_100a (DFMA; compiled with -fmad=false).
 *
 * tests/test_pow.py checks the host build of this header against libm's powf on >1e8 random and edge-case inputs
 * and requires zero mismatches (NaNs compared as a class); the GPU build is checked against both.
 *
 *   log2(x)  : x = 2^k * z, z in [0x1.66p-1, 0x1.66p0); 16-entry table of (1/c, log2 c); degree-5 polynomial in r = z/c - 1
 *   2^(y*log2 x): k/32 + r split with the 0x1.8p47 shift trick; 32-entry table of 2^(i/32); degree-3 polynomial
 */
#ifndef MCB_POW_H
#define MCB_POW_H

#if defined(__CUDACC_RTC__) /* run-time compilation (mcb_jit.cpp): no host headers, device code only */
typedef unsigned int uint32_t;
typedef int int32_t;
typedef unsigned long long uint64_t;
typedef long long int64_t;
#else
#include <stdint.h>
#include <string.h>
#if !defined(__CUDACC__)
#include <math.h>
#endif
#endif

#if defined(__CUDACC__)
#define MCB_POW_FN __host__ __device__ __forceinline__
#else
#define MCB_POW_FN static inline
#endif

/* (invc, logc) pairs, then the polynomial / table constants, as IEEE-754 binary64 bit patterns. */
#define MCB_POW_LOG2_TAB                                                                                     \
    0x3ff661ec79f8f3beull, 0xbfdefec65b963019ull, 0x3ff571ed4aaf883dull, 0xbfdb0b6832d4fca4ull,              \
    0x3ff49539f0f010b0ull, 0xbfd7418b0a1fb77bull, 0x3ff3c995b0b80385ull, 0xbfd39de91a6dcf7bull,              \
    0x3ff30d190c8864a5ull, 0xbfd01d9bf3f2b631ull, 0x3ff25e227b0b8ea0ull, 0xbfc97c1d1b3b7af0ull,              \
    0x3ff1bb4a4a1a343full, 0xbfc2f9e393af3c9full, 0x3ff12358f08ae5baull, 0xbfb960cbbf788d5cull,              \
    0x3ff0953f419900a7ull, 0xbfaa6f9db6475fceull, 0x3ff0000000000000ull, 0x0000000000000000ull,              \
    0x3fee608cfd9a47acull, 0x3fb338ca9f24f53dull, 0x3feca4b31f026aa0ull, 0x3fc476a9543891baull,              \
    0x3feb2036576afce6ull, 0x3fce840b4ac4e4d2ull, 0x3fe9c2d163a1aa2dull, 0x3fd40645f0c6651cull,              \
    0x3fe886e6037841edull, 0x3fd88e9c2c1b9ff8ull, 0x3fe767dcf5534862ull, 0x3fdce0a44eb17bccull

#define MCB_POW_EXP2_TAB                                                                                     \
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,              \
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,              \
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,              \
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,              \
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,              \
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,              \
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,              \
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull

static const uint64_t mcb_pow_log2_tab_h[32] = {MCB_POW_LOG2_TAB};
static const uint64_t mcb_pow_exp2_tab_h[32] = {MCB_POW_EXP2_TAB};
#if defined(__CUDACC__)
static __device__ const uint64_t mcb_pow_log2_tab_d[32] = {MCB_POW_LOG2_TAB};
static __device__ const uint64_t mcb_pow_exp2_tab_d[32] = {MCB_POW_EXP2_TAB};
#endif

MCB_POW_FN uint32_t mcb_f2u(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}
MCB_POW_FN float mcb_u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}
MCB_POW_FN uint64_t mcb_d2u(double d) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(d);
#else
    uint64_t u; memcpy(&u, &d, 8); return u;
#endif
}
MCB_POW_FN double mcb_u2d(uint64_t u) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double d; memcpy(&d, &u, 8); return d;
#endif
}
MCB_POW_FN double mcb_log2_tab(int i) {
#if defined(__CUDA_ARCH__)
    return mcb_u2d(mcb_pow_log2_tab_d[i]);
#else
    return mcb_u2d(mcb_pow_log2_tab_h[i]);
#endif
}
MCB_POW_FN uint64_t mcb_exp2_tab(int i) {
#if defined(__CUDA_ARCH__)
    return mcb_pow_exp2_tab_d[i];
#else
    return mcb_pow_exp2_tab_h[i];
#endif
}

/* 0: y is not an integer, 1: odd integer, 2: even integer */
MCB_POW_FN int mcb_pow_checkint(uint32_t iy) {
    int e = (int)(iy >> 23 & 0xff);
    if (e < 0x7f) return 0;
    if (e > 0x7f + 23) return 2;
    if (iy & ((1u << (0x7f + 23 - e)) - 1)) return 0;
    if (iy & (1u << (0x7f + 23 - e))) return 1;
    return 2;
}
MCB_POW_FN int mcb_pow_zeroinfnan(uint32_t ix) { return 2 * ix - 1 >= 2u * 0x7f800000u - 1; }
MCB_POW_FN int mcb_pow_issignaling(uint32_t ix) { return ((ix ^ 0x00400000u) & 0x7fffffffu) > 0x7fc00000u; }

/* log2_inline of the algorithm: log2(x) in fp64 for the bits ix of a positive, normal, finite x (a subnormal x arrives
 * normalised, its exponent below the range of the field).  mcb_powf_full below and mcb_lnf of the analytic normals. */
MCB_POW_FN double mcb_pow_log2(uint32_t ix) {
    uint32_t tmp = ix - 0x3f330000u;
    int i = (int)((tmp >> 19) & 15u);
    uint32_t top = tmp & 0xff800000u;
    uint32_t iz = ix - top;
    int k = (int32_t)top >> 23;
    double invc = mcb_log2_tab(2 * i), logc = mcb_log2_tab(2 * i + 1);
    double z = (double)mcb_u2f(iz);
    const double A0 = mcb_u2d(0x3fd27616c9496e0bull), A1 = mcb_u2d(0xbfd71969a075c67aull),
                 A2 = mcb_u2d(0x3fdec70a6ca7baddull), A3 = mcb_u2d(0xbfe7154748bef6c8ull),
                 A4 = mcb_u2d(0x3ff71547652ab82bull);
    double r = fma(z, invc, -1.0);
    double y0 = logc + (double)k;
    double r2 = r * r;
    double yy = fma(A0, r, A1);
    double p = fma(A2, r, A3);
    double r4 = r2 * r2;
    double q = fma(A4, r, y0);
    q = fma(p, r2, q);
    return fma(yy, r4, q);
}

MCB_POW_FN float mcb_powf_full(float x, float y) {
    uint32_t sign_bias = 0;
    uint32_t ix = mcb_f2u(x), iy = mcb_f2u(y);
    if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u || mcb_pow_zeroinfnan(iy)) {
        /* x < 0x1p-126, inf or nan; or y is 0, inf or nan */
        if (mcb_pow_zeroinfnan(iy)) {
            if (2 * iy == 0) return mcb_pow_issignaling(ix) ? x + y : 1.0f;
            if (ix == 0x3f800000u) return mcb_pow_issignaling(iy) ? x + y : 1.0f;
            if (2 * ix > 2u * 0x7f800000u || 2 * iy > 2u * 0x7f800000u) return x + y;
            if (2 * ix == 2u * 0x3f800000u) return 1.0f;
            if ((2 * ix < 2u * 0x3f800000u) == !(iy & 0x80000000u)) return 0.0f;
            return y * y;
        }
        if (mcb_pow_zeroinfnan(ix)) {
            float x2 = x * x;
            if ((ix & 0x80000000u) && mcb_pow_checkint(iy) == 1) { x2 = -x2; sign_bias = 1; }
            if (2 * ix == 0 && (iy & 0x80000000u)) return mcb_u2f(sign_bias ? 0xff800000u : 0x7f800000u);
            return (iy & 0x80000000u) ? 1 / x2 : x2;
        }
        if (ix & 0x80000000u) { /* finite x < 0 */
            int yint = mcb_pow_checkint(iy);
            if (yint == 0) return mcb_u2f(0x7fc00000u) ; /* invalid: (x-x)/(x-x) */
            if (yint == 1) sign_bias = 1u << 16;
            ix &= 0x7fffffffu;
        }
        if (ix < 0x00800000u) { /* subnormal x: normalise */
            ix = mcb_f2u(x * 8388608.0f);
            ix &= 0x7fffffffu;
            ix -= 23u << 23;
        }
    }
    double logx = mcb_pow_log2(ix); /* log2_inline */
    double ylogx = (double)y * logx;
    if ((mcb_d2u(ylogx) >> 47 & 0xffff) >= 0x80bfu) { /* |y*log2(x)| >= 126 */
        /* (the round-away check for 0x1.fffffffa3aae2p+6 < ylogx is a no-op in round-to-nearest) */
        if (ylogx > mcb_u2d(0x405fffffffd1d571ull)) /* 0x1.fffffffd1d571p+6 */ return mcb_u2f(sign_bias ? 0xff800000u : 0x7f800000u);
        if (ylogx <= -150.0) return mcb_u2f(sign_bias ? 0x80000000u : 0x00000000u);
        if (ylogx < -149.0) return mcb_u2f(sign_bias ? 0x80000001u : 0x00000001u);
    }
    /* exp2_inline */
    const double SHIFT = mcb_u2d(0x42e8000000000000ull); /* 0x1.8p47 */
    const double C0 = mcb_u2d(0x3fac6af84b912394ull), C1 = mcb_u2d(0x3fcebfce50fac4f3ull),
                 C2 = mcb_u2d(0x3fe62e42ff0c52d6ull);
    double kd = ylogx + SHIFT;
    uint64_t ki = mcb_d2u(kd);
    kd -= SHIFT;
    double rr = ylogx - kd;
    uint64_t t = mcb_exp2_tab((int)(ki & 31u));
    uint64_t ski = ki + sign_bias;
    t += ski << 47;
    double s = mcb_u2d(t);
    double zz = fma(C0, rr, C1);
    double rr2 = rr * rr;
    double out = fma(C2, rr, 1.0);
    out = fma(zz, rr2, out);
    out = out * s;
    return (float)out;
}

/* x^2, the exponent every example equation uses, without the fp64 log2/exp2 round trip — and still bit-identical
 * to the algorithm above (hence to glibc's powf(x, 2)).
 *
 * powf(x,2) is the correctly rounded square EXCEPT when x*x lies so close to the midpoint of two floats that the
 * ~2^-33 relative error of the fp64 evaluation pushes it across.  An exhaustive run over all 2^32 inputs
 * (oracle/pow2_exhaustive.c) shows that every such input has x*x within 0.00166 ulp of a midpoint (results in
 * [2^-100, 2^100]).  So: r = RN(x*x), err = fma(x, x, -r) is the exact rounding residual, and whenever
 * |err| <= (1/2 - 2^-9) ulp(r) the result is r; the rare remainder (0.4 % of inputs) takes the full algorithm.
 * All of it is fp32: one multiply, one fused multiply-add, a few integer operations. */
MCB_POW_FN int mcb_pow2_try(float x, float* out) {
#if defined(__CUDA_ARCH__)
    const float r = __fmul_rn(x, x);
    const float err = __fmaf_rn(x, x, -r);
#else
    const float r = x * x;
    const float err = fmaf(x, x, -r);
#endif
    const uint32_t ex = mcb_f2u(r) >> 23; /* r >= 0 or NaN: no sign bit to strip for finite values */
    if (ex < 27u || ex > 227u) return 0;   /* result outside [2^-100, 2^100] (or NaN/inf): full algorithm */
    const float lim = 0.498046875f * mcb_u2f((ex - 23u) << 23); /* (1/2 - 2^-9) * ulp(r), exact */
    if (!(mcb_u2f(mcb_f2u(err) & 0x7fffffffu) <= lim)) return 0;
    *out = r;
    return 1;
}

MCB_POW_FN float mcb_powf(float x, float y) {
    float r;
    if (mcb_f2u(y) == 0x40000000u && mcb_pow2_try(x, &r)) return r;
    return mcb_powf_full(x, y);
}

#endif /* MCB_POW_H */
