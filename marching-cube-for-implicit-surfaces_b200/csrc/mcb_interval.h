/* Interval evaluation of a fused grid program (mcb_bytecode.h) over a BOX of grid vertices: an exact proof that every
 * vertex of the box lies on the same side of the iso value, without evaluating the vertices.
 *
 * Why it is exact and not approximate.  The reference evaluates f at a vertex as a fixed sequence of fp32 operations
 * (evaluator.cpp:22-107); the product executes the same sequence (mcb_lower.cpp).  IEEE round-to-nearest is monotone:
 * a <= a' and b <= b' imply fl(a+b) <= fl(a'+b'), and likewise for -, *, / in each argument on an interval that does
 * not change the operation's direction.  So running the SAME operation sequence on [lo, hi] pairs with the usual
 * interval rules, each end point computed in fp32 round-to-nearest, encloses the COMPUTED value (rounding errors and
 * all) of every vertex whose leaf operands lie inside the leaf intervals.  The leaves are the per-axis tables of the
 * hoisted single-variable subtrees, whose minimum and maximum over the box are taken from the actual table entries.
 * Nothing is assumed about the real-valued function.  When the final interval lies entirely above iso (lo > iso) every
 * vertex has sign bit 1; when hi > iso is false every vertex has sign bit 0 (marching.cpp:497-505: strict >); otherwise,
 * or whenever an intermediate end point is not finite (overflow, division by an interval containing zero, a power
 * the rules below do not cover, a NaN or infinity in a table), the box is "unknown" and is evaluated vertex by vertex.
 *
 * `^` (mcb_powf, the restated glibc powf: not correctly rounded, error < 1 ulp): covered for a constant exponent e
 *   - e == 2: the fast path returns fl(x*x) or a value at most one ulp away from it (oracle/pow2_exhaustive.c);
 *   - base interval > 0: x^e is monotone in x; the end point results are widened by 4 ulps;
 *   - e a positive integer and any base: odd powers are monotone, even powers are monotone in |x|; widened likewise.
 * Everything else is "unknown".  tests/test_interval.py checks the enclosure and the proof against brute force on the
 * example equations and on random programs.
 *
 * The function grammar's functions (tests/test_functions_host.py checks them against brute force likewise):
 *   - abs: exact, [|lo|, |hi|] ordered, or [0, max(-lo, hi)] when the interval contains 0;
 *   - sqrt: correctly rounded, hence monotone: [sqrt(lo), sqrt(hi)] when lo >= 0; lo < 0 is "unknown";
 *   - sin, cos: [-1, 1] for any argument interval.  mcb_sinf / mcb_cosf are not the real functions, so no bound may be
 *     taken from analysis; this one rests on the exhaustive run of oracle/trig_exhaustive.c (every finite result of
 *     either function, over all 2^32 inputs, lies in [-1, 1]).  Hoisted sin / cos need no rule at all: their values
 *     are axis-table entries, whose exact minimum and maximum over the box are the leaves;
 *   - min, max (mcb_minf / mcb_maxf): exact and monotone in each argument, [min(a.lo, b.lo), min(a.hi, b.hi)] and the
 *     same for max.  This rests on the invariant that a known interval never encloses a NaN value: sqrt of a possibly
 *     negative interval, division across 0 and non-finite end points already make the box unknown, so the NaN-ignoring
 *     rule of minimumNumber never applies to a value the interval stands for.  An unknown argument makes the result
 *     unknown (the whole program is).  So a box left undecided for min(A, B) is undecided for A or for B.
 */
#ifndef MCB_INTERVAL_H
#define MCB_INTERVAL_H

#include "mcb_bytecode.h"

typedef struct { float lo, hi; } mcb_ival;

MCB_BC_FN int mcb_iv_finite(float v) { return (mcb_f2u(v) & 0x7f800000u) != 0x7f800000u; }

/* v moved n ulps towards -inf (n < 0) or +inf (n > 0) on the ordered line of fp32 values (through the denormals and
 * zero); leaving the finite range yields an inf / NaN pattern, which the caller's finiteness check rejects */
MCB_BC_FN float mcb_iv_step(float v, int n) {
    const uint32_t b = mcb_f2u(v);
    long long key = (b & 0x80000000u) ? -(long long)(b & 0x7fffffffu) : (long long)b;
    key += n;
    const uint32_t r = key < 0 ? (0x80000000u | (uint32_t)(-key)) : (uint32_t)key;
    return mcb_u2f(r);
}

MCB_BC_FN float mcb_iv_min(float a, float b) { return b < a ? b : a; }
MCB_BC_FN float mcb_iv_max(float a, float b) { return b > a ? b : a; }

/* base ^ e for a constant exponent; *bad is set when the rules do not cover the case */
MCB_BC_FN mcb_ival mcb_iv_pow(mcb_ival a, mcb_ival ex, int* bad) {
    mcb_ival r;
    r.lo = 0.f; r.hi = 0.f;
    if (!(ex.lo == ex.hi)) { *bad = 1; return r; }
    const float e = ex.lo;
    if (e == 2.0f) {
        const float l = a.lo * a.lo, h = a.hi * a.hi;
        r.hi = mcb_iv_step(mcb_iv_max(l, h), 2);
        if (a.lo <= 0.f && a.hi >= 0.f) r.lo = 0.f;
        else {
            r.lo = mcb_iv_step(mcb_iv_min(l, h), -2);
            if (r.lo < 0.f) r.lo = 0.f; /* a square is never negative */
        }
        return r;
    }
    if (e == 0.0f) { r.lo = 1.f; r.hi = 1.f; return r; } /* powf(x, 0) = 1 for every x */
    if (a.lo > 0.f) {
        const float l = mcb_powf(a.lo, e), h = mcb_powf(a.hi, e);
        r.lo = mcb_iv_step(mcb_iv_min(l, h), -4);
        r.hi = mcb_iv_step(mcb_iv_max(l, h), 4);
        if (r.lo < 0.f) r.lo = 0.f;
        return r;
    }
    if (e >= 1.0f && e <= 1024.0f && e == (float)(int)e) { /* positive integer power of a base that may be <= 0 */
        const int odd = ((int)e) & 1;
        const float l = mcb_powf(a.lo, e), h = mcb_powf(a.hi, e);
        if (odd) { r.lo = mcb_iv_step(l, -4); r.hi = mcb_iv_step(h, 4); return r; }
        r.hi = mcb_iv_step(mcb_iv_max(l, h), 4);
        if (a.hi < 0.f) { r.lo = mcb_iv_step(h, -4); if (r.lo < 0.f) r.lo = 0.f; }
        else r.lo = 0.f; /* the base interval contains 0 (a.lo <= 0 <= a.hi, since a.lo > 0 was handled above) */
        return r;
    }
    *bad = 1;
    return r;
}

MCB_BC_FN mcb_ival mcb_iv_op(uint32_t fop, mcb_ival acc, mcb_ival v, int* bad) {
    mcb_ival r;
    switch (fop) {
        case MCB_F_ADD: r.lo = acc.lo + v.lo; r.hi = acc.hi + v.hi; break;
        case MCB_F_SUB: r.lo = acc.lo - v.hi; r.hi = acc.hi - v.lo; break;
        case MCB_F_RSUB: r.lo = v.lo - acc.hi; r.hi = v.hi - acc.lo; break;
        case MCB_F_MUL: {
            const float p1 = acc.lo * v.lo, p2 = acc.lo * v.hi, p3 = acc.hi * v.lo, p4 = acc.hi * v.hi;
            r.lo = mcb_iv_min(mcb_iv_min(p1, p2), mcb_iv_min(p3, p4));
            r.hi = mcb_iv_max(mcb_iv_max(p1, p2), mcb_iv_max(p3, p4));
            break;
        }
        case MCB_F_DIV:
        case MCB_F_RDIV: {
            const mcb_ival n = fop == MCB_F_DIV ? acc : v, d = fop == MCB_F_DIV ? v : acc;
            if (!(d.lo > 0.f || d.hi < 0.f)) { *bad = 1; r.lo = r.hi = 0.f; break; }
            const float q1 = n.lo / d.lo, q2 = n.lo / d.hi, q3 = n.hi / d.lo, q4 = n.hi / d.hi;
            r.lo = mcb_iv_min(mcb_iv_min(q1, q2), mcb_iv_min(q3, q4));
            r.hi = mcb_iv_max(mcb_iv_max(q1, q2), mcb_iv_max(q3, q4));
            break;
        }
        case MCB_F_POW: r = mcb_iv_pow(acc, v, bad); break;
        case MCB_F_RPOW: r = mcb_iv_pow(v, acc, bad); break;
        case MCB_F_MIN: r.lo = mcb_minf(acc.lo, v.lo); r.hi = mcb_minf(acc.hi, v.hi); break;
        case MCB_F_MAX: r.lo = mcb_maxf(acc.lo, v.lo); r.hi = mcb_maxf(acc.hi, v.hi); break;
        default: r = v; break; /* LOAD, PUSH */
    }
    if (!mcb_iv_finite(r.lo) || !mcb_iv_finite(r.hi)) *bad = 1;
    return r;
}

/* f(a) for the function grammar's fop SIN / COS / SQRT / ABS; *bad is set when the rules do not cover the case */
MCB_BC_FN mcb_ival mcb_iv_fn(uint32_t fop, mcb_ival a, int* bad) {
    mcb_ival r;
    switch (fop) {
        case MCB_F_ABS:
            if (a.lo >= 0.f) r = a;
            else if (a.hi <= 0.f) { r.lo = -a.hi; r.hi = -a.lo; }
            else { r.lo = 0.f; r.hi = mcb_iv_max(-a.lo, a.hi); }
            break;
        case MCB_F_SQRT:
            if (!(a.lo >= 0.f)) { *bad = 1; r.lo = r.hi = 0.f; break; }
            r.lo = mcb_fn(2, a.lo);
            r.hi = mcb_fn(2, a.hi);
            break;
        default: /* sin, cos */
            r.lo = -1.f;
            r.hi = 1.f;
            break;
    }
    return r;
}

/* Bounds of the axis-table operands over the box: B[(axis * slots_per_axis + slot) * nb + b] = {min, max} of that
 * table over block b of that axis (a non-finite entry makes the pair {-inf, +inf}).  bx, by, bz = the box's block
 * index per axis.  Returns 0 = unknown, 1 = every vertex has sign bit 0 (value > iso is false), 2 = every vertex has
 * sign bit 1. */
MCB_BC_FN int mcb_interval_class(const uint32_t* code, int n, const float* k, const mcb_ival* B, int slots_per_axis, int nb,
                                 int bx, int by, int bz, float iso, mcb_ival* out) {
    mcb_ival st[MCB_MAX_STACK];
    int sp = 0, bad = 0;
    mcb_ival acc;
    acc.lo = 0.f; acc.hi = 0.f;
    for (int pc = 0; pc < n && !bad; pc++) {
        const uint32_t w = code[pc], arg = MCB_FINSN_ARG(w);
        uint32_t fop = MCB_FINSN_OP(w), src = MCB_FINSN_SRC(w);
        MCB_FINSN_DECODE(fop, src);
        if (fop == MCB_F_NEG) { const float t = acc.lo; acc.lo = -acc.hi; acc.hi = -t; continue; }
        if (MCB_F_IS_FN(fop)) { acc = mcb_iv_fn(fop, acc, &bad); continue; }
        if (fop == MCB_F_PUSH) { if (sp >= MCB_MAX_STACK) { bad = 1; break; } st[sp++] = acc; }
        mcb_ival v;
        switch (src) {
            case MCB_SRC_K: v.lo = k[arg]; v.hi = v.lo; break;
            case MCB_SRC_TX: v = B[((size_t)0 * slots_per_axis + arg) * nb + bx]; break;
            case MCB_SRC_TY: v = B[((size_t)1 * slots_per_axis + arg) * nb + by]; break;
            case MCB_SRC_TZ: v = B[((size_t)2 * slots_per_axis + arg) * nb + bz]; break;
            case MCB_SRC_POP: if (sp <= 0) { bad = 1; v.lo = v.hi = 0.f; } else v = st[--sp]; break;
            default: bad = 1; v.lo = v.hi = 0.f; break; /* raw coordinates do not occur in grid programs */
        }
        if (!mcb_iv_finite(v.lo) || !mcb_iv_finite(v.hi)) { bad = 1; break; }
        acc = mcb_iv_op(fop, acc, v, &bad);
    }
    if (out) *out = acc;
    if (bad || n <= 0) return 0;
    if (acc.lo > iso) return 2;
    if (!(acc.hi > iso)) return 1;
    return 0;
}

#endif /* MCB_INTERVAL_H */
