/* Refined vertices (mcb_set_refine_vertices, include/mcb.h, DESIGN.md §13): every output vertex that lies strictly inside
 * a grid edge moves along that edge to where the equation's point program reaches the surface constant.  One source for
 * g++ (the host build the tests compare with) and nvcc (refine_vertices_kernel); all arithmetic is fp32 without FMA
 * contraction, so both give the same bits.
 *
 * A refined position is a function of the input position's bits, the point program, the surface constant, the scale and
 * the grid's coordinate table c[0..M] only: not of the cube, the mode or the slab that produced the vertex. */
#ifndef MCB_REFINE_H
#define MCB_REFINE_H

#include <math.h>

#include "mcb_bytecode.h"

#define MCB_REFINE_EVALS 40       /* cap on evaluations of the equation per vertex, the two edge ends included */
#define MCB_REFINE_SAME_SIGN (-1) /* mcb_refine_vertex: both edge ends on the same side of the level, vertex unchanged */

/* Marching::interp (marching.cpp:437-446), with t = (c - v_s) / (v_e - v_s) computed once by the caller: the reference
 * calls it three times per edge with the same field values, so the quotient has the same bits every time */
MCB_BC_FN float mcb_interp_ref(float xs, float xe, float t) {
    const float v = t * (xe - xs);
    if (isinf(v) || isnan(v)) return (float)((double)xs + 0.5 * (double)(xe - xs));
    return xs + v;
}

/* Where v lies on the strictly increasing table c[0..M], by exact comparisons: 1 = v equals c[*i]; 2 = v lies strictly
 * inside (c[*i], c[*i + 1]); 0 = outside [c[0], c[M]] or NaN. */
MCB_BC_FN int mcb_refine_locate(const float* c, int M, float v, int* i) {
    if (!(v >= c[0] && v <= c[M])) return 0;
    int lo = 0, hi = M;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (c[mid] <= v) lo = mid;
        else hi = mid;
    }
    if (v == c[lo] || v == c[hi]) {
        *i = v == c[lo] ? lo : hi;
        return 1;
    }
    *i = lo;
    return 2;
}

/* The next float above a finite a */
MCB_BC_FN float mcb_refine_next_up(float a) {
    const uint32_t u = mcb_f2u(a);
    if ((u & 0x7fffffffu) == 0u) return mcb_u2f(1u);
    return mcb_u2f(u >> 31 ? u - 1u : u + 1u);
}

/* |f - iso| as a selection key: d is better than the best so far when smaller, or when the best so far is NaN */
MCB_BC_FN bool mcb_refine_better(float d, float best) { return d < best || (best != best && d == d); }

/* Refine p[3] in place (see include/mcb.h, mcb_set_refine_vertices, for the rule this implements step by step).
 * code / n / k = the point program, c[0..M] = the grid's coordinates (the same table on every axis).
 * Returns the evaluations made (>= 2), 0 when p is not strictly inside a grid edge, MCB_REFINE_SAME_SIGN when both ends
 * of its edge are on the same side of the level; p is unchanged in the last two cases.  bracket, when not null, receives
 * the bracket the search ended with (the tests follow the search with it). */
MCB_BC_FN int mcb_refine_vertex(const uint32_t* code, int n, const float* k, const float* c, int M, float iso, float sx, float sy,
                                float sz, float p[3], float* bracket) {
    int ax = -1, iv = 0, on = 0;
    for (int d = 0; d < 3; d++) {
        int i = 0;
        const int w = mcb_refine_locate(c, M, p[d], &i);
        if (w == 1) on++;
        else if (w == 2 && ax < 0) { ax = d; iv = i; }
        else return 0;
    }
    if (ax < 0 || on != 2) return 0;
    float q[3] = {p[0], p[1], p[2]};
    float a = c[iv], b = c[iv + 1];
    q[ax] = a;
    const float fa = mcb_interp_scalar(code, n, k, sx * q[0], sy * q[1], sz * q[2], 0, 0, 0);
    q[ax] = b;
    const float fb = mcb_interp_scalar(code, n, k, sx * q[0], sy * q[1], sz * q[2], 0, 0, 0);
    const bool sa = fa > iso; /* the classifier's predicate: strict, NaN counts as false */
    if (sa == (fb > iso)) return MCB_REFINE_SAME_SIGN;
    int evals = 2;
    float best = a, bd = mcb_abs(fa - iso);
    const float db = mcb_abs(fb - iso);
    if (mcb_refine_better(db, bd)) { best = b; bd = db; }
    if (bd != 0.f) {
        float ga = fa - iso, gb = fb - iso;            /* Illinois-weighted residuals of the two ends */
        float w1 = b - a, w2 = mcb_u2f(0x7f800000u); /* bracket widths after the previous two steps */
        int last = 0;                                  /* end the previous step replaced: -1 lower, +1 upper */
        float x = mcb_interp_ref(a, b, (iso - fa) / (fb - fa)); /* the edge's canonical linear point, lower -> upper */
        for (;;) {
            if (!(x > a && x < b)) { /* not strictly inside the bracket, or NaN: the midpoint */
                x = a + (b - a) * 0.5f;
                if (!(x > a && x < b)) x = mcb_refine_next_up(a);
            }
            q[ax] = x;
            const float fx = mcb_interp_scalar(code, n, k, sx * q[0], sy * q[1], sz * q[2], 0, 0, 0);
            evals++;
            const float dx = mcb_abs(fx - iso);
            if (mcb_refine_better(dx, bd)) { best = x; bd = dx; }
            if (fx == iso) break;
            if ((fx > iso) == sa) {
                a = x; ga = fx - iso;
                if (last < 0) gb = gb * 0.5f;
                last = -1;
            } else {
                b = x; gb = fx - iso;
                if (last > 0) ga = ga * 0.5f;
                last = 1;
            }
            if (!(mcb_refine_next_up(a) < b)) break;   /* no float strictly between the ends */
            const float w = b - a;
            if (w <= 5.9604644775390625e-8f) break;    /* 2^-24, absolute */
            if (evals >= MCB_REFINE_EVALS) break;
            const bool halved = !(w > 0.5f * w2);      /* over the last two steps */
            w2 = w1;
            w1 = w;
            if (halved) { /* secant; kept 2^-24 clear of the ends, so that a converged side lets the far end in */
                x = a + (b - a) * (ga / (ga - gb));
                if (x - a < 5.9604644775390625e-8f) x = a + 5.9604644775390625e-8f;
                else if (b - x < 5.9604644775390625e-8f) x = b - 5.9604644775390625e-8f;
            } else {
                x = a + (b - a) * 0.5f;
            }
        }
    }
    if (bracket) { bracket[0] = a; bracket[1] = b; }
    p[ax] = best;
    return evals;
}

#endif /* MCB_REFINE_H */
