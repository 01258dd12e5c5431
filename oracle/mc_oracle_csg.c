/* TEST INFRASTRUCTURE ONLY — never linked into, imported by or executed from the product path.
 *
 * mc_oracle_csg.c: the plain-C oracle (mc_oracle.c, compiled into this file unchanged) extended to the whole of the
 * product's opt-in function grammar (MCB_GRAMMAR_FUNCTIONS: sin( cos( sqrt( abs( and the two-argument min( max( ), so that
 * the reference pipeline — field, cases with the ambiguity redirect, soup, welded Poly_Data — can be run on equations
 * that combine shapes.  It extends mc_oracle_fn.c (the one-argument functions, which it restates the same way) with
 * min and max.
 *
 * It is a restatement of the grammar independent of the product's (csrc/mcb_lower.cpp): its own tokenizer, below, and
 * the oracle's own two-stack walk, with libm's sinf / cosf / sqrtf / fabsf doing the arithmetic.  The grammar says that
 * `f(E)` behaves exactly like the bracketed operand `(E)` with f applied at its closing bracket.  The tokenizer spells
 * that with the tokens the oracle's walk already knows: `f(E)` becomes `((E) ^ K_f)`, where K_f is a NaN with a payload
 * that names f.  The inner brackets make E one operand, the outer ones close `^` before anything outside can reach it,
 * so the walk applies `^` to (E, K_f) at exactly the point where it would close `(E)`; `^` of the oracle (powf, or
 * mcb_powf in pow_mode 1) is intercepted here and applies f when its exponent is one of the four markers.  No literal
 * or computed value can be such a NaN: literals are digit strings, and arithmetic never sees the markers.
 *
 * The two-argument min(A,B) and max(A,B) close A at the ',' as `(A)` is closed at ')', and B at the ')'.  They are
 * spelt `((A) ^ ((B) ^ K_i))` with a marker K_i per occurrence i: the inner `^` stashes B in slot i and returns a second
 * marker M_i, the outer `^` returns min(A, slot i) (or max).  The walk evaluates the inner `^` before the outer one, and
 * every nested occurrence has its own slot.  min and max are written out below from their definition (IEEE 754-2019
 * minimumNumber / maximumNumber: a NaN operand is ignored, -0 < +0), with no fminf and nothing shared with the product.
 *
 * Exports, besides every mco_* function of mc_oracle.h:
 *   int mcoc_parse_ok(const char* eq)                    accept/reject under the function grammar
 *   int mcoc_set_equation(mco*, int slot, const char* eq) mco_set_equation under the function grammar
 *   float mcoc_min(float, float), mcoc_max(float, float) the restatement of min / max used by the walk
 * Built by tests/csg_common.py (gcc -O2 -ffp-contract=off, like oracle/Makefile builds mc_oracle.c).
 */
#define _GNU_SOURCE
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../marching-cube-for-implicit-surfaces_b200/csrc/mcb_pow.h"

static const uint32_t kFnMarker[4] = {0x7fc0f001u, 0x7fc0f002u, 0x7fc0f003u, 0x7fc0f004u}; /* sin cos sqrt abs */

static int fn_marker(float b) {
    uint32_t u;
    memcpy(&u, &b, 4);
    for (int f = 0; f < 4; f++)
        if (u == kFnMarker[f]) return f + 1;
    return 0;
}
static float fn_apply(int f, float v) { /* libm itself */
    switch (f) {
        case 1: return sinf(v);
        case 2: return cosf(v);
        case 3: return sqrtf(v);
        default: return fabsf(v);
    }
}
/* min / max markers: quiet NaNs 0x7fe0_0000 (inner, K_i) and 0x7fd0_0000 (outer, M_i), | 0x1000 for max, | i */
#define MM_MAX_OCC 4096
#define MM_INNER 0x7fe00000u
#define MM_OUTER 0x7fd00000u
static __thread float mm_slot[MM_MAX_OCC];

static float mm_min(float a, float b) {
    if (isnan(a)) return b; /* NaN when both are */
    if (isnan(b)) return a;
    if (a == b) return signbit(a) ? a : b; /* +0 and -0: -0 */
    return a < b ? a : b;
}
static float mm_max(float a, float b) {
    if (isnan(a)) return b;
    if (isnan(b)) return a;
    if (a == b) return signbit(a) ? b : a; /* +0 and -0: +0 */
    return a > b ? a : b;
}
float mcoc_min(float a, float b) { return mm_min(a, b); }
float mcoc_max(float a, float b) { return mm_max(a, b); }

/* 1 and *r set when b is a min / max marker */
static int mm_intercept(float a, float b, float* r) {
    uint32_t u;
    memcpy(&u, &b, 4);
    const uint32_t tag = u & 0xfff00000u, i = u & 0xfffu;
    if (tag == MM_INNER) { mm_slot[i] = a; u = MM_OUTER | (u & 0x1fffu); memcpy(r, &u, 4); return 1; }
    if (tag == MM_OUTER) { *r = (u & 0x1000u) ? mm_max(a, mm_slot[i]) : mm_min(a, mm_slot[i]); return 1; }
    return 0;
}

static float fn_powf(float a, float b) {
    float r;
    if (mm_intercept(a, b, &r)) return r;
    const int f = fn_marker(b);
    return f ? fn_apply(f, a) : powf(a, b);
}
static float fn_mcb_powf(float a, float b) {
    float r;
    if (mm_intercept(a, b, &r)) return r;
    const int f = fn_marker(b);
    return f ? fn_apply(f, a) : mcb_powf(a, b);
}

#define powf(a, b) fn_powf(a, b)
#define mcb_powf(a, b) fn_mcb_powf(a, b)
#include "mc_oracle.c"
#undef powf
#undef mcb_powf

/* The function grammar's tokenizer: the reference's rules (evaluator.cpp:139-237, as tokenize() in mc_oracle.c) plus a
 * lowercase function name immediately followed by '(' as one more kind of opening bracket, and exactly one ',' directly
 * inside min( / max(, after which the rules that follow '(' apply. */
static int fn_tokenize(const char* in, Tokens* t) {
    static const char* const names[6] = {"sin(", "cos(", "sqrt(", "abs(", "min(", "max("};
    t->n = 0; t->valid = 0;
    if (!in || !in[0]) return 0;
    char s[4096]; int len = 0;
    for (const char* p = in; *p && len < 4095; p++) if (*p != ' ') s[len++] = *p;
    s[len] = 0;
    int neg = 0, last = -1, depth = 0, occ = 0;
    int open_fn[4096];    /* per open bracket: 0 plain, 1..4 the function it applies when it closes, 5 min, 6 max */
    int open_comma[4096]; /* min / max: 1 once its ',' is seen */
    int open_occ[4096];   /* min / max: its occurrence number */
    for (int i = 0; i < len; i++) {
        char ch = s[i];
        if (ch == '-' && (i == 0 || s[i - 1] == '(' || s[i - 1] == ',' || is_op(s[i - 1]))) {
            if (neg) return 0;
            neg = 1;
            if (!push_tok(t, T_NEG, 'N', 0)) return 0;
            continue;
        }
        int f = 0;
        if (ch >= 'a' && ch <= 'z' && !is_var(ch)) {
            for (int k = 0; k < 6 && !f; k++)
                if (strncmp(s + i, names[k], strlen(names[k])) == 0) f = k + 1;
            if (!f) return 0;
        }
        if (ch == '(' || f) {
            if (last == T_VAR || last == T_NUM || last == T_BC) if (!push_tok(t, T_OP, '*', 0)) return 0;
            if (!push_tok(t, T_BO, '(', 0)) return 0;
            if (f && !push_tok(t, T_BO, '(', 0)) return 0; /* f(E) -> ((E) ^ K_f), min(A,B) -> ((A) ^ ((B) ^ K_i)) */
            if (f >= 5) {
                if (occ >= MM_MAX_OCC) return 0;
                open_occ[depth] = occ++;
            }
            open_comma[depth] = 0;
            open_fn[depth++] = f;
            if (f) i += (int)strlen(names[f - 1]) - 1; /* s[i] is the '(': the unary-minus test of the next character sees it */
            last = T_BO;
        } else if (ch == ')') {
            if (neg || last == T_BO || last == T_OP) return 0;
            if (depth == 0) return 0;
            if (open_fn[depth - 1] >= 5 && !open_comma[depth - 1]) return 0; /* min( / max( with one argument */
            if (!push_tok(t, T_BC, ')', 0)) return 0;
            f = open_fn[--depth];
            if (f >= 5) {
                const uint32_t u = MM_INNER | (f == 6 ? 0x1000u : 0u) | (uint32_t)open_occ[depth];
                float k;
                memcpy(&k, &u, 4);
                if (!push_tok(t, T_OP, '^', 0) || !push_tok(t, T_NUM, '0', k) || !push_tok(t, T_BC, ')', 0) ||
                    !push_tok(t, T_BC, ')', 0)) return 0;
            } else if (f) {
                float k;
                memcpy(&k, &kFnMarker[f - 1], 4);
                if (!push_tok(t, T_OP, '^', 0) || !push_tok(t, T_NUM, '0', k) || !push_tok(t, T_BC, ')', 0)) return 0;
            }
            last = T_BC;
        } else if (ch == ',') {
            if (neg || last == T_BO || last == T_OP) return 0;
            if (depth == 0 || open_fn[depth - 1] < 5 || open_comma[depth - 1]) return 0;
            open_comma[depth - 1] = 1;
            /* (A) closed; ^ ( ( opens B */
            if (!push_tok(t, T_BC, ')', 0) || !push_tok(t, T_OP, '^', 0) || !push_tok(t, T_BO, '(', 0) ||
                !push_tok(t, T_BO, '(', 0)) return 0;
            last = T_BO;
        } else if (is_op(ch)) {
            if (neg || last == T_BO || last == T_OP || last == -1) return 0;
            if (!push_tok(t, T_OP, ch, 0)) return 0;
            last = T_OP;
        } else if (is_num(ch)) {
            if (last == T_VAR || last == T_BC) if (!push_tok(t, T_OP, '*', 0)) return 0;
            char buf[512]; int bl = 0; int dot = (ch == '.');
            buf[bl++] = ch;
            while (i + 1 < len && is_num(s[i + 1])) {
                if (s[i + 1] == '.') { if (dot) return 0; dot = 1; }
                if (bl < 510) buf[bl++] = s[++i]; else ++i;
            }
            buf[bl] = 0;
            if (bl == 1 && buf[0] == '.') return 0;
            if (!push_tok(t, T_NUM, '0', strtof(buf, NULL))) return 0;
            last = T_NUM;
        } else if (is_var(ch)) {
            if (last == T_VAR || last == T_NUM || last == T_BC) if (!push_tok(t, T_OP, '*', 0)) return 0;
            char v = (ch == 'x' || ch == 'X') ? 'x' : (ch == 'y' || ch == 'Y') ? 'y' : 'z';
            if (!push_tok(t, T_VAR, v, 0)) return 0;
            last = T_VAR;
        } else return 0;
        neg = 0;
    }
    if (depth != 0) return 0;
    t->valid = 1;
    return 1;
}

int mcoc_parse_ok(const char* eq) {
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = fn_tokenize(eq, t);
    if (ok) { int uf = 0; eval_tokens(t, 0.5f, 0.25f, 0.75f, 1, &uf); ok = !uf; }
    free(t);
    return ok;
}

int mcoc_set_equation(mco* m, int slot, const char* eq) {
    if (slot < 0 || slot > 3) return 0;
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = fn_tokenize(eq, t);
    if (ok) { int uf = 0; eval_tokens(t, 0.5f, 0.25f, 0.75f, 1, &uf); ok = !uf; }
    if (ok) m->eq[slot] = *t;
    free(t);
    return ok;
}
