/* TEST INFRASTRUCTURE ONLY — never linked into, imported by or executed from the product path.
 *
 * mc_oracle_fn.c: the plain-C oracle (mc_oracle.c, compiled into this file unchanged) extended to the product's opt-in
 * function grammar (MCB_GRAMMAR_FUNCTIONS: sin( cos( sqrt( abs( ), so that the whole reference pipeline — field, cases
 * with the ambiguity redirect, soup, welded Poly_Data — can be run on function equations.
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
 * Exports, besides every mco_* function of mc_oracle.h:
 *   int mcof_parse_ok(const char* eq)                    accept/reject under the function grammar
 *   int mcof_set_equation(mco*, int slot, const char* eq) mco_set_equation under the function grammar
 * Built by tests/functions_common.py (gcc -O2 -ffp-contract=off, like oracle/Makefile builds mc_oracle.c).
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
static float fn_powf(float a, float b) { const int f = fn_marker(b); return f ? fn_apply(f, a) : powf(a, b); }
static float fn_mcb_powf(float a, float b) { const int f = fn_marker(b); return f ? fn_apply(f, a) : mcb_powf(a, b); }

#define powf(a, b) fn_powf(a, b)
#define mcb_powf(a, b) fn_mcb_powf(a, b)
#include "mc_oracle.c"
#undef powf
#undef mcb_powf

/* The function grammar's tokenizer: the reference's rules (evaluator.cpp:139-237, as tokenize() in mc_oracle.c) plus a
 * lowercase function name immediately followed by '(' as one more kind of opening bracket. */
static int fn_tokenize(const char* in, Tokens* t) {
    static const char* const names[4] = {"sin(", "cos(", "sqrt(", "abs("};
    t->n = 0; t->valid = 0;
    if (!in || !in[0]) return 0;
    char s[4096]; int len = 0;
    for (const char* p = in; *p && len < 4095; p++) if (*p != ' ') s[len++] = *p;
    s[len] = 0;
    int neg = 0, last = -1, depth = 0;
    int open_fn[4096]; /* per open bracket: 0 plain, 1..4 the function it applies when it closes */
    for (int i = 0; i < len; i++) {
        char ch = s[i];
        if (ch == '-' && (i == 0 || s[i - 1] == '(' || is_op(s[i - 1]))) {
            if (neg) return 0;
            neg = 1;
            if (!push_tok(t, T_NEG, 'N', 0)) return 0;
            continue;
        }
        int f = 0;
        if (ch >= 'a' && ch <= 'z' && !is_var(ch)) {
            for (int k = 0; k < 4 && !f; k++)
                if (strncmp(s + i, names[k], strlen(names[k])) == 0) f = k + 1;
            if (!f) return 0;
        }
        if (ch == '(' || f) {
            if (last == T_VAR || last == T_NUM || last == T_BC) if (!push_tok(t, T_OP, '*', 0)) return 0;
            if (!push_tok(t, T_BO, '(', 0)) return 0;
            if (f && !push_tok(t, T_BO, '(', 0)) return 0; /* f(E) -> ((E) ^ K_f) */
            open_fn[depth++] = f;
            if (f) i += (int)strlen(names[f - 1]) - 1; /* s[i] is the '(': the unary-minus test of the next character sees it */
            last = T_BO;
        } else if (ch == ')') {
            if (neg || last == T_BO || last == T_OP) return 0;
            if (depth == 0) return 0;
            if (!push_tok(t, T_BC, ')', 0)) return 0;
            f = open_fn[--depth];
            if (f) {
                float k;
                memcpy(&k, &kFnMarker[f - 1], 4);
                if (!push_tok(t, T_OP, '^', 0) || !push_tok(t, T_NUM, '0', k) || !push_tok(t, T_BC, ')', 0)) return 0;
            }
            last = T_BC;
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

int mcof_parse_ok(const char* eq) {
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = fn_tokenize(eq, t);
    if (ok) { int uf = 0; eval_tokens(t, 0.5f, 0.25f, 0.75f, 1, &uf); ok = !uf; }
    free(t);
    return ok;
}

int mcof_set_equation(mco* m, int slot, const char* eq) {
    if (slot < 0 || slot > 3) return 0;
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = fn_tokenize(eq, t);
    if (ok) { int uf = 0; eval_tokens(t, 0.5f, 0.25f, 0.75f, 1, &uf); ok = !uf; }
    if (ok) m->eq[slot] = *t;
    free(t);
    return ok;
}
