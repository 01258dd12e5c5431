/* TEST INFRASTRUCTURE ONLY — never linked into, imported by or executed from the product path.
 *
 * mc_oracle.c: a CPU restatement, in plain C, of the reference's hot path (equation -> field -> cube cases with the
 * ambiguity redirect -> interpolated triangles -> welded Poly_Data -> normal.h normals), written from the behaviour
 * of the reference, function by function, with the file:line each part follows.  It is a second, independent
 * implementation: it walks the token list with two stacks like the reference does (it does NOT share the product's
 * bytecode lowering), so agreement between the CUDA path and this file is agreement between two different
 * derivations of the same semantics.
 *
 * Pinning: tests/test_oracle.py checks this file against the golden vectors produced by the UNMODIFIED reference
 * (tests/golden/cases.npz <- oracle/_ref) — per-cube codes, table rows, soup, welded mesh and normal.h normals, all
 * bit-exact — and, where oracle/_ref is present, against the reference live on further inputs.
 *
 * Who may use it: tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.  Nothing else.
 */
#define _GNU_SOURCE
#include "mc_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "../marching-cube-for-implicit-surfaces_b200/csrc/mcb_pow.h"    /* mcb_powf (pow_mode 1) */
#include "../marching-cube-for-implicit-surfaces_b200/csrc/mcb_tables.h" /* packed tri table, edge/face conventions */

#define MAXTOK 1024
enum { T_OP, T_NUM, T_VAR, T_BO, T_BC, T_NEG };

typedef struct {
    int n;
    unsigned char type[MAXTOK];
    char ch[MAXTOK];   /* operator / variable character */
    float num[MAXTOK]; /* value of a NUM token: strtof, like stof at evaluator.cpp:82 */
    int valid;
} Tokens;

typedef struct {
    int op; /* 0 '>', 1 '<', 2 '>=', 3 '<=' (marching.h:58) */
    float rhs;
    int in_use;
} Cons;

struct mco {
    Tokens eq[4];
    Cons cons[3];
    int pow_mode;
    float step, sx, sy, sz, iso;
    int repeat;  /* repeating-surface mode, marching.cpp:481-494 */
    float rstep;
    int M;
    float* c;  /* loop values c[0..M-1], c[M] = c[M-1]+step */
    float* cs; /* with apron: cs[v+1] = c[v], v in [-1, M+1] */
    int8_t face[256];
    /* welded mesh (Poly_Data, marching.h:26-30) */
    float* verts; long nverts, capv;
    unsigned* tris; long ntris, capt;
};

/* ---- tokenizer: Evaluator::tokenize, evaluator.cpp:139-237 ---------------------------------------------------- */
static int is_op(char c) { return c == '+' || c == '-' || c == '*' || c == '/' || c == '^'; }
static int is_num(char c) { return (c >= '0' && c <= '9') || c == '.'; }
static int is_var(char c) { return (c >= 'x' && c <= 'z') || (c >= 'X' && c <= 'Z'); }

static int push_tok(Tokens* t, int type, char ch, float num) {
    if (t->n >= MAXTOK) return 0;
    t->type[t->n] = (unsigned char)type; t->ch[t->n] = ch; t->num[t->n] = num; t->n++;
    return 1;
}

static int tokenize(const char* in, Tokens* t) {
    t->n = 0; t->valid = 0;
    if (!in || !in[0]) return 0;                          /* :141 */
    char s[4096]; int len = 0;
    for (const char* p = in; *p && len < 4095; p++) if (*p != ' ') s[len++] = *p; /* :147 */
    s[len] = 0;
    int neg = 0, brac = 0, last = -1;                     /* last: -1 = NONE */
    for (int i = 0; i < len; i++) {
        char ch = s[i];
        if (ch == '-' && (i == 0 || s[i - 1] == '(' || is_op(s[i - 1]))) { /* :162 */
            if (neg) return 0;
            neg = 1;
            if (!push_tok(t, T_NEG, 'N', 0)) return 0;
            continue;
        } else if (ch == '(') {
            if (last == T_VAR || last == T_NUM || last == T_BC) if (!push_tok(t, T_OP, '*', 0)) return 0;
            if (!push_tok(t, T_BO, '(', 0)) return 0;
            brac++; last = T_BO;
        } else if (ch == ')') {
            if (neg || last == T_BO || last == T_OP) return 0;
            if (brac == 0) return 0;
            if (!push_tok(t, T_BC, ')', 0)) return 0;
            brac--; last = T_BC;
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
    if (brac != 0) return 0;
    t->valid = 1;
    return 1;
}

/* ---- evaluation: Evaluator::evaluate / evaluate_op / operator_precedence / evaluate_operation,
 *      evaluator.cpp:22-136 — two stacks, no reduction on push, one-level precedence look-back ------------------- */
typedef struct {
    char ops[MAXTOK]; int nops;
    float vals[MAXTOK]; int nvals;
    int underflow;
    int pow_mode;
} Stacks;

static int prec(char c) {
    switch (c) { case 'N': return 4; case '^': return 3; case '/': case '*': return 2; case '+': case '-': return 1; default: return 0; }
}
static float apply(const Stacks* s, char op, float a, float b) { /* a (op) b, evaluator.cpp:127-136 */
    switch (op) {
        case '+': return a + b;
        case '-': return a - b;
        case '*': return a * b;
        case '/': return a / b;
        default: return s->pow_mode ? mcb_powf(a, b) : powf(a, b);
    }
}
static float popv(Stacks* s) { if (s->nvals <= 0) { s->underflow = 1; return 0.f; } return s->vals[--s->nvals]; }
static void reduce(Stacks* s) { /* evaluate_op */
    if (s->nops <= 0) { s->underflow = 1; return; }
    char op = s->ops[--s->nops];
    if (is_op(op)) {
        float val1 = popv(s);
        if (s->nops > 0 && prec(s->ops[s->nops - 1]) > prec(op)) reduce(s);
        float val2 = popv(s);
        s->vals[s->nvals++] = apply(s, op, val2, val1);
    } else if (op == 'N') {
        float v = popv(s);
        s->vals[s->nvals++] = -v;
    } else s->underflow = 1;
}
static float eval_tokens(const Tokens* t, float x, float y, float z, int pow_mode, int* underflow) {
    Stacks s; s.nops = 0; s.nvals = 0; s.underflow = 0; s.pow_mode = pow_mode;
    for (int i = 0; i < t->n; i++) {
        switch (t->type[i]) {
            case T_NEG: s.ops[s.nops++] = 'N'; break;
            case T_VAR: s.vals[s.nvals++] = t->ch[i] == 'x' ? x : t->ch[i] == 'y' ? y : z; break;
            case T_NUM: s.vals[s.nvals++] = t->num[i]; break;
            case T_BO: s.ops[s.nops++] = '('; break;
            case T_BC:
                while (s.nops > 0 && s.ops[s.nops - 1] != '(' && !s.underflow) reduce(&s);
                if (s.nops > 0) s.nops--; else s.underflow = 1;
                break;
            default: s.ops[s.nops++] = t->ch[i]; break;
        }
    }
    while (s.nops > 0 && !s.underflow) reduce(&s);
    if (s.nvals <= 0) s.underflow = 1;
    if (underflow) *underflow = s.underflow;
    return s.underflow ? 0.f : s.vals[s.nvals - 1];
}

/* ---- object ------------------------------------------------------------------------------------------------- */
static void build_axis(mco* m) { /* marching.cpp:372-377 */
    float lower = -1.0f, upper = (float)(1.0 + 0.5 * (double)m->step);
    int n = 0;
    for (float v = lower; v <= upper; v += m->step) n++;
    m->M = n;
    free(m->c); free(m->cs);
    m->c = (float*)malloc(sizeof(float) * (size_t)(n + 1));
    m->cs = (float*)malloc(sizeof(float) * (size_t)(n + 3));
    int i = 0;
    for (float v = lower; v <= upper; v += m->step) m->c[i++] = v;
    m->c[n] = m->c[n - 1] + m->step; /* x_1 = x_0 + step, marching.cpp:458 */
    m->cs[0] = m->c[0] - m->step;
    for (i = 0; i <= n; i++) m->cs[i + 1] = m->c[i];
    m->cs[n + 2] = m->c[n] + m->step;
}

mco* mco_create(void) {
    mco* m = (mco*)calloc(1, sizeof(mco));
    m->step = 0.25f; m->sx = m->sy = m->sz = 1.0f; m->iso = 0.f; /* marching.cpp:23-37 */
    tokenize("x+y", &m->eq[0]);                                   /* evaluator.cpp:6-8 */
    mcb_build_ambiguity_faces(m->face);
    build_axis(m);
    return m;
}
void mco_destroy(mco* m) { if (!m) return; free(m->c); free(m->cs); free(m->verts); free(m->tris); free(m); }
void mco_set_pow_mode(mco* m, int mode) { m->pow_mode = mode; }

int mco_parse_ok(const char* eq) {
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = tokenize(eq, t);
    if (ok) { int uf = 0; eval_tokens(t, 0.5f, 0.25f, 0.75f, 1, &uf); ok = !uf; }
    free(t);
    return ok;
}
int mco_tokenize_ok(const char* eq) {
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = tokenize(eq, t);
    free(t);
    return ok;
}
int mco_set_equation(mco* m, int slot, const char* eq) {
    if (slot < 0 || slot > 3) return 0;
    Tokens* t = (Tokens*)malloc(sizeof(Tokens));
    int ok = tokenize(eq, t);
    if (ok) { int uf = 0; eval_tokens(t, 0.5f, 0.25f, 0.75f, 1, &uf); ok = !uf; }
    if (ok) m->eq[slot] = *t;
    free(t);
    return ok;
}
float mco_evaluate(mco* m, int slot, float x, float y, float z) { return eval_tokens(&m->eq[slot], x, y, z, m->pow_mode, NULL); }
static float march_eval(const mco* m, int slot, float x, float y, float z) { /* Marching::evaluate, marching.cpp:209-224 */
    return eval_tokens(&m->eq[slot], m->sx * x, m->sy * y, m->sz * z, m->pow_mode, NULL);
}
void mco_eval_points(mco* m, int slot, const float* p, float* out, long n, int apply_scale) {
    for (long i = 0; i < n; i++)
        out[i] = apply_scale ? march_eval(m, slot, p[3 * i], p[3 * i + 1], p[3 * i + 2]) : mco_evaluate(m, slot, p[3 * i], p[3 * i + 1], p[3 * i + 2]);
}
int mco_set_step(mco* m, float step) { if (!(step > 0.f) || step > 1.f) return -1; m->step = step; build_axis(m); return m->M; }
void mco_set_scale(mco* m, float sx, float sy, float sz) { m->sx = sx; m->sy = sy; m->sz = sz; }
void mco_set_iso(mco* m, float iso) { m->iso = iso; }
/* Marching::set_surface_repeat_step_distance + repeating_surface_mode, marching.cpp:156-170 */
int mco_set_repeat(mco* m, int on, float distance) { if (on && !(distance > 0.f)) return 0; m->repeat = on != 0; if (on) m->rstep = distance; return 1; }
int mco_set_constraint(mco* m, int i, int op, float rhs, int in_use) {
    if (i < 0 || i > 2 || op < 0 || op > 3) return 0;
    m->cons[i].op = op; m->cons[i].rhs = rhs; m->cons[i].in_use = in_use;
    return 1;
}
int mco_grid(mco* m, float* coords, int cap) {
    if (coords && cap >= m->M + 1) memcpy(coords, m->c, sizeof(float) * (size_t)(m->M + 1));
    return m->M;
}

/* ---- one cube: Marching::calculate_step, marching.cpp:456-595 ------------------------------------------------ */
typedef struct {
    int code, tidx, ntri, nedges, amb, red;
    int edges[12];       /* crossing edges, ascending (edge_list) */
    float pts[12][3];    /* intersect_coord per entry of edges[] */
    int tri[15];         /* tri_vlist: local indices into pts */
    float gn[12][3];     /* gradient normal per entry of edges[] (product definition) */
} Cube;

static int check_constraints(const mco* m, float x, float y, float z) { /* marching.cpp:255-280 */
    int ok = 1;
    for (int i = 0; i < 3; i++) {
        if (!m->cons[i].in_use || !m->eq[i + 1].valid) continue;
        float lhs = march_eval(m, i + 1, x, y, z), rhs = m->cons[i].rhs;
        switch (m->cons[i].op) {
            case 2: ok &= lhs >= rhs; break;
            case 3: ok &= lhs <= rhs; break;
            case 0: ok &= lhs > rhs; break;
            default: ok &= lhs < rhs; break;
        }
    }
    return ok;
}

static float interp(const mco* m, float xs, float xe, float vs, float ve) { /* marching.cpp:437-446 */
    float v = ((m->iso - vs) / (ve - vs)) * (xe - xs);
    if (isinf(v)) return (float)((double)xs + 0.5 * (double)(xe - xs));
    if (isnan(v)) return (float)((double)xs + 0.5 * (double)(xe - xs));
    return xs + v;
}

static void calc_cube(const mco* m, int i, int j, int k, Cube* q, int want_grad) {
    const float x0 = m->c[i], y0 = m->c[j], z0 = m->c[k];
    const float x1 = x0 + m->step, y1 = y0 + m->step, z1 = z0 + m->step; /* :458-460 */
    const float cc[8][3] = {{x0, y0, z0}, {x1, y0, z0}, {x1, y1, z0}, {x0, y1, z0},
                            {x0, y0, z1}, {x1, y0, z1}, {x1, y1, z1}, {x0, y1, z1}}; /* :471-472 */
    float val[8];
    q->code = q->tidx = q->ntri = q->nedges = q->amb = q->red = 0;
    for (int v = 0; v < 8; v++) { /* :475-479 */
        if (!check_constraints(m, cc[v][0], cc[v][1], cc[v][2])) return;
        val[v] = march_eval(m, 0, cc[v][0], cc[v][1], cc[v][2]);
    }
    float level = m->iso; /* repeating-surface mode, :481-494: the cube's own level decides the code and the ambiguity test... */
    if (m->repeat) {
        float vmax = val[0];
        for (int v = 1; v < 8; v++) if (vmax < val[v]) vmax = val[v];
        float a = (vmax - m->iso) / m->rstep;
        a = floorf(a);
        level = m->iso + m->rstep * a;
    }                     /* ...while interp() below keeps using the surface constant itself (:437-446) */
    int code = 0;
    for (int v = 0; v < 8; v++) if (val[v] > level) code |= 1 << v; /* :497-505 */
    q->code = q->tidx = code;
    if (code == 0 || code == 255) return;                              /* :508-510 */
    int tidx = code;
    const int face = m->face[code];                                    /* :521-549 */
    if (face >= 0) {
        q->amb = 1;
        float mx = 0, my = 0, mz = 0;
        for (int f = 0; f < 4; f++) {
            const int vi = mcb_face_corner(face, f);
            mx += cc[vi][0]; my += cc[vi][1]; mz += cc[vi][2];
        }
        mx /= 4.0; my /= 4.0; mz /= 4.0; /* float /= double constant: exact for a power of two */
        const float mid = march_eval(m, 0, mx, my, mz);
        if (mid > level) { tidx = 255 - code; q->red = 1; }
    }
    q->tidx = tidx;
    int mapper[12];
    for (int e = 0; e < 12; e++) mapper[e] = 12;
    for (int e = 0; e < 12; e++) { /* :557-583 */
        const int a = mcb_edge_a(e), b = mcb_edge_b(e);
        if ((((code >> a) ^ (code >> b)) & 1) == 0) continue;
        const int n = q->nedges++;
        q->edges[n] = e;
        mapper[e] = n;
        q->pts[n][0] = interp(m, cc[a][0], cc[b][0], val[a], val[b]);
        q->pts[n][1] = interp(m, cc[a][1], cc[b][1], val[a], val[b]);
        q->pts[n][2] = interp(m, cc[a][2], cc[b][2], val[a], val[b]);
    }
    const uint64_t w = MCB_TRI_WORDS[tidx]; /* :586-594 */
    for (int f = 0; f < 15; f += 3) {
        const int e0 = (int)((w >> (4 * f)) & 0xF);
        if (e0 == 0xF) break;
        q->tri[f] = mapper[e0];
        q->tri[f + 1] = mapper[(w >> (4 * (f + 1))) & 0xF];
        q->tri[f + 2] = mapper[(w >> (4 * (f + 2))) & 0xF];
        q->ntri++;
    }
    if (want_grad) {
        /* Product definition of the normals (north_star "central-difference field gradients", DESIGN.md §normals):
         * gradient at each cube corner by central differences of the field over the grid coordinates, blended along the
         * grid edge (lower end point -> upper end point) with that direction's interpolation parameter, normalised like
         * glm::normalize (x * (1/sqrt(dot))). */
        float g[8][3];
        for (int v = 0; v < 8; v++) {
            const int o = mcb_corner_ofs(v);
            const int xi = i + 1 + (o & 1), yi = j + 1 + ((o >> 1) & 1), zi = k + 1 + ((o >> 2) & 1); /* cs indices */
            const float X = m->cs[xi], Y = m->cs[yi], Z = m->cs[zi];
            /* the difference times the fp32 reciprocal of the coordinate difference (one table of reciprocals per grid) */
            const float rx = 1.0f / (m->cs[xi + 1] - m->cs[xi - 1]), ry = 1.0f / (m->cs[yi + 1] - m->cs[yi - 1]), rz = 1.0f / (m->cs[zi + 1] - m->cs[zi - 1]);
            g[v][0] = (march_eval(m, 0, m->cs[xi + 1], Y, Z) - march_eval(m, 0, m->cs[xi - 1], Y, Z)) * rx;
            g[v][1] = (march_eval(m, 0, X, m->cs[yi + 1], Z) - march_eval(m, 0, X, m->cs[yi - 1], Z)) * ry;
            g[v][2] = (march_eval(m, 0, X, Y, m->cs[zi + 1]) - march_eval(m, 0, X, Y, m->cs[zi - 1])) * rz;
        }
        for (int n = 0; n < q->nedges; n++) {
            int a = mcb_edge_a(q->edges[n]), b = mcb_edge_b(q->edges[n]);
            /* the normal is defined on the grid edge: blended from its lower end point to the upper one, whichever way
             * this cube's edge runs (the up to four cubes sharing the edge get the same normal) */
            if (mcb_corner_ofs(a) > mcb_corner_ofs(b)) { const int sw = a; a = b; b = sw; }
            float t = (m->iso - val[a]) / (val[b] - val[a]);
            if (isinf(t) || isnan(t)) t = 0.5f;
            const float nx = g[a][0] + t * (g[b][0] - g[a][0]);
            const float ny = g[a][1] + t * (g[b][1] - g[a][1]);
            const float nz = g[a][2] + t * (g[b][2] - g[a][2]);
            const float inv = 1.0f / sqrtf(nx * nx + ny * ny + nz * nz);
            q->gn[n][0] = nx * inv; q->gn[n][1] = ny * inv; q->gn[n][2] = nz * inv;
        }
    }
}

/* ---- weld: add_step_to_poly_data / add_point, marching.cpp:599-643; set<xyz> with the tolerance comparator of
 *      marching.h:38-54.  std::set is a red-black tree; the comparator is not a strict weak order, so the result
 *      depends on the tree's shape — we therefore restate libstdc++'s insert-unique descent and the textbook
 *      (CLRS) rebalancing it uses, node for node. ------------------------------------------------------------------ */
typedef struct { float x, y, z; int idx; int left, right, parent; char red; } RBNode;
typedef struct { RBNode* n; int count, cap, root; } RBTree;

static int close_enough(float a, float b) { return (double)fabsf(a - b) < 0.000001; }
static int xyz_less(const RBNode* a, const RBNode* b) {
    if (!close_enough(a->x, b->x)) return a->x < b->x;
    else if (!close_enough(a->y, b->y)) return a->y < b->y;
    else if (!close_enough(a->z, b->z)) return a->z < b->z;
    return 0;
}
static void rot_left(RBTree* t, int x) {
    RBNode* n = t->n; int y = n[x].right;
    n[x].right = n[y].left; if (n[y].left >= 0) n[n[y].left].parent = x;
    n[y].parent = n[x].parent;
    if (n[x].parent < 0) t->root = y; else if (x == n[n[x].parent].left) n[n[x].parent].left = y; else n[n[x].parent].right = y;
    n[y].left = x; n[x].parent = y;
}
static void rot_right(RBTree* t, int x) {
    RBNode* n = t->n; int y = n[x].left;
    n[x].left = n[y].right; if (n[y].right >= 0) n[n[y].right].parent = x;
    n[y].parent = n[x].parent;
    if (n[x].parent < 0) t->root = y; else if (x == n[n[x].parent].right) n[n[x].parent].right = y; else n[n[x].parent].left = y;
    n[y].right = x; n[x].parent = y;
}
static int rb_prev(const RBTree* t, int x) {
    const RBNode* n = t->n;
    if (n[x].left >= 0) { x = n[x].left; while (n[x].right >= 0) x = n[x].right; return x; }
    int p = n[x].parent;
    while (p >= 0 && x == n[p].left) { x = p; p = n[p].parent; }
    return p;
}
/* returns idx of the element found or inserted (set::insert(...).first->idx) */
static int rb_insert_unique(RBTree* t, float x, float y, float z, int idx) {
    RBNode key; key.x = x; key.y = y; key.z = z; key.idx = idx;
    RBNode* n = t->n;
    int cur = t->root, parent = -1, comp = 1;
    while (cur >= 0) { parent = cur; comp = xyz_less(&key, &n[cur]); cur = comp ? n[cur].left : n[cur].right; }
    int j = parent;
    int do_insert = 0;
    if (comp) {
        /* leftmost? */
        int lm = t->root; if (lm >= 0) while (n[lm].left >= 0) lm = n[lm].left;
        if (parent < 0 || j == lm) do_insert = 1; else j = rb_prev(t, j);
    }
    if (!do_insert) { if (j >= 0 && xyz_less(&n[j], &key)) do_insert = 1; else return n[j].idx; }
    if (t->count == t->cap) { t->cap = t->cap ? t->cap * 2 : 1024; t->n = (RBNode*)realloc(t->n, sizeof(RBNode) * (size_t)t->cap); n = t->n; }
    int z_ = t->count++;
    n[z_] = key; n[z_].left = n[z_].right = -1; n[z_].parent = parent; n[z_].red = 1;
    if (parent < 0) t->root = z_;
    else if (comp) n[parent].left = z_; /* insert_left = (p == header || key < key(p)); comp is that last comparison */
    else n[parent].right = z_;
    /* rebalance */
    int c = z_;
    while (c != t->root && n[n[c].parent].red) {
        int p = n[c].parent, gp = n[p].parent;
        if (p == n[gp].left) {
            int u = n[gp].right;
            if (u >= 0 && n[u].red) { n[p].red = 0; n[u].red = 0; n[gp].red = 1; c = gp; }
            else {
                if (c == n[p].right) { c = p; rot_left(t, c); n = t->n; p = n[c].parent; gp = n[p].parent; }
                n[p].red = 0; n[gp].red = 1; rot_right(t, gp);
            }
        } else {
            int u = n[gp].left;
            if (u >= 0 && n[u].red) { n[p].red = 0; n[u].red = 0; n[gp].red = 1; c = gp; }
            else {
                if (c == n[p].left) { c = p; rot_right(t, c); n = t->n; p = n[c].parent; gp = n[p].parent; }
                n[p].red = 0; n[gp].red = 1; rot_left(t, gp);
            }
        }
    }
    n[t->root].red = 0;
    return idx;
}

static int add_point(mco* m, RBTree* t, float x, float y, float z) { /* marching.cpp:627-643 */
    int new_i = (int)m->nverts;
    int found = rb_insert_unique(t, x, y, z, new_i);
    if (found == new_i) {
        if (m->nverts == m->capv) { m->capv = m->capv ? m->capv * 2 : 4096; m->verts = (float*)realloc(m->verts, sizeof(float) * 3 * (size_t)m->capv); }
        m->verts[3 * m->nverts] = x; m->verts[3 * m->nverts + 1] = y; m->verts[3 * m->nverts + 2] = z;
        m->nverts++;
    }
    return found;
}
static void add_cube_to_mesh(mco* m, RBTree* t, const Cube* q) { /* marching.cpp:599-623 */
    int vi[12];
    for (int n = 0; n < 12; n++) vi[n] = -1;
    for (int n = 0; n < q->nedges; n++)
        if (!isnan(q->pts[n][0])) vi[n] = add_point(m, t, q->pts[n][0], q->pts[n][1], q->pts[n][2]);
    for (int f = 0; f < q->ntri; f++) { /* add_triangle, marching.cpp:646-654 */
        if (m->ntris == m->capt) { m->capt = m->capt ? m->capt * 2 : 4096; m->tris = (unsigned*)realloc(m->tris, sizeof(unsigned) * 3 * (size_t)m->capt); }
        for (int v = 0; v < 3; v++) m->tris[3 * m->ntris + v] = (unsigned)vi[q->tri[3 * f + v]];
        m->ntris++;
    }
}

/* ---- sweeps ------------------------------------------------------------------------------------------------- */
typedef struct {
    mco* m; long row0, row1; /* rows = k*M + j */
    long base_row;           /* first row of the whole sweep (for per-cube output indexing) */
    uint8_t *code, *tidx, *ntri;
    Cube* cubes; long* cube_index; /* compact list of active cubes for this worker */
    long ncubes, capcubes;
    int want_grad, keep;
    long T, A, AMB, RED;
} Job;

static void* worker(void* arg) {
    Job* jb = (Job*)arg; mco* m = jb->m; const long M = m->M;
    Cube q;
    for (long r = jb->row0; r < jb->row1; r++) {
        const int k = (int)(r / M), j = (int)(r % M);
        for (int i = 0; i < M; i++) {
            calc_cube(m, i, j, k, &q, jb->want_grad);
            const long idx = (r - jb->base_row) * M + i;
            if (jb->code) jb->code[idx] = (uint8_t)q.code;
            if (jb->tidx) jb->tidx[idx] = (uint8_t)q.tidx;
            if (jb->ntri) jb->ntri[idx] = (uint8_t)q.ntri;
            if (q.code != 0 && q.code != 255) {
                jb->A++; jb->AMB += q.amb; jb->RED += q.red; jb->T += q.ntri;
                if (jb->keep) {
                    if (jb->ncubes == jb->capcubes) {
                        jb->capcubes = jb->capcubes ? jb->capcubes * 2 : 1024;
                        jb->cubes = (Cube*)realloc(jb->cubes, sizeof(Cube) * (size_t)jb->capcubes);
                    }
                    jb->cubes[jb->ncubes++] = q;
                }
            }
        }
    }
    return NULL;
}

static long run_rows(mco* m, long row0, long nrows, int nthreads, Job** out_jobs, int* out_nj, uint8_t* code, uint8_t* tidx,
                     uint8_t* ntri, int want_grad, int keep) {
    if (nthreads < 1) nthreads = 1;
    if (nthreads > nrows) nthreads = nrows > 0 ? (int)nrows : 1;
    Job* jobs = (Job*)calloc((size_t)nthreads, sizeof(Job));
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)nthreads);
    for (int t = 0; t < nthreads; t++) {
        jobs[t].m = m; jobs[t].row0 = row0 + nrows * t / nthreads; jobs[t].row1 = row0 + nrows * (t + 1) / nthreads;
        jobs[t].base_row = row0; jobs[t].code = code; jobs[t].tidx = tidx; jobs[t].ntri = ntri;
        jobs[t].want_grad = want_grad; jobs[t].keep = keep;
        pthread_create(&th[t], NULL, worker, &jobs[t]);
    }
    long T = 0;
    for (int t = 0; t < nthreads; t++) { pthread_join(th[t], NULL); T += jobs[t].T; }
    free(th);
    *out_jobs = jobs; *out_nj = nthreads;
    return T;
}

long mco_sweep(mco* m, int k0, int k1, int nthreads, uint8_t* code, uint8_t* tidx, uint8_t* ntri, float* soup,
               float* gnrm, long cap_tris, long* n_active, long* n_amb, long* n_red) {
    if (k0 < 0) k0 = 0;
    if (k1 > m->M) k1 = m->M;
    Job* jobs; int nj;
    const int keep = (soup != NULL || gnrm != NULL);
    long T = run_rows(m, (long)k0 * m->M, (long)(k1 - k0) * m->M, nthreads, &jobs, &nj, code, tidx, ntri, gnrm != NULL, keep);
    long A = 0, AMB = 0, RED = 0, t_out = 0;
    for (int t = 0; t < nj; t++) {
        A += jobs[t].A; AMB += jobs[t].AMB; RED += jobs[t].RED;
        for (long c = 0; c < jobs[t].ncubes; c++) {
            const Cube* q = &jobs[t].cubes[c];
            for (int f = 0; f < q->ntri; f++, t_out++) {
                if (t_out >= cap_tris) continue;
                for (int v = 0; v < 3; v++) {
                    const int li = q->tri[3 * f + v];
                    if (soup) for (int a = 0; a < 3; a++) soup[9 * t_out + 3 * v + a] = q->pts[li][a];
                    if (gnrm) for (int a = 0; a < 3; a++) gnrm[9 * t_out + 3 * v + a] = q->gn[li][a];
                }
            }
        }
        free(jobs[t].cubes);
    }
    free(jobs);
    if (n_active) *n_active = A;
    if (n_amb) *n_amb = AMB;
    if (n_red) *n_red = RED;
    return T;
}

long mco_recalculate(mco* m, int nthreads) { /* Marching::recalculate full-grid branch, marching.cpp:368-384 */
    Job* jobs; int nj;
    m->nverts = 0; m->ntris = 0;
    run_rows(m, 0, (long)m->M * m->M, nthreads, &jobs, &nj, NULL, NULL, NULL, 0, 1);
    RBTree t; t.n = NULL; t.count = 0; t.cap = 0; t.root = -1;
    for (int j = 0; j < nj; j++) { /* workers hold contiguous row ranges in order: this is the loop order */
        for (long c = 0; c < jobs[j].ncubes; c++) add_cube_to_mesh(m, &t, &jobs[j].cubes[c]);
        free(jobs[j].cubes);
    }
    free(jobs); free(t.n);
    return m->ntris;
}
long mco_num_vertices(mco* m) { return m->nverts; }
long mco_num_triangles(mco* m) { return m->ntris; }
void mco_copy_mesh(mco* m, float* v, unsigned* t) {
    if (v) memcpy(v, m->verts, sizeof(float) * 3 * (size_t)m->nverts);
    if (t) memcpy(t, m->tris, sizeof(unsigned) * 3 * (size_t)m->ntris);
}

/* CalculateNormal, normal.h:3-42 with glm 0.9.5.3 cross / normalize (func_geometric.inl:217-229, 257-267;
 * inversesqrt = 1.0f/sqrt(x), func_exponential.inl:226-229). */
void mco_normals(mco* m, float* out) {
    memset(out, 0, sizeof(float) * 3 * (size_t)m->nverts);
    for (long i = 0; i < m->ntris; i++) {
        const unsigned i1 = m->tris[3 * i], i2 = m->tris[3 * i + 1], i3 = m->tris[3 * i + 2];
        const float* A = &m->verts[3 * (size_t)i1]; const float* B = &m->verts[3 * (size_t)i2]; const float* C = &m->verts[3 * (size_t)i3];
        const float bx = B[0] - A[0], by = B[1] - A[1], bz = B[2] - A[2];
        const float cx = C[0] - A[0], cy = C[1] - A[1], cz = C[2] - A[2];
        const float nx = by * cz - cy * bz, ny = bz * cx - cz * bx, nz = bx * cy - cx * by;
        const unsigned ids[3] = {i1, i2, i3};
        for (int q = 0; q < 3; q++) { /* vNormal[i] = normal + vNormal[i], in this order: a repeated index accumulates twice */
            float* o = &out[3 * (size_t)ids[q]];
            o[0] = nx + o[0]; o[1] = ny + o[1]; o[2] = nz + o[2];
        }
    }
    for (long v = 0; v < m->nverts; v++) {
        float* o = &out[3 * v];
        const float sqr = o[0] * o[0] + o[1] * o[1] + o[2] * o[2];
        const float inv = 1.0f / sqrtf(sqr);
        o[0] = o[0] * inv; o[1] = o[1] * inv; o[2] = o[2] * inv;
    }
}

double mco_timed_rows(mco* m, long row0, long nrows, int nthreads, long* cubes, long* tris) {
    const long MM = (long)m->M * m->M;
    if (row0 < 0) row0 = 0;
    if (row0 > MM) row0 = MM;
    if (row0 + nrows > MM) nrows = MM - row0;
    struct timespec a, b;
    clock_gettime(CLOCK_MONOTONIC, &a);
    Job* jobs; int nj;
    long T = run_rows(m, row0, nrows, nthreads, &jobs, &nj, NULL, NULL, NULL, 0, 0);
    clock_gettime(CLOCK_MONOTONIC, &b);
    for (int t = 0; t < nj; t++) free(jobs[t].cubes);
    free(jobs);
    if (cubes) *cubes = nrows * m->M;
    if (tris) *tris = T;
    return (double)(b.tv_sec - a.tv_sec) + 1e-9 * (double)(b.tv_nsec - a.tv_nsec);
}
