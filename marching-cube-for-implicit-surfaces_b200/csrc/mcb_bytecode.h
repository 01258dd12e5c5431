/* Bytecode of the field evaluator: what the host lowering (mcb_lower.cpp) emits and the device interprets.
 *
 * One instruction = one 32-bit word: opcode in bits 0..7, argument in bits 8..31.  A program is a postfix
 * sequence over an operand stack; a binary opcode pops `top` then `second` and pushes
 *      second (op) top         for OP_ADD/SUB/MUL/DIV/POW
 *      top (op) second         for the reversed forms OP_RSUB/RDIV/RPOW
 * so the lowering can evaluate the operands of the reference's `val2 (op) val1` (evaluator.cpp:38-40) in either
 * order while each value keeps its role.  All arithmetic is fp32 without FMA contraction; `^` is mcb_powf.
 * The function grammar's unary operators: sin / cos are mcb_sinf / mcb_cosf (mcb_trig.h, glibc's sinf / cosf), sqrt is
 * the correctly rounded square root (sqrtf on the host, __fsqrt_rn on the device), abs clears the sign bit.
 * Its two-argument functions min / max are mcb_minf / mcb_maxf below (IEEE 754-2019 minimumNumber / maximumNumber).
 *
 * Programs travel to the kernels inside the kernel-parameter block, i.e. in the constant bank: every lane of a
 * warp executes the same instruction word, fetched with a uniform constant load.
 */
#ifndef MCB_BYTECODE_H
#define MCB_BYTECODE_H

#if !defined(__CUDACC_RTC__) /* the run-time compiled kernels include this file for mcb_minf / mcb_maxf */
#include <stdint.h>
#endif

#include "mcb_pow.h"
#include "mcb_trig.h"

enum {
    MCB_OP_END = 0,
    MCB_OP_PUSH_X,  /* scaled coordinate sx*x (marching.cpp:211) */
    MCB_OP_PUSH_Y,
    MCB_OP_PUSH_Z,
    MCB_OP_PUSH_K,  /* arg = constant-pool index (literal or folded constant subtree) */
    MCB_OP_PUSH_TX, /* arg = axis-table slot: value of a hoisted x-only subtree at this vertex's x index */
    MCB_OP_PUSH_TY,
    MCB_OP_PUSH_TZ,
    MCB_OP_ADD,
    MCB_OP_SUB,
    MCB_OP_RSUB,
    MCB_OP_MUL,
    MCB_OP_DIV,
    MCB_OP_RDIV,
    MCB_OP_POW,
    MCB_OP_RPOW,
    MCB_OP_NEG,
    MCB_OP_SIN,  /* function grammar: unary, act on the top of the stack like NEG */
    MCB_OP_COS,
    MCB_OP_SQRT,
    MCB_OP_ABS,
    MCB_OP_MIN,  /* function grammar: binary, commutative (no reversed forms) */
    MCB_OP_MAX,
    MCB_OP_COUNT
};
#define MCB_OP_IS_UNARY(op) ((op) == MCB_OP_NEG || ((op) >= MCB_OP_SIN && (op) <= MCB_OP_ABS))

#define MCB_MAX_CODE 384   /* instructions per program (a 256-char equation yields < 300) */
#define MCB_MAX_K 128      /* constant pool entries */
#define MCB_MAX_SLOTS 96   /* hoisted subtrees (constant + per-axis) */
#define MCB_MAX_STACK 24   /* operand stack depth any program may need */

#define MCB_INSN(op, arg) ((uint32_t)(op) | ((uint32_t)(arg) << 8))
#define MCB_INSN_OP(w) ((w) & 0xFFu)
#define MCB_INSN_ARG(w) ((w) >> 8)

/* A program + constant pool, passed by value as a __grid_constant__ kernel parameter (constant bank). */
typedef struct {
    int n;
    uint32_t code[MCB_MAX_CODE];
    float k[MCB_MAX_K];
} mcb_program;

#if defined(__CUDACC__)
#define MCB_BC_FN __host__ __device__ __forceinline__
#else
#define MCB_BC_FN static inline
#endif

/* min and max of the function grammar: IEEE 754-2019 minimumNumber / maximumNumber.  A NaN operand is ignored (two NaNs
 * give the canonical quiet NaN), -0 < +0, otherwise the smaller / larger operand exactly.  Both are commutative bit for
 * bit, so the lowering may order their operands freely.  Explicit compares and selects, not fminf / fmaxf: C leaves the
 * sign of a zero result of fmin to the implementation.  One source for g++, nvcc and NVRTC (mcb_jit.cpp). */
MCB_BC_FN float mcb_minf(float a, float b) {
    const int na = a != a, nb = b != b;
    if (na || nb) return na && nb ? mcb_u2f(0x7fc00000u) : na ? b : a;
    if (a == b) return mcb_u2f(mcb_f2u(a) | mcb_f2u(b)); /* equal bits, or +0 and -0: -0 */
    return a < b ? a : b;
}
MCB_BC_FN float mcb_maxf(float a, float b) {
    const int na = a != a, nb = b != b;
    if (na || nb) return na && nb ? mcb_u2f(0x7fc00000u) : na ? b : a;
    if (a == b) return mcb_u2f(mcb_f2u(a) & mcb_f2u(b)); /* equal bits, or +0 and -0: +0 */
    return a > b ? a : b;
}

MCB_BC_FN float mcb_binop(uint32_t op, float second, float top) {
    switch (op) {
        case MCB_OP_ADD: return second + top;
        case MCB_OP_SUB: return second - top;
        case MCB_OP_RSUB: return top - second;
        case MCB_OP_MUL: return second * top;
        case MCB_OP_DIV: return second / top;
        case MCB_OP_RDIV: return top / second;
        case MCB_OP_POW: return mcb_powf(second, top);
        case MCB_OP_MIN: return mcb_minf(second, top);
        case MCB_OP_MAX: return mcb_maxf(second, top);
        default: return mcb_powf(top, second); /* MCB_OP_RPOW */
    }
}

/* The function grammar's functions, fn = 0 sin, 1 cos, 2 sqrt, 3 abs.  Out of line: the scalar interpreters call it
 * rarely and should not carry the inlined fp64 trigonometry in every kernel that interprets a program. */
#if defined(__CUDACC__)
static __host__ __device__ __noinline__
#else
static
#endif
float mcb_fn(uint32_t fn, float v) {
    switch (fn) {
        case 0: return mcb_sinf(v);
        case 1: return mcb_cosf(v);
        case 2:
#if defined(__CUDA_ARCH__)
            return __fsqrt_rn(v);
#else
            return sqrtf(v);
#endif
        default: return mcb_u2f(mcb_f2u(v) & 0x7fffffffu);
    }
}

/* Plain scalar interpreter: one point, memory stack.  Used for the rare, divergent evaluations (ambiguity face
 * centres, mcb_eval_points, constant folding, axis tables); the per-vertex grid kernel has its own register-cached
 * version.  tx/ty/tz = this point's table values per slot (may be NULL when the program has no table loads). */
MCB_BC_FN float mcb_interp_scalar(const uint32_t* code, int n, const float* k, float x, float y, float z,
                                  const float* tx, const float* ty, const float* tz) {
    float st[MCB_MAX_STACK];
    int sp = 0;
    for (int pc = 0; pc < n; pc++) {
        uint32_t w = code[pc], op = MCB_INSN_OP(w), arg = MCB_INSN_ARG(w);
        switch (op) {
            case MCB_OP_PUSH_X: st[sp++] = x; break;
            case MCB_OP_PUSH_Y: st[sp++] = y; break;
            case MCB_OP_PUSH_Z: st[sp++] = z; break;
            case MCB_OP_PUSH_K: st[sp++] = k[arg]; break;
            case MCB_OP_PUSH_TX: st[sp++] = tx[arg]; break;
            case MCB_OP_PUSH_TY: st[sp++] = ty[arg]; break;
            case MCB_OP_PUSH_TZ: st[sp++] = tz[arg]; break;
            case MCB_OP_NEG: st[sp - 1] = -st[sp - 1]; break;
            case MCB_OP_SIN: case MCB_OP_COS: case MCB_OP_SQRT: case MCB_OP_ABS:
                st[sp - 1] = mcb_fn(op - MCB_OP_SIN, st[sp - 1]);
                break;
            case MCB_OP_END: pc = n; break;
            default: {
                float top = st[--sp];
                st[sp - 1] = mcb_binop(op, st[sp - 1], top);
            }
        }
    }
    return st[0];
}

/* ---- analytic normals (mcb_set_normals 3, mcb_eval_gradients) ---------------------------------------------------
 * Forward-mode differentiation of a point program: every stack entry is a dual number, a value and its three partials
 * with respect to the unscaled coordinates.  The value part runs exactly the operations of mcb_interp_scalar, so its bits
 * are those of mcb_eval_points.  The partials follow one fixed fp32 rule per operation of the equation, in the order
 * written, with a the left and b the right operand whatever stack order the lowering chose (the reversed forms swap them
 * back), so the gradient is a function of the operation graph alone:
 *      x, y, z  (sx,0,0) (0,sy,0) (0,0,sz)          constant  0
 *      a+b, a-b ga+-gb                              a*b       ga*b + a*gb
 *      a/b      (ga - q*gb) / b, q = a/b            -a        -ga
 *      a^b      gb == 0 exactly: (b * a^(b-1)) * ga, else v * (ln(a)*gb + (b/a)*ga), v = a^b, ln a = mcb_lnf(a)
 *      sin a    cos(a)*ga      cos a  (-sin(a))*ga  sqrt a    ga / (s+s), s = sqrt(a)
 *      abs a    sign bit of a set ? -ga : ga
 *      min, max the gradient of the operand whose bits equal the result; (ga+gb)*0.5f when both or neither do
 *               (symmetric, so the free operand order of min / max cannot change a bit)
 * Point programs use no axis tables. */

/* ln x for the x^y rule: mcb_powf_full's fp64 log2 times ln 2, rounded once.  NaN for x <= 0 or NaN, +inf for +inf. */
MCB_BC_FN float mcb_lnf(float x) {
    uint32_t ix = mcb_f2u(x);
    if (!(x > 0.f)) return mcb_u2f(0x7fc00000u);
    if (ix >= 0x7f800000u) return x;
    if (ix < 0x00800000u) { /* subnormal: normalised as mcb_powf_full does */
        ix = mcb_f2u(x * 8388608.0f);
        ix -= 23u << 23;
    }
    return (float)(mcb_pow_log2(ix) * mcb_u2d(0x3fe62e42fefa39efull) /* ln 2 */);
}

MCB_BC_FN float mcb_interp_grad_scalar(const uint32_t* code, int n, const float* k, float x, float y, float z,
                                       float sx, float sy, float sz, float g[3]) {
    float st[MCB_MAX_STACK], gs[MCB_MAX_STACK][3];
    int sp = 0;
    for (int pc = 0; pc < n; pc++) {
        const uint32_t w = code[pc], op = MCB_INSN_OP(w), arg = MCB_INSN_ARG(w);
        if (op == MCB_OP_END) break;
        if (op <= MCB_OP_PUSH_K) {
            st[sp] = op == MCB_OP_PUSH_X ? x : op == MCB_OP_PUSH_Y ? y : op == MCB_OP_PUSH_Z ? z : k[arg];
            gs[sp][0] = op == MCB_OP_PUSH_X ? sx : 0.f;
            gs[sp][1] = op == MCB_OP_PUSH_Y ? sy : 0.f;
            gs[sp][2] = op == MCB_OP_PUSH_Z ? sz : 0.f;
            sp++;
            continue;
        }
        if (MCB_OP_IS_UNARY(op)) {
            const float a = st[sp - 1];
            float* ga = gs[sp - 1];
            if (op == MCB_OP_NEG) {
                st[sp - 1] = -a;
                for (int c = 0; c < 3; c++) ga[c] = -ga[c];
            } else {
                const float v = mcb_fn(op - MCB_OP_SIN, a);
                st[sp - 1] = v;
                if (op == MCB_OP_SIN || op == MCB_OP_COS) {
                    const float d = op == MCB_OP_SIN ? mcb_fn(1, a) : -mcb_fn(0, a);
                    for (int c = 0; c < 3; c++) ga[c] = d * ga[c];
                } else if (op == MCB_OP_SQRT) {
                    const float d = v + v;
                    for (int c = 0; c < 3; c++) ga[c] = ga[c] / d;
                } else if (mcb_f2u(a) >> 31) {
                    for (int c = 0; c < 3; c++) ga[c] = -ga[c];
                }
            }
            continue;
        }
        const float top = st[--sp], second = st[sp - 1];
        const bool rev = op == MCB_OP_RSUB || op == MCB_OP_RDIV || op == MCB_OP_RPOW;
        const float a = rev ? top : second, b = rev ? second : top;
        float ga[3], gb[3], r[3];
        for (int c = 0; c < 3; c++) {
            ga[c] = rev ? gs[sp][c] : gs[sp - 1][c];
            gb[c] = rev ? gs[sp - 1][c] : gs[sp][c];
        }
        const float v = mcb_binop(op, second, top);
        switch (op) {
            case MCB_OP_ADD:
                for (int c = 0; c < 3; c++) r[c] = ga[c] + gb[c];
                break;
            case MCB_OP_SUB: case MCB_OP_RSUB:
                for (int c = 0; c < 3; c++) r[c] = ga[c] - gb[c];
                break;
            case MCB_OP_MUL:
                for (int c = 0; c < 3; c++) r[c] = ga[c] * b + a * gb[c];
                break;
            case MCB_OP_DIV: case MCB_OP_RDIV:
                for (int c = 0; c < 3; c++) r[c] = (ga[c] - v * gb[c]) / b;
                break;
            case MCB_OP_MIN: case MCB_OP_MAX: {
                const uint32_t iv = mcb_f2u(v);
                const bool ma = mcb_f2u(a) == iv, mb = mcb_f2u(b) == iv;
                for (int c = 0; c < 3; c++) r[c] = ma && !mb ? ga[c] : mb && !ma ? gb[c] : (ga[c] + gb[c]) * 0.5f;
                break;
            }
            default: /* POW, RPOW */
                if (gb[0] == 0.f && gb[1] == 0.f && gb[2] == 0.f) {
                    const float d = b * mcb_powf(a, b - 1.f);
                    for (int c = 0; c < 3; c++) r[c] = d * ga[c];
                } else {
                    const float la = mcb_lnf(a), ba = b / a;
                    for (int c = 0; c < 3; c++) r[c] = v * (la * gb[c] + ba * ga[c]);
                }
        }
        st[sp - 1] = v;
        for (int c = 0; c < 3; c++) gs[sp - 1][c] = r[c];
    }
    for (int c = 0; c < 3; c++) g[c] = gs[0][c];
    return st[0];
}

/* The analytic normal of a gradient: m = max |g_i|; (0,0,0) when m is 0, infinite or NaN or a component is NaN; otherwise
 * u = g/m, d = ux*ux + uy*uy + uz*uz (left to right), r = 1/sqrt(d) (correctly rounded, no rsqrt), n = u*r.  Scaling by m
 * first keeps a huge gradient (1/x near 0) a direction instead of an overflow. */
MCB_BC_FN void mcb_grad_normalise(const float g[3], float out[3]) {
    const float ax = mcb_u2f(mcb_f2u(g[0]) & 0x7fffffffu), ay = mcb_u2f(mcb_f2u(g[1]) & 0x7fffffffu),
                az = mcb_u2f(mcb_f2u(g[2]) & 0x7fffffffu);
    float m = ax > ay ? ax : ay;
    m = m > az ? m : az;
    if (g[0] != g[0] || g[1] != g[1] || g[2] != g[2] || !(m > 0.f) || mcb_f2u(m) == 0x7f800000u) {
        out[0] = out[1] = out[2] = 0.f;
        return;
    }
    const float ux = g[0] / m, uy = g[1] / m, uz = g[2] / m;
    float d = ux * ux + uy * uy;
    d = d + uz * uz;
#if defined(__CUDA_ARCH__)
    const float r = 1.f / __fsqrt_rn(d);
#else
    const float r = 1.f / sqrtf(d);
#endif
    out[0] = ux * r; out[1] = uy * r; out[2] = uz * r;
}

/* ---- fused ("accumulator") form of a grid program -----------------------------------------------------------
 * The grid kernel does not run the postfix words above directly.  mcb::fuse() (mcb_lower.cpp) rewrites them so
 * that a push which is immediately consumed by a binary operator becomes that operator's second operand:
 *      word = fop | src << 4 | arg << 8
 * The machine state is an accumulator `acc` (= the top of the operand stack, in registers) and a memory stack
 * holding the deeper levels.  `v` is the operand named by src:
 *      src X,Y,Z     scaled coordinate of the vertex            src K       constant pool entry arg
 *      src TX,TY,TZ  axis table arg at the vertex's index       src POP     pop the memory stack
 *      fop LOAD      acc = v                                    fop PUSH    spill acc to the memory stack; acc = v
 *      fop ADD, MUL  acc = acc (op) v                           fop NEG     acc = -acc  (src unused)
 *      fop SUB/DIV/POW  acc = acc (op) v                        fop RSUB/RDIV/RPOW  acc = v (op) acc
 *      fop SIN, COS, SQRT, ABS  acc = f(acc)  (src unused; the function grammar, like NEG)
 *      fop MINMAX    acc = min(acc, v), or max(acc, v) when bit 3 of the src field is set (the function grammar; src
 *                    takes only 0..7, so that bit is free, and the 4-bit op field has no room for two more ops)
 * Every fp32 operation and the role of each operand are those of the postfix program; only pushes and pops of
 * the operand stack disappear.  `x^2+y^2+z^2-0.49` (grid form TX0 TY0 TZ0 K0 - + +) becomes
 *      LOAD TZ0; SUB K0; ADD TY0; ADD TX0 — 4 words and no memory-stack traffic at all.
 */
enum { MCB_SRC_X = 0, MCB_SRC_Y, MCB_SRC_Z, MCB_SRC_K, MCB_SRC_TX, MCB_SRC_TY, MCB_SRC_TZ, MCB_SRC_POP };
enum {
    MCB_F_LOAD = 0, MCB_F_PUSH, MCB_F_ADD, MCB_F_SUB, MCB_F_RSUB, MCB_F_MUL, MCB_F_DIV, MCB_F_RDIV, MCB_F_POW,
    MCB_F_RPOW, MCB_F_NEG, MCB_F_SIN, MCB_F_COS, MCB_F_SQRT, MCB_F_ABS, MCB_F_MINMAX,
    MCB_F_MIN, MCB_F_MAX /* never in a word: what the readers decode an MCB_F_MINMAX word into (MCB_FINSN_DECODE) */
};
#define MCB_F_IS_FN(fop) ((fop) >= MCB_F_SIN && (fop) <= MCB_F_ABS)
#define MCB_SRC_MAX_BIT 8u /* src bit of an MCB_F_MINMAX word that selects max */
#define MCB_FINSN(fop, src, arg) ((uint32_t)(fop) | ((uint32_t)(src) << 4) | ((uint32_t)(arg) << 8))
#define MCB_FINSN_OP(w) ((w) & 0xFu)
#define MCB_FINSN_SRC(w) (((w) >> 4) & 0xFu)
#define MCB_FINSN_ARG(w) ((w) >> 8)
/* fop, src of a word with MCB_F_MINMAX resolved into MCB_F_MIN / MCB_F_MAX and a plain src */
#define MCB_FINSN_DECODE(fop, src)                                        \
    do {                                                                  \
        if ((fop) == MCB_F_MINMAX) {                                      \
            (fop) = ((src) & MCB_SRC_MAX_BIT) ? MCB_F_MAX : MCB_F_MIN;    \
            (src) &= ~MCB_SRC_MAX_BIT;                                    \
        }                                                                 \
    } while (0)

MCB_BC_FN float mcb_fop(uint32_t fop, float acc, float v) {
    switch (fop) {
        case MCB_F_ADD: return acc + v;
        case MCB_F_SUB: return acc - v;
        case MCB_F_RSUB: return v - acc;
        case MCB_F_MUL: return acc * v;
        case MCB_F_DIV: return acc / v;
        case MCB_F_RDIV: return v / acc;
        case MCB_F_POW: return mcb_powf(acc, v);
        case MCB_F_RPOW: return mcb_powf(v, acc);
        case MCB_F_MIN: return mcb_minf(acc, v);
        case MCB_F_MAX: return mcb_maxf(acc, v);
        default: return v; /* LOAD, PUSH */
    }
}

/* Scalar interpreter of the fused form (host-side checks of mcb::fuse(); the grid kernel has its own). */
MCB_BC_FN float mcb_interp_fused_scalar(const uint32_t* code, int n, const float* k, float x, float y, float z,
                                        const float* tx, const float* ty, const float* tz) {
    float st[MCB_MAX_STACK];
    int sp = 0;
    float acc = 0.f;
    for (int pc = 0; pc < n; pc++) {
        uint32_t w = code[pc], fop = MCB_FINSN_OP(w), src = MCB_FINSN_SRC(w), arg = MCB_FINSN_ARG(w);
        MCB_FINSN_DECODE(fop, src);
        if (fop == MCB_F_NEG) { acc = -acc; continue; }
        if (MCB_F_IS_FN(fop)) { acc = mcb_fn(fop - MCB_F_SIN, acc); continue; }
        if (fop == MCB_F_PUSH) st[sp++] = acc;
        float v;
        switch (src) {
            case MCB_SRC_X: v = x; break;
            case MCB_SRC_Y: v = y; break;
            case MCB_SRC_Z: v = z; break;
            case MCB_SRC_K: v = k[arg]; break;
            case MCB_SRC_TX: v = tx[arg]; break;
            case MCB_SRC_TY: v = ty[arg]; break;
            case MCB_SRC_TZ: v = tz[arg]; break;
            default: v = st[--sp]; break;
        }
        acc = mcb_fop(fop, acc, v);
    }
    return acc;
}

#endif /* MCB_BYTECODE_H */
