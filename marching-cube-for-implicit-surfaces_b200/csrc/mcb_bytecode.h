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
