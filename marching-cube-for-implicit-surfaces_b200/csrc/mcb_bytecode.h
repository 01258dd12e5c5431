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
 * Its two-argument functions min / max are mcb_min / mcb_max below (IEEE 754-2019 minimumNumber / maximumNumber).
 * Every operation is written once, in the operator table below.
 *
 * Programs travel to the kernels inside the kernel-parameter block, i.e. in the constant bank: every lane of a
 * warp executes the same instruction word, fetched with a uniform constant load.
 */
#ifndef MCB_BYTECODE_H
#define MCB_BYTECODE_H

#if !defined(__CUDACC_RTC__) /* the run-time compiled kernels include this file for mcb_min / mcb_max */
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
#define MCB_BC_MEMBER __host__ __device__ __forceinline__
#define MCB_BC_NOINLINE static __host__ __device__ __noinline__
#else
#define MCB_BC_FN static inline
#define MCB_BC_MEMBER inline
#define MCB_BC_NOINLINE static
#endif

/* ---- the operator table ---------------------------------------------------------------------------------------------
 * Every operation of the grammar, written once for two scalar types, in one source for g++, nvcc and NVRTC (mcb_jit.cpp):
 *   float     the value that every interpreter computes, on the host and on the device;
 *   mcb_dual  a value and its three partials with respect to the unscaled coordinates (analytic normals: mcb_set_normals 3,
 *             mcb_eval_gradients).  Each dual rule computes its value with the float rule above it, so the value part of
 *             a dual evaluation has the bits of the plain one, then the partials by one fixed fp32 rule:
 *      x, y, z  (sx,0,0) (0,sy,0) (0,0,sz)          constant  0
 *      a+b, a-b ga+-gb                              a*b       ga*b + a*gb
 *      a/b      (ga - q*gb) / b, q = a/b            -a        -ga
 *      a^b      gb == 0 exactly: (b * a^(b-1)) * ga, else v * (ln(a)*gb + (b/a)*ga), v = a^b, ln a = mcb_lnf(a)
 *      sin a    cos(a)*ga      cos a  (-sin(a))*ga  sqrt a    ga / (s+s), s = sqrt(a)
 *      abs a    sign bit of a set ? -ga : ga
 *      min, max the gradient of the operand whose bits equal the result; (ga+gb)*0.5f when both or neither do
 *               (symmetric, so the free operand order of min / max cannot change a bit)
 * a is the left and b the right operand as the equation writes them: mcb_binop undoes the reversed stack forms, so a
 * gradient is a function of the operation graph alone.  All arithmetic is fp32 without FMA contraction (nvcc -fmad=false,
 * g++ -ffp-contract=off). */
struct mcb_dual {
    float v, g[3];
    mcb_dual() = default;
    MCB_BC_MEMBER explicit mcb_dual(float c) : v(c), g{0.f, 0.f, 0.f} {} /* a constant */
    MCB_BC_MEMBER mcb_dual(float c, float gx, float gy, float gz) : v(c), g{gx, gy, gz} {}
};

MCB_BC_FN mcb_dual operator+(mcb_dual a, mcb_dual b) {
    mcb_dual r;
    r.v = a.v + b.v;
    for (int c = 0; c < 3; c++) r.g[c] = a.g[c] + b.g[c];
    return r;
}
MCB_BC_FN mcb_dual operator-(mcb_dual a, mcb_dual b) {
    mcb_dual r;
    r.v = a.v - b.v;
    for (int c = 0; c < 3; c++) r.g[c] = a.g[c] - b.g[c];
    return r;
}
MCB_BC_FN mcb_dual operator*(mcb_dual a, mcb_dual b) {
    mcb_dual r;
    r.v = a.v * b.v;
    for (int c = 0; c < 3; c++) r.g[c] = a.g[c] * b.v + a.v * b.g[c];
    return r;
}
MCB_BC_FN mcb_dual operator/(mcb_dual a, mcb_dual b) {
    mcb_dual r;
    r.v = a.v / b.v;
    for (int c = 0; c < 3; c++) r.g[c] = (a.g[c] - r.v * b.g[c]) / b.v;
    return r;
}
MCB_BC_FN mcb_dual operator-(mcb_dual a) {
    mcb_dual r;
    r.v = -a.v;
    for (int c = 0; c < 3; c++) r.g[c] = -a.g[c];
    return r;
}
/* the chain rule of a function of one dual: value v, partials d * ga */
MCB_BC_FN mcb_dual mcb_chain(float v, float d, mcb_dual a) {
    mcb_dual r;
    r.v = v;
    for (int c = 0; c < 3; c++) r.g[c] = d * a.g[c];
    return r;
}

/* a^b is mcb_powf.  x^2 takes the exact fp32 fast path inline; the fp64 algorithm is out of line, one copy per module, so
 * the grid kernels keep their registers and every kernel that interprets a program does not carry it inlined. */
MCB_BC_NOINLINE float mcb_pow_call(float a, float b) { return mcb_powf(a, b); }
MCB_BC_FN float mcb_pow(float a, float b) {
    float r;
    if (mcb_f2u(b) == 0x40000000u && mcb_pow2_try(a, &r)) return r;
    return mcb_pow_call(a, b);
}
/* ln x for the a^b rule: mcb_powf_full's fp64 log2 times ln 2, rounded once.  NaN for x <= 0 or NaN, +inf for +inf. */
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
MCB_BC_FN mcb_dual mcb_pow(mcb_dual a, mcb_dual b) {
    const float v = mcb_pow(a.v, b.v);
    if (b.g[0] == 0.f && b.g[1] == 0.f && b.g[2] == 0.f) return mcb_chain(v, b.v * mcb_pow(a.v, b.v - 1.f), a);
    mcb_dual r;
    r.v = v;
    const float la = mcb_lnf(a.v), ba = b.v / a.v;
    for (int c = 0; c < 3; c++) r.g[c] = v * (la * b.g[c] + ba * a.g[c]);
    return r;
}

/* min and max: IEEE 754-2019 minimumNumber / maximumNumber.  A NaN operand is ignored (two NaNs give the canonical quiet
 * NaN), -0 < +0, otherwise the smaller / larger operand exactly.  Both are commutative bit for bit, so the lowering may
 * order their operands freely.  Explicit compares and selects, not fminf / fmaxf: C leaves the sign of a zero result of
 * fmin to the implementation.  The interval bounds (mcb_interval.h) and the run-time compiled kernels use them too. */
MCB_BC_FN float mcb_min(float a, float b) {
    const int na = a != a, nb = b != b;
    if (na || nb) return na && nb ? mcb_u2f(0x7fc00000u) : na ? b : a;
    if (a == b) return mcb_u2f(mcb_f2u(a) | mcb_f2u(b)); /* equal bits, or +0 and -0: -0 */
    return a < b ? a : b;
}
MCB_BC_FN float mcb_max(float a, float b) {
    const int na = a != a, nb = b != b;
    if (na || nb) return na && nb ? mcb_u2f(0x7fc00000u) : na ? b : a;
    if (a == b) return mcb_u2f(mcb_f2u(a) & mcb_f2u(b)); /* equal bits, or +0 and -0: +0 */
    return a > b ? a : b;
}
/* the partials of min / max, whose value is v */
MCB_BC_FN mcb_dual mcb_minmax_grad(float v, mcb_dual a, mcb_dual b) {
    mcb_dual r;
    r.v = v;
    const bool ma = mcb_f2u(a.v) == mcb_f2u(v), mb = mcb_f2u(b.v) == mcb_f2u(v);
    for (int c = 0; c < 3; c++) r.g[c] = ma && !mb ? a.g[c] : mb && !ma ? b.g[c] : (a.g[c] + b.g[c]) * 0.5f;
    return r;
}
MCB_BC_FN mcb_dual mcb_min(mcb_dual a, mcb_dual b) { return mcb_minmax_grad(mcb_min(a.v, b.v), a, b); }
MCB_BC_FN mcb_dual mcb_max(mcb_dual a, mcb_dual b) { return mcb_minmax_grad(mcb_max(a.v, b.v), a, b); }

/* sin / cos: mcb_sinf / mcb_cosf (mcb_trig.h, glibc's sinf / cosf), out of line for the reason mcb_pow_call is */
MCB_BC_NOINLINE float mcb_sin(float a) { return mcb_sinf(a); }
MCB_BC_NOINLINE float mcb_cos(float a) { return mcb_cosf(a); }
MCB_BC_FN mcb_dual mcb_sin(mcb_dual a) { return mcb_chain(mcb_sin(a.v), mcb_cos(a.v), a); }
MCB_BC_FN mcb_dual mcb_cos(mcb_dual a) { return mcb_chain(mcb_cos(a.v), -mcb_sin(a.v), a); }

/* sqrt: correctly rounded on both sides (the device spells it as the intrinsic, so no compile flag can change it) */
MCB_BC_FN float mcb_sqrt(float a) {
#if defined(__CUDA_ARCH__)
    return __fsqrt_rn(a);
#else
    return sqrtf(a);
#endif
}
MCB_BC_FN mcb_dual mcb_sqrt(mcb_dual a) {
    mcb_dual r;
    r.v = mcb_sqrt(a.v);
    const float d = r.v + r.v;
    for (int c = 0; c < 3; c++) r.g[c] = a.g[c] / d;
    return r;
}

/* abs clears the sign bit */
MCB_BC_FN float mcb_abs(float a) { return mcb_u2f(mcb_f2u(a) & 0x7fffffffu); }
MCB_BC_FN mcb_dual mcb_abs(mcb_dual a) {
    mcb_dual r = a;
    r.v = mcb_abs(a.v);
    if (mcb_f2u(a.v) >> 31)
        for (int c = 0; c < 3; c++) r.g[c] = -a.g[c];
    return r;
}

/* The postfix opcodes on the table: a binary opcode with the operand stack's second and top entries, a unary one with
 * the top */
template <typename T>
MCB_BC_FN T mcb_binop(uint32_t op, T second, T top) {
    switch (op) {
        case MCB_OP_ADD: return second + top;
        case MCB_OP_SUB: return second - top;
        case MCB_OP_RSUB: return top - second;
        case MCB_OP_MUL: return second * top;
        case MCB_OP_DIV: return second / top;
        case MCB_OP_RDIV: return top / second;
        case MCB_OP_POW: return mcb_pow(second, top);
        case MCB_OP_MIN: return mcb_min(second, top);
        case MCB_OP_MAX: return mcb_max(second, top);
        default: return mcb_pow(top, second); /* MCB_OP_RPOW */
    }
}
template <typename T>
MCB_BC_FN T mcb_unop(uint32_t op, T a) {
    switch (op) {
        case MCB_OP_NEG: return -a;
        case MCB_OP_SIN: return mcb_sin(a);
        case MCB_OP_COS: return mcb_cos(a);
        case MCB_OP_SQRT: return mcb_sqrt(a);
        default: return mcb_abs(a); /* MCB_OP_ABS */
    }
}

/* Point interpreter: one point, memory stack, on the scalar type T (never deduced: a caller's integer 0 must not turn the
 * interpreter into integer arithmetic).  tx/ty/tz = this point's table values per slot (may be NULL when the program has
 * no table loads). */
template <typename T>
MCB_BC_FN T mcb_interp_point(const uint32_t* code, int n, const float* k, T x, T y, T z,
                             const float* tx, const float* ty, const float* tz) {
    T st[MCB_MAX_STACK];
    int sp = 0;
    for (int pc = 0; pc < n; pc++) {
        uint32_t w = code[pc], op = MCB_INSN_OP(w), arg = MCB_INSN_ARG(w);
        switch (op) {
            case MCB_OP_PUSH_X: st[sp++] = x; break;
            case MCB_OP_PUSH_Y: st[sp++] = y; break;
            case MCB_OP_PUSH_Z: st[sp++] = z; break;
            case MCB_OP_PUSH_K: st[sp++] = T(k[arg]); break;
            case MCB_OP_PUSH_TX: st[sp++] = T(tx[arg]); break;
            case MCB_OP_PUSH_TY: st[sp++] = T(ty[arg]); break;
            case MCB_OP_PUSH_TZ: st[sp++] = T(tz[arg]); break;
            case MCB_OP_NEG: case MCB_OP_SIN: case MCB_OP_COS: case MCB_OP_SQRT: case MCB_OP_ABS:
                st[sp - 1] = mcb_unop(op, st[sp - 1]);
                break;
            case MCB_OP_END: pc = n; break;
            default: {
                T top = st[--sp];
                st[sp - 1] = mcb_binop(op, st[sp - 1], top);
            }
        }
    }
    return st[0];
}

/* Plain values: the rare, divergent evaluations (ambiguity face centres, mcb_eval_points, refined vertices, constant
 * folding, axis tables); the grid kernels run the fused form below. */
MCB_BC_FN float mcb_interp_scalar(const uint32_t* code, int n, const float* k, float x, float y, float z,
                                  const float* tx, const float* ty, const float* tz) {
    return mcb_interp_point<float>(code, n, k, x, y, z, tx, ty, tz);
}

/* The value of a point program at (x, y, z) (its bits are those of mcb_interp_scalar) and its gradient g with respect to
 * the unscaled coordinates, x = sx * unscaled x and so on.  Point programs use no axis tables. */
MCB_BC_FN float mcb_interp_grad_scalar(const uint32_t* code, int n, const float* k, float x, float y, float z,
                                       float sx, float sy, float sz, float g[3]) {
    const mcb_dual r = mcb_interp_point<mcb_dual>(code, n, k, mcb_dual(x, sx, 0.f, 0.f), mcb_dual(y, 0.f, sy, 0.f),
                                                  mcb_dual(z, 0.f, 0.f, sz), nullptr, nullptr, nullptr);
    for (int c = 0; c < 3; c++) g[c] = r.g[c];
    return r.v;
}

/* The analytic normal of a gradient: m = max |g_i|; (0,0,0) when m is 0, infinite or NaN or a component is NaN; otherwise
 * u = g/m, d = ux*ux + uy*uy + uz*uz (left to right), r = 1/sqrt(d) (correctly rounded, no rsqrt), n = u*r.  Scaling by m
 * first keeps a huge gradient (1/x near 0) a direction instead of an overflow. */
MCB_BC_FN void mcb_grad_normalise(const float g[3], float out[3]) {
    const float ax = mcb_abs(g[0]), ay = mcb_abs(g[1]), az = mcb_abs(g[2]);
    float m = ax > ay ? ax : ay;
    m = m > az ? m : az;
    if (g[0] != g[0] || g[1] != g[1] || g[2] != g[2] || !(m > 0.f) || mcb_f2u(m) == 0x7f800000u) {
        out[0] = out[1] = out[2] = 0.f;
        return;
    }
    const float ux = g[0] / m, uy = g[1] / m, uz = g[2] / m;
    float d = ux * ux + uy * uy;
    d = d + uz * uz;
    const float r = 1.f / mcb_sqrt(d);
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

static_assert(MCB_F_RPOW - MCB_F_ADD == MCB_OP_RPOW - MCB_OP_ADD && MCB_F_ABS - MCB_F_NEG == MCB_OP_ABS - MCB_OP_NEG,
              "fused operations ADD..RPOW and NEG..ABS follow their postfix opcodes in order");
/* One fused word on the operator table: acc = acc (op) v (acc takes the role of the stack's second entry, v of its top),
 * or v for LOAD / PUSH. */
MCB_BC_FN float mcb_fop(uint32_t fop, float acc, float v) {
    if (fop == MCB_F_LOAD || fop == MCB_F_PUSH) return v;
    return mcb_binop(fop == MCB_F_MIN ? (uint32_t)MCB_OP_MIN : fop == MCB_F_MAX ? (uint32_t)MCB_OP_MAX : fop - MCB_F_ADD + MCB_OP_ADD,
                     acc, v);
}

/* Scalar interpreter of the fused form (host-side checks of mcb::fuse(); the grid kernels run the same words through
 * mcb_fop on their register-tiled accumulators, mcb_kernels.cuh). */
MCB_BC_FN float mcb_interp_fused_scalar(const uint32_t* code, int n, const float* k, float x, float y, float z,
                                        const float* tx, const float* ty, const float* tz) {
    float st[MCB_MAX_STACK];
    int sp = 0;
    float acc = 0.f;
    for (int pc = 0; pc < n; pc++) {
        uint32_t w = code[pc], fop = MCB_FINSN_OP(w), src = MCB_FINSN_SRC(w), arg = MCB_FINSN_ARG(w);
        MCB_FINSN_DECODE(fop, src);
        if (fop == MCB_F_NEG || MCB_F_IS_FN(fop)) { acc = mcb_unop(fop - MCB_F_NEG + MCB_OP_NEG, acc); continue; }
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
