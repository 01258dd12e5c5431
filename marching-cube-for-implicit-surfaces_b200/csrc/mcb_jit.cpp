#include "mcb_jit.h"

#include <dlfcn.h>

#include <cstdio>
#include <mutex>
#include <sstream>

namespace mcbjit {
namespace {

const char* const kPowHeader =
#include "mcb_pow_src.inc" /* mcb_pow.h as a raw string literal, written by build.py: one source for nvcc and NVRTC */
    ;
const char* const kTrigHeader =
#include "mcb_trig_src.inc" /* mcb_trig.h, likewise */
    ;
const char* const kBytecodeHeader =
#include "mcb_bytecode_src.inc" /* mcb_bytecode.h, likewise: mcb_minf / mcb_maxf */
    ;

/* Everything around the generated body.  It restates the tile of eval_field_kernel (mcb_kernels.cuh): a warp owns 128
 * columns x 4 rows of one plane, a lane the columns x0 + 32 q; evict-first field stores, sign words by ballot.  The Grid
 * struct must match mcbk::Grid (checked by a static_assert against the size the host passes in as MCB_GRID_BYTES). */
const char* const kHead = R"SRC(
#include "mcb_pow.h"
struct Grid { int M, NV, P, WP, kb, ke, NZ; float sx, sy, sz, iso; int repeat; float rstep; };
static_assert(sizeof(Grid) == MCB_GRID_BYTES, "Grid layout differs from the library's");
struct Consts { float k[MCB_MAX_K]; };
__device__ __forceinline__ float op_add(float a, float b) { return __fadd_rn(a, b); }   /* never contracted into FMAs */
__device__ __forceinline__ float op_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float op_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float op_div(float a, float b) { return __fdiv_rn(a, b); }
__device__ __noinline__ float pow_call(float a, float b) { return mcb_powf(a, b); }
__device__ __forceinline__ float op_pow(float a, float b) { /* as fused_op<MCB_F_POW>: exact x^2 fast path inline, the rest out of line */
    float r;
    if (__float_as_uint(b) == 0x40000000u && mcb_pow2_try(a, &r)) return r;
    return pow_call(a, b);
}
#define R(e) ((e) >> 2)
#define Q(e) ((e) & 3)
)SRC";
/* The function grammar's operations, added to the source only when the program uses them: sin / cos out of line (one
 * copy of the fp64 restatement of glibc's sinf / cosf each), sqrt correctly rounded, abs the sign bit cleared. */
const char* const kHeadTrig = R"SRC(#include "mcb_trig.h"
__device__ __noinline__ float op_sin(float a) { return mcb_sinf(a); }
__device__ __noinline__ float op_cos(float a) { return mcb_cosf(a); }
)SRC";
const char* const kHeadSqrtAbs = R"SRC(__device__ __forceinline__ float op_sqrt(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ float op_abs(float a) { return __uint_as_float(__float_as_uint(a) & 0x7fffffffu); }
)SRC";
/* min / max: the interpreters' own mcb_minf / mcb_maxf (minimumNumber / maximumNumber), also only when used */
const char* const kHeadMinMax = R"SRC(#include "mcb_bytecode.h"
__device__ __forceinline__ float op_min(float a, float b) { return mcb_minf(a, b); }
__device__ __forceinline__ float op_max(float a, float b) { return mcb_maxf(a, b); }
)SRC";
const char* const kHeadPlane = R"SRC(
extern "C" __global__ void __launch_bounds__(128, MCB_MIN_BLOCKS)
MCB_KERNEL_NAME(const __grid_constant__ Consts C, const Grid g, const float* __restrict__ tables, float* __restrict__ F,
             unsigned int* __restrict__ S, int row_groups, int slots_per_axis) {
    const int lane = threadIdx.x & 31;
    const int cx = (int)blockIdx.x;
    const int yq = (int)blockIdx.y * 4 + (threadIdx.x >> 5);
    const int pz = (int)blockIdx.z;
    if (yq >= row_groups) return;
    const int x0 = cx * 128 + lane, y0 = yq * 4, zi = pz + g.kb;
)SRC";

const char* const kTail = R"SRC(
    const unsigned row0 = (unsigned)pz * (unsigned)g.NV + (unsigned)y0;
    float* fp = F + (size_t)row0 * g.P + x0;
    uint4* sw = reinterpret_cast<uint4*>(S + ((size_t)row0 + (lane & 3)) * g.WP + cx * 4);
#pragma unroll
    for (int r = 0; r < 4; r++) {
        if (y0 + r >= g.NV) break;
        unsigned int w[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            if (MCB_STORE_F && x0 + 32 * q < g.P) __stcs(fp + (size_t)r * g.P + 32 * q, RESULT[4 * r + q]);
            w[q] = __ballot_sync(0xffffffffu, RESULT[4 * r + q] > g.iso);
        }
        if (lane == r) *sw = make_uint4(w[0], w[1], w[2], w[3]);
    }
}
)SRC";

/* The sparse-field mode's refill (eval_blocks_kernel): a warp per listed 32 x 4 x 4 vertex block, a lane per x column
 * holding 4 rows (R) x 4 planes (Q). */
const char* const kHeadBlocks = R"SRC(
extern "C" __global__ void __launch_bounds__(128, MCB_MIN_BLOCKS)
mcb_fill_jit(const __grid_constant__ Consts C, const Grid g, const float* __restrict__ tables, float* __restrict__ F,
             unsigned int* __restrict__ S, const unsigned int* __restrict__ list /* bx | by << 8 | bz << 20 */,
             const unsigned int* __restrict__ count, int slots_per_axis) {
    const int lane = threadIdx.x & 31;
    const unsigned nwarps = gridDim.x * 4, n = *count;
    for (unsigned b = blockIdx.x * 4 + (threadIdx.x >> 5); b < n; b += nwarps) {
        const unsigned id = list[b];
        const int bx = (int)(id & 0xFFu), by = (int)((id >> 8) & 0xFFFu), bz = (int)(id >> 20);
        const int xc = bx * 32 + lane, y0 = by * 4, z0 = bz * 4 + g.kb;
)SRC";
const char* const kTailBlocks = R"SRC(
        unsigned int mine = 0; /* lane 4 r + q keeps the sign word of row r, plane q (as eval_blocks_kernel) */
#pragma unroll
        for (int e = 0; e < 16; e++) {
            const unsigned int wv = __ballot_sync(0xffffffffu, RESULT[e] > g.iso);
            if (lane == e) mine = wv;
        }
        const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
        float* fb = F + (size_t)(bz * 4) * planep + (size_t)y0 * rowp + xc;
        const int ny = min(4, g.NV - y0), nz = min(4, g.NZ - bz * 4);
        if (ny == 4 && nz == 4) { /* a whole block: sixteen 128-byte lines */
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int r = 0; r < 4; r++) fb[q * planep + r * rowp] = RESULT[4 * r + q];
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int r = 0; r < 4; r++)
                    if (q < nz && r < ny) fb[q * planep + r * rowp] = RESULT[4 * r + q];
        }
        if (lane < 16 && (lane >> 2) < ny && (lane & 3) < nz)
            S[((size_t)(bz * 4 + (lane & 3)) * g.NV + (y0 + (lane >> 2))) * g.WP + bx] = mine;
#undef RESULT
    }
}
)SRC";
struct Nvrtc {
    void* lib = nullptr;
    int (*CreateProgram)(void**, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*CompileProgram)(void*, int, const char* const*) = nullptr;
    int (*GetCUBINSize)(void*, size_t*) = nullptr;
    int (*GetCUBIN)(void*, char*) = nullptr;
    int (*GetProgramLogSize)(void*, size_t*) = nullptr;
    int (*GetProgramLog)(void*, char*) = nullptr;
    int (*DestroyProgram)(void**) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string error;
};

Nvrtc& nvrtc() {
    static Nvrtc n;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* name : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"}) {
            n.lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
            if (n.lib) break;
        }
        if (!n.lib) { n.error = "libnvrtc.so.12 not found: run-time specialisation is unavailable"; return; }
#define MCB_SYM(field, sym)                                                \
    n.field = reinterpret_cast<decltype(n.field)>(dlsym(n.lib, sym));      \
    if (!n.field) n.error = std::string("libnvrtc lacks ") + sym;
        MCB_SYM(CreateProgram, "nvrtcCreateProgram")
        MCB_SYM(CompileProgram, "nvrtcCompileProgram")
        MCB_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
        MCB_SYM(GetCUBIN, "nvrtcGetCUBIN")
        MCB_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
        MCB_SYM(GetProgramLog, "nvrtcGetProgramLog")
        MCB_SYM(DestroyProgram, "nvrtcDestroyProgram")
        MCB_SYM(GetErrorString, "nvrtcGetErrorString")
#undef MCB_SYM
    });
    return n;
}

} /* namespace */

static std::string generate_one(const uint32_t* code, int n, int kind /* 0 plane tiles (dense field), 1 listed 32 x 4 x 4 blocks */, bool* has_pow,
                                int* fns /* |= 1: sin or cos, 2: sqrt or abs, 4: min or max */, std::string* err) {
    const bool blocks = kind == 1;
    const char* const N = "16";   /* values per lane */
    const char* const I = "e";    /* their index variable */
    std::ostringstream loads, body;
    bool pow = false;
    /* operand fetches, one declaration per distinct (axis, slot): exactly the loads of eval_step / LeafOperand */
    bool seen[3][256] = {};
    auto operand = [&](uint32_t src, uint32_t arg) -> std::string { /* C expression of the operand of element e */
        char buf[64];
        if (src == MCB_SRC_K) { std::snprintf(buf, sizeof buf, "C.k[%u]", arg); return buf; }
        const int axis = (int)src - (int)MCB_SRC_TX;
        if (axis < 0 || axis > 2 || arg > 255) return std::string();
        if (!seen[axis][arg]) {
            seen[axis][arg] = true;
            char d[256];
            if (blocks) { /* per block: x is the lane's column, y the four rows, z the four planes */
                if (axis == 0)
                    std::snprintf(d, sizeof d, "    const float tx%u = __ldg(tables + (size_t)(0 * slots_per_axis + %u) * g.P + xc);\n", arg, arg);
                else if (axis == 1)
                    std::snprintf(d, sizeof d, "    const float4 vy%u = __ldg(reinterpret_cast<const float4*>(tables + (size_t)(1 * slots_per_axis + %u) * g.P + y0));\n"
                                  "    const float ty%u[4] = {vy%u.x, vy%u.y, vy%u.z, vy%u.w};\n", arg, arg, arg, arg, arg, arg, arg);
                else
                    std::snprintf(d, sizeof d, "    const float* pz%u = tables + (size_t)(2 * slots_per_axis + %u) * g.P + z0;\n"
                                  "    const float tz%u[4] = {__ldg(pz%u), __ldg(pz%u + 1), __ldg(pz%u + 2), __ldg(pz%u + 3)};\n", arg, arg, arg, arg, arg, arg, arg);
            } else if (axis == 0)
                std::snprintf(d, sizeof d, "    const float* px%u = tables + (size_t)(0 * slots_per_axis + %u) * g.P + x0;\n"
                              "    const float tx%u[4] = {__ldg(px%u), __ldg(px%u + 32), __ldg(px%u + 64), __ldg(px%u + 96)};\n", arg, arg, arg, arg, arg, arg, arg);
            else if (axis == 1)
                std::snprintf(d, sizeof d, "    const float4 vy%u = __ldg(reinterpret_cast<const float4*>(tables + (size_t)(1 * slots_per_axis + %u) * g.P + y0));\n"
                              "    const float ty%u[4] = {vy%u.x, vy%u.y, vy%u.z, vy%u.w};\n", arg, arg, arg, arg, arg, arg, arg);
            else
                std::snprintf(d, sizeof d, "    const float tz%u = __ldg(tables + (size_t)(2 * slots_per_axis + %u) * g.P + zi);\n", arg, arg);
            loads << d;
        }
        if (axis == 0) std::snprintf(buf, sizeof buf, blocks ? "tx%u" : "tx%u[Q(e)]", arg);
        else if (axis == 1) std::snprintf(buf, sizeof buf, "ty%u[R(e)]", arg);
        else std::snprintf(buf, sizeof buf, blocks ? "tz%u[Q(e)]" : "tz%u", arg);
        return buf;
    };
    std::vector<std::string> stack; /* names of the spilled accumulators (the interpreter's memory stack) */
    std::string acc;                /* name of the current accumulator array */
    int next = 0;
    auto fresh = [&] { return "v" + std::to_string(next++); };
    for (int pc = 0; pc < n; pc++) {
        const uint32_t w = code[pc], arg = MCB_FINSN_ARG(w);
        uint32_t fop = MCB_FINSN_OP(w), src = MCB_FINSN_SRC(w);
        MCB_FINSN_DECODE(fop, src);
        if (fop == MCB_F_NEG) {
            if (acc.empty()) { *err = "NEG without a value"; return std::string(); }
            const std::string t = fresh();
            body << "    float " << t << "[" << N << "];\n#pragma unroll\n    for (int " << I << " = 0; " << I << " < " << N << "; " << I << "++) " << t << "[" << I << "] = -" << acc << "[" << I << "];\n";
            acc = t;
            continue;
        }
        if (MCB_F_IS_FN(fop)) {
            if (acc.empty()) { *err = "function without a value"; return std::string(); }
            static const char* const names[] = {"op_sin", "op_cos", "op_sqrt", "op_abs"};
            *fns |= fop <= MCB_F_COS ? 1 : 2;
            const std::string t = fresh();
            body << "    float " << t << "[" << N << "];\n#pragma unroll\n    for (int " << I << " = 0; " << I << " < " << N << "; " << I << "++) " << t << "[" << I << "] = " << names[fop - MCB_F_SIN] << "(" << acc << "[" << I << "]);\n";
            acc = t;
            continue;
        }
        std::string v;
        if (src == MCB_SRC_POP) {
            if (stack.empty()) { *err = "POP from an empty stack"; return std::string(); }
            v = stack.back() + "[" + I + "]";
            stack.pop_back();
        } else {
            v = operand(src, arg);
            if (v.empty()) { *err = "operand the grid kernel does not take (raw coordinate)"; return std::string(); }
        }
        const std::string t = fresh();
        std::string expr;
        if (fop == MCB_F_LOAD || fop == MCB_F_PUSH) {
            if (fop == MCB_F_PUSH) { if (acc.empty()) { *err = "PUSH without a value"; return std::string(); } stack.push_back(acc); }
            expr = v;
        } else {
            if (acc.empty()) { *err = "operator without an accumulator"; return std::string(); }
            const std::string a = acc + "[" + I + "]";
            switch (fop) {
                case MCB_F_ADD: expr = "op_add(" + a + ", " + v + ")"; break;
                case MCB_F_SUB: expr = "op_sub(" + a + ", " + v + ")"; break;
                case MCB_F_RSUB: expr = "op_sub(" + v + ", " + a + ")"; break;
                case MCB_F_MUL: expr = "op_mul(" + a + ", " + v + ")"; break;
                case MCB_F_DIV: expr = "op_div(" + a + ", " + v + ")"; break;
                case MCB_F_RDIV: expr = "op_div(" + v + ", " + a + ")"; break;
                case MCB_F_POW: expr = "op_pow(" + a + ", " + v + ")"; pow = true; break;
                case MCB_F_RPOW: expr = "op_pow(" + v + ", " + a + ")"; pow = true; break;
                case MCB_F_MIN: expr = "op_min(" + a + ", " + v + ")"; *fns |= 4; break;
                case MCB_F_MAX: expr = "op_max(" + a + ", " + v + ")"; *fns |= 4; break;
                default: *err = "unknown operation"; return std::string();
            }
        }
        body << "    float " << t << "[" << N << "];\n#pragma unroll\n    for (int " << I << " = 0; " << I << " < " << N << "; " << I << "++) " << t << "[" << I << "] = " << expr << ";\n";
        acc = t;
    }
    if (acc.empty() || !stack.empty()) { *err = "program does not leave exactly one value"; return std::string(); }
    if (has_pow) *has_pow = pow;
    std::string src;
    src = blocks ? "" : "#define MCB_KERNEL_NAME mcb_eval_jit\n#define MCB_STORE_F 1\n";
    src += blocks ? kHeadBlocks : kHeadPlane;
    src += loads.str();
    src += body.str();
    src += "#define RESULT " + acc + "\n";
    src += blocks ? kTailBlocks : kTail;
    if (!blocks) src += "#undef RESULT\n#undef MCB_KERNEL_NAME\n#undef MCB_STORE_F\n";
    return src;
}

std::string generate(const uint32_t* code, int n, bool* has_pow, std::string* err) {
    /* one translation unit, two kernels: mcb_eval_jit (plane tiles: the whole field + signs, MCB_FIELD_DENSE) and
     * mcb_fill_jit (listed 32 x 4 x 4 vertex blocks: field + signs, the block-field mode) — one compile per equation
     * whatever mode runs later */
    std::string parts;
    int fns = 0;
    for (int kind = 0; kind < 2; kind++) {
        const std::string part = generate_one(code, n, kind, has_pow, &fns, err);
        if (part.empty()) return part;
        parts += part;
    }
    std::string out = kHead;
    if (fns & 1) out += kHeadTrig;
    if (fns & 2) out += kHeadSqrtAbs;
    if (fns & 4) out += kHeadMinMax;
    if ((fns & 1) && has_pow) *has_pow = true; /* out-of-line fp64 calls: the register budget of the powf kernels */
    return out + parts;
}

std::string compile(const std::string& source, bool pow, int grid_size, std::vector<char>* cubin) {
    Nvrtc& N = nvrtc();
    if (!N.error.empty()) return N.error;
    void* prog = nullptr;
    const char* hdr_src[] = {kPowHeader, kTrigHeader, kBytecodeHeader};
    const char* hdr_name[] = {"mcb_pow.h", "mcb_trig.h", "mcb_bytecode.h"};
    int rc = N.CreateProgram(&prog, source.c_str(), "mcb_eval_jit.cu", 3, hdr_src, hdr_name);
    if (rc != 0) return std::string("nvrtcCreateProgram: ") + N.GetErrorString(rc);
    char grid_bytes[64], max_k[64];
    std::snprintf(grid_bytes, sizeof grid_bytes, "-DMCB_GRID_BYTES=%d", grid_size);
    std::snprintf(max_k, sizeof max_k, "-DMCB_MAX_K=%d", MCB_MAX_K);
    const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "--fmad=false", "-lineinfo", "-default-device", grid_bytes, max_k,
                          pow ? "-DMCB_MIN_BLOCKS=8" : "-DMCB_MIN_BLOCKS=10"};
    rc = N.CompileProgram(prog, (int)(sizeof opts / sizeof opts[0]), opts);
    std::string log;
    size_t ls = 0;
    if (N.GetProgramLogSize(prog, &ls) == 0 && ls > 1) { log.resize(ls); N.GetProgramLog(prog, &log[0]); }
    if (rc != 0) {
        N.DestroyProgram(&prog);
        return std::string("nvrtcCompileProgram: ") + N.GetErrorString(rc) + "\n" + log;
    }
    size_t cs = 0;
    rc = N.GetCUBINSize(prog, &cs);
    if (rc == 0 && cs > 0) { cubin->resize(cs); rc = N.GetCUBIN(prog, cubin->data()); }
    N.DestroyProgram(&prog);
    if (rc != 0 || cs == 0) return std::string("nvrtcGetCUBIN: ") + (rc ? N.GetErrorString(rc) : "empty cubin");
    return std::string();
}

} /* namespace mcbjit */
