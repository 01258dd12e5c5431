/* sm_100a kernels of the polygoniser.  Included once by mcb_api.cu.
 *
 * Device data layout (one z-slab of cube layers [kb,ke), M cubes per axis, see DESIGN.md §layout):
 *   vertices carry a one-vertex apron on every side (needed by the central-difference normals and, in z, the slab
 *   halo):  NV = M+3 vertex columns per axis, vertex v in [-1, M+1] stored at index v+1;
 *   coords   cs[P]              cs[v+1] = coordinate of vertex v (host-accumulated exactly like marching.cpp:375-377)
 *   field    F[NZ][NV][P]       fp32, x fastest, row pitch P = NV rounded up to 32, NZ = (ke-kb)+3 planes
 *   signs    S[NZ][NV][WP]      1 bit per vertex: F > iso (strict, NaN -> 0; marching.cpp:497-505), WP = P/32 rounded up to 4
 *   valid    V[NZ][NV][WP]      1 bit per vertex: all constraints in use hold (marching.cpp:255-280); optional
 *   tables   T[axis][slot][P]   hoisted single-variable subtrees per grid coordinate
 *   records  R[capA] (u64)      i | j<<12 | k<<24 | code<<36 | table_idx<<44, in cube loop order
 *   trioff   O[capA] (u32)      index of the cube's first triangle
 *   pos,nrm  float4[3*capT]     triangle soup in the reference's emission order
 *   item     I[NZ-3][M][WC] u64 per 32-cube word: first record | active mask << 32 (compact -> weld, seed walk)
 *   vinfo    [capA] (u64)       per active cube: first new welded vertex | new-edge mask << 32 | on-vertex mask << 44
 *   vlist    float[3*capV], tlist u32[3*capT], vnrm float[3*capV]   the welded Poly_Data (marching.h:26-30)
 *
 * Kernels, in launch order of one mcb_polygonise (DESIGN.md §kernels has the roofline of each):
 *   K0  fold_constants, axis_tables      constant subtrees once; single-variable subtrees per grid coordinate
 *   K1  eval_field<HAS_POW>              field + sign bit-plane; warp tile 128 x 4, a lane holds a 4 x 4 patch
 *   K1b eval_constraint                  validity bit-plane of the constraints in use
 *   K2  classify<HAS_V>, compact         case codes + ambiguity redirect per tile; look-back scan + records
 *   K6  seed_*                           seed mode: component of the seed cube by monotone marking
 *   K3  emit<NORMALS>                    triangle soup, one thread per crossing edge, coalesced float4 stores
 *   K4  weld_count/scan/base/emit        the reference's welded, indexed mesh
 *   K5  nh_*                             normal.h normals on the welded mesh
 *   K8  dc_edges, dc_vertex, dc_emit     dual contouring (MCB_MESH_DC) in place of K3 / K4
 *   K7  inspect_cube                     calculate_step for one cube (step-by-step mode)
 *
 * The wait rule.  The kernels of a call follow each other on one stream, most of them launched with MCB_LAUNCH_PDL
 * (mcb_launch.h), so that a kernel's blocks are placed while its predecessor drains.  Such a kernel opens with
 * MCB_GRID_WAIT(): before it, nothing but arithmetic on the parameters and shared-memory set-up — no global load or
 * store, counters and atomics included.  The wait returns once the predecessor has completed and its writes are visible;
 * that predecessor waited for its own, so everything earlier in the call is covered too.  MCB_GRID_DEPENDENTS() right
 * after it lets the next grid be placed during this one's tail.  A kernel without the wait is launched with MCB_LAUNCH.
 */
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <type_traits>

#include "mcb_bytecode.h"
#include "mcb_interval.h"
#include "mcb_launch.h"
#include "mcb_qef.h"
#include "mcb_refine.h"
#include "mcb_tables.h"

namespace mcbk {

constexpr int kEvalThreads = 128;   /* 4 warps; each warp: one 128-column x 4-row tile of one z-plane */
constexpr int kEvalRows = 16;       /* field values per lane: a 4 x 4 patch */
constexpr int kClsThreads = 256;
constexpr int kEmitCubes = 64;      /* active cubes per emit chunk */
constexpr int kEmitThreads = 128;   /* threads working on one chunk */
constexpr int kEmitSlots = 512;     /* crossing-edge slots per chunk run */
constexpr int kEmitBlocksPerSM = 10; /* the emitter's grid is one resident wave of this many blocks per SM */

struct Grid {
    int M;        /* cubes per axis */
    int NV;       /* M + 3 */
    int P;        /* row pitch of F (floats) */
    int WP;       /* row pitch of S/V (words) */
    int kb, ke;   /* cube layers of the slab */
    int NZ;       /* (ke-kb) + 3 vertex planes */
    float sx, sy, sz;
    float iso;
    int repeat;   /* repeating-surface mode (marching.cpp:481-494): every cube takes its own iso level, see cube_iso */
    float rstep;  /* distance between the levels */
};

/* The iso value one cube is polygonised with.  Plain mode: the surface constant.  Repeating-surface mode
 * (Marching::calculate_step, marching.cpp:481-494): the highest level  c + n * step  that does not exceed the largest of
 * the cube's eight corner values — same comparison chain (a NaN corner never raises the maximum), same fp32 division,
 * floor and multiply-add order.  (i, j, k) = cube indices, k global.  The level decides the cube code and the
 * ambiguity test only: Marching::interp (marching.cpp:437-446) keeps interpolating towards the surface constant
 * itself, so in that mode the reference's crossing points are extrapolated along their edges; that is reproduced. */
__device__ __noinline__ float cube_level(const Grid& g, const float* __restrict__ F, int i, int j, int k) {
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    const float* f0 = F + (size_t)(k - g.kb + 1) * planep + (size_t)(j + 1) * rowp + (i + 1);
    float mx = __ldg(f0);
#pragma unroll
    for (int v = 1; v < 8; v++) {
        const int o = mcb_corner_ofs(v);
        const float f = __ldg(f0 + (size_t)(o >> 2) * planep + (size_t)((o >> 1) & 1) * rowp + (o & 1));
        if (mx < f) mx = f;
    }
    float a = (mx - g.iso) / g.rstep;
    a = floorf(a);
    return g.iso + g.rstep * a;
}
/* kept out of line: the plain mode pays one uniform branch for it, not its eight loads in every caller */
__device__ __forceinline__ float cube_iso(const Grid& g, const float* __restrict__ F, int i, int j, int k) {
    return g.repeat ? cube_level(g, F, i, j, k) : g.iso;
}


struct Counters {
    unsigned long long active;
    unsigned long long triangles;
    unsigned long long ambiguous;
    unsigned long long redirected;
    unsigned long long vertices; /* welded vertices (weld_scan_kernel) */
    unsigned long long seed_active, seed_triangles; /* seed mode: counts of the kept component */
    unsigned int tile_ticket;
    unsigned int error; /* 2 = 2^31 or more triangles in the slab */
    unsigned int field_blocks, amb_n; /* blocks the apron refill wrote; ambiguous cubes appended to the face-test list */
    unsigned long long nh_vertices, nh_triangles; /* what the normal.h stage works on: the mesh, or nothing when it is truncated */
    /* ---- everything above is zero before every classify pass (the call's clear, or the re-run's); what follows belongs to the evaluation stage ---- */
    unsigned int eval_blocks, eval_supers; /* block-field mode: 32 x 4 x 4 vertex blocks / 32 x 16 x 16 super-blocks the interval test could not decide */
    unsigned int emit_next, emit_done;     /* emit2: next chunk to hand out / blocks that have finished (the last one resets both) */
    unsigned long long dc_n;               /* dual contouring: active cubes the stage works on (active, capped by the records) */
};
constexpr size_t kCountersClassifyBytes = offsetof(Counters, eval_blocks);

/* ---------------------------------------------------------------------------------------------------------------
 * K0a  fold_constants: evaluate every maximal constant subtree once (same interpreter, same arithmetic as the
 *      per-point evaluation, so the folded value is bit-identical to what the reference recomputes per call).
 * K0b  axis_tables: evaluate every hoisted single-variable subtree at each grid coordinate of its axis.
 * ------------------------------------------------------------------------------------------------------------- */
struct SlotDesc {
    int begin, len; /* program inside slot_code */
    int axis;       /* -1 constant, else 0..2 */
    int index;      /* constant-pool index / table index within the axis */
};

__global__ void fold_constants_kernel(const uint32_t* __restrict__ slot_code, const SlotDesc* __restrict__ slots,
                                      int nslots, const float* kpool, float* out /* may alias kpool */) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nslots || slots[s].axis >= 0) return;
    out[slots[s].index] = mcb_interp_scalar(slot_code + slots[s].begin, slots[s].len, kpool, 0.f, 0.f, 0.f,
                                            nullptr, nullptr, nullptr);
}

__global__ void axis_tables_kernel(const uint32_t* __restrict__ slot_code, const SlotDesc* __restrict__ slots,
                                   int first_axis_slot, const float* __restrict__ kpool,
                                   const float* __restrict__ cs, int NV, int P, int max_slots_per_axis,
                                   float sx, float sy, float sz, float* __restrict__ tables) {
    int s = first_axis_slot + blockIdx.y;
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= P) return;
    SlotDesc d = slots[s];
    float scale = d.axis == 0 ? sx : d.axis == 1 ? sy : sz;
    float c = scale * cs[v < NV ? v : NV - 1]; /* Marching::evaluate scales first (marching.cpp:211) */
    float r = mcb_interp_scalar(slot_code + d.begin, d.len, kpool, c, c, c, nullptr, nullptr, nullptr);
    tables[((size_t)d.axis * max_slots_per_axis + d.index) * P + v] = r;
}

/* ---------------------------------------------------------------------------------------------------------------
 * K1  eval_field: the bytecode interpreter over the grid.
 *     A warp owns a tile of 128 consecutive x-columns x 4 consecutive y-rows of one z-plane; a lane owns 4
 *     columns, 32 apart, of each of the 4 rows (16 vertices, accumulator acc[row][x] in 16 registers).  Every lane
 *     executes the same fused instruction word (mcb_bytecode.h), fetched from the kernel-parameter block (constant
 *     bank), so there is no divergence and the cost of fetching/decoding a word is shared by 16 vertices per lane.
 *     An operator's other operand comes straight from its source: a constant-bank constant or a z-table entry (one
 *     register for all 16), an x-table (four coalesced loads: 4 values shared by the rows), a y-table (one broadcast
 *     LDG.128: 4 values shared by the columns) or, only for products of two compound subtrees, the shared-memory
 *     stack ([level][16][thread], conflict free).
 *     Outputs: a lane's four columns are x0 + 32 q, so a field store is one evict-first, fully coalesced 128-byte
 *     line per warp (the field is far larger than L2 and is only revisited around the surface), and the warp ballot
 *     of (value > iso) for column group q is sign word q of the tile row: the sign bit-plane S costs one compare
 *     and one vote per vertex and one 16-byte store per tile row.  The comparison against iso is fused here so that
 *     classification never reads the 4 B/vertex field.
 * ------------------------------------------------------------------------------------------------------------- */
struct EvalLane { /* what an operand fetch needs besides the instruction argument */
    const float* __restrict__ tables;
    int x0, y0, zi; /* the lane's first column (its others: x0 + 32 q), first of the warp's 4 rows, index into the z tables */
};
constexpr int kEvalLevel = kEvalRows * kEvalThreads; /* floats per memory-stack level (kEvalRows = 16 values per lane) */

/* One fused instruction, fully specialised on (operation, operand source): straight-line code, no inner dispatch.
 * acc[4 * r + q] = row r, column q of the lane. */
template <int FOP, int SRC, int QS>
__device__ __forceinline__ void eval_step(float (&acc)[kEvalRows], float*& sp, const uint32_t arg, const mcb_program& prog,
                                          const EvalLane& L) {
    if (FOP == MCB_F_PUSH) {
#pragma unroll
        for (int e = 0; e < kEvalRows; e++) sp[e * kEvalThreads] = acc[e];
        sp += kEvalLevel;
    }
    if (SRC == MCB_SRC_POP) {
        sp -= kEvalLevel;
#pragma unroll
        for (int e = 0; e < kEvalRows; e++) acc[e] = mcb_fop(FOP, acc[e], sp[e * kEvalThreads]);
    } else if (SRC == MCB_SRC_TY) { /* 4 rows of a y-table: 16-byte aligned, same address in every lane */
        const float4 t = __ldg(reinterpret_cast<const float4*>(L.tables + arg + L.y0));
        const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[4 * r + q] = mcb_fop(FOP, acc[4 * r + q], tv[r]);
    } else if (SRC == MCB_SRC_TX) { /* the lane's 4 columns of an x-table (the tables are padded past the last tile) */
        const float* t = L.tables + arg + L.x0;
        const float tv[4] = {__ldg(t), __ldg(t + QS), __ldg(t + 2 * QS), __ldg(t + 3 * QS)};
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[4 * r + q] = mcb_fop(FOP, acc[4 * r + q], tv[q]);
    } else { /* one value for all 16 vertices of the lane */
        const float u = SRC == MCB_SRC_K ? prog.k[arg] : __ldg(L.tables + arg + L.zi);
#pragma unroll
        for (int e = 0; e < kEvalRows; e++) acc[e] = mcb_fop(FOP, acc[e], u);
    }
}

/* A leaf operand as the 4 x 4 patch of a lane sees it: class 0 constant, 1 x-table, 2 y-table, 3 z-table */
template <int CLS, int QS>
struct LeafOperand {
    float4 v;
    __device__ __forceinline__ LeafOperand(uint32_t arg, const mcb_program& prog, const EvalLane& L) {
        if (CLS == 0) v = make_float4(prog.k[arg], 0.f, 0.f, 0.f);
        else if (CLS == 1) {
            const float* t = L.tables + arg + L.x0;
            v = make_float4(__ldg(t), __ldg(t + QS), __ldg(t + 2 * QS), __ldg(t + 3 * QS));
        }
        else if (CLS == 2) v = __ldg(reinterpret_cast<const float4*>(L.tables + arg + L.y0));
        else v = make_float4(__ldg(L.tables + arg + L.zi), 0.f, 0.f, 0.f);
    }
    __device__ __forceinline__ float at(int r, int q) const {
        const int c = CLS == 1 ? q : CLS == 2 ? r : 0;
        return c == 0 ? v.x : c == 1 ? v.y : c == 2 ? v.z : v.w;
    }
};
/* LOAD a ; op b  in one step: acc = a (op) b without first copying a into the 16 accumulator registers.  The host
 * pairs them up when it encodes the launch program (two words: handler | arg(a) << 8, then arg(b)). */
template <int FOP, int CA, int CB, int QS>
__device__ __forceinline__ void eval_pair(float (&acc)[kEvalRows], uint32_t arg_a, uint32_t arg_b, const mcb_program& prog,
                                          const EvalLane& L) {
    const LeafOperand<CA, QS> a(arg_a, prog, L);
    const LeafOperand<CB, QS> b(arg_b, prog, L);
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int q = 0; q < 4; q++) acc[4 * r + q] = mcb_fop(FOP, a.at(r, q), b.at(r, q));
}
#define MCB_HANDLER_SPILL 55 /* push the accumulator on the memory stack; the new value comes from the next (pair) word */
#define MCB_HANDLER_FN(FOP) (56 + (FOP) - MCB_F_SIN) /* sin, cos, sqrt, abs of the accumulator: 56..59 (function grammar) */
#define MCB_HANDLER_PAIR(FOP, CA, CB) (64 + ((FOP) - MCB_F_ADD) * 16 + (CA) * 4 + (CB))
/* min and max (function grammar): pairs 192..223, steps 224..233 (operand class as MCB_HANDLER's) */
#define MCB_HANDLER_MINMAX_FIRST 192
#define MCB_HANDLER_MINMAX_PAIR(FOP, CA, CB) (192 + ((FOP) - MCB_F_MIN) * 16 + (CA) * 4 + (CB))
#define MCB_HANDLER_MINMAX(FOP, CLS) (224 + ((FOP) - MCB_F_MIN) * 5 + (CLS))

/* `prog` is the fused grid program with its table operands already resolved by the host for this launch:
 * for src TX/TY/TZ the argument is the float offset of the table row inside `tables` ((axis*slots + slot) * PT),
 * so an operand fetch is one address add and one load.  Grid programs contain no raw X/Y/Z operands: bare
 * variables are axis tables too (mcb_lower.cpp).  The host also replaces the low byte of each word by a dense
 * handler number (operation * 5 + operand class), so that the dispatch is one jump table, not a compare tree. */
#define MCB_HANDLER(FOP, SRC) ((FOP) * 5 + ((SRC) == MCB_SRC_K ? 0 : (SRC) == MCB_SRC_TX ? 1 : (SRC) == MCB_SRC_TY ? 2 : (SRC) == MCB_SRC_TZ ? 3 : 4))
#define MCB_HANDLER_NEG (MCB_F_NEG * 5)
#define MCB_STEP(FOP, SRC) \
    case MCB_HANDLER(FOP, SRC): eval_step<FOP, SRC, QS>(acc, sp, arg, prog, L); break;
#define MCB_STEP_LEAF(FOP) MCB_STEP(FOP, MCB_SRC_K) MCB_STEP(FOP, MCB_SRC_TX) MCB_STEP(FOP, MCB_SRC_TY) MCB_STEP(FOP, MCB_SRC_TZ)
#define MCB_STEP_ALL(FOP) MCB_STEP_LEAF(FOP) MCB_STEP(FOP, MCB_SRC_POP)

constexpr int kEvalTileX = 128; /* columns per warp tile */
constexpr int kEvalTileY = 4;   /* rows per warp tile */
static_assert(kEvalRows == 16, "a lane carries a 4 x 4 patch");

/* The function grammar's functions on the 16 accumulators (handlers 56..59) */
__device__ __forceinline__ void eval_fn(float (&acc)[kEvalRows], uint32_t handler) {
    switch (handler) {
        case MCB_HANDLER_FN(MCB_F_SIN):
#pragma unroll
            for (int e = 0; e < kEvalRows; e++) acc[e] = mcb_sin(acc[e]);
            break;
        case MCB_HANDLER_FN(MCB_F_COS):
#pragma unroll
            for (int e = 0; e < kEvalRows; e++) acc[e] = mcb_cos(acc[e]);
            break;
        case MCB_HANDLER_FN(MCB_F_SQRT):
#pragma unroll
            for (int e = 0; e < kEvalRows; e++) acc[e] = mcb_sqrt(acc[e]);
            break;
        default: /* abs */
#pragma unroll
            for (int e = 0; e < kEvalRows; e++) acc[e] = mcb_abs(acc[e]);
            break;
    }
}

/* min / max steps and  LOAD a ; MIN b  pairs (handlers 192..233), dispatched apart from the main switch so that the
 * kernels of programs without them keep their code */
template <int QS>
__device__ __forceinline__ void eval_minmax(float (&acc)[kEvalRows], float*& sp, const uint32_t insn, const mcb_program& prog,
                                            const EvalLane& L, int& pc) {
    const uint32_t arg = MCB_FINSN_ARG(insn);
    switch (insn & 0xffu) {
#define MCB_MM_STEP(FOP, SRC, CLS) \
    case MCB_HANDLER_MINMAX(FOP, CLS): eval_step<FOP, SRC, QS>(acc, sp, arg, prog, L); break;
#define MCB_MM_STEPS(FOP) MCB_MM_STEP(FOP, MCB_SRC_K, 0) MCB_MM_STEP(FOP, MCB_SRC_TX, 1) MCB_MM_STEP(FOP, MCB_SRC_TY, 2) \
    MCB_MM_STEP(FOP, MCB_SRC_TZ, 3) MCB_MM_STEP(FOP, MCB_SRC_POP, 4)
        MCB_MM_STEPS(MCB_F_MIN) MCB_MM_STEPS(MCB_F_MAX)
#define MCB_MM_PAIR(FOP, CA, CB) \
    case MCB_HANDLER_MINMAX_PAIR(FOP, CA, CB): eval_pair<FOP, CA, CB, QS>(acc, arg, prog.code[++pc], prog, L); break;
#define MCB_MM_PAIR_B(FOP, CA) MCB_MM_PAIR(FOP, CA, 0) MCB_MM_PAIR(FOP, CA, 1) MCB_MM_PAIR(FOP, CA, 2) MCB_MM_PAIR(FOP, CA, 3)
#define MCB_MM_PAIR_AB(FOP) MCB_MM_PAIR_B(FOP, 0) MCB_MM_PAIR_B(FOP, 1) MCB_MM_PAIR_B(FOP, 2) MCB_MM_PAIR_B(FOP, 3)
        MCB_MM_PAIR_AB(MCB_F_MIN) MCB_MM_PAIR_AB(MCB_F_MAX)
#undef MCB_MM_STEP
#undef MCB_MM_STEPS
#undef MCB_MM_PAIR
#undef MCB_MM_PAIR_B
#undef MCB_MM_PAIR_AB
        default: break;
    }
}

/* The interpreter proper: runs the launch program on the lane's 16 accumulators.  QS = distance, in table entries,
 * between the lane's four class-1 operands (32 in the plane-tile kernel, 1 in the block kernel below).  HAS_FN: the
 * program uses a function (handlers 56..59); HAS_MINMAX: min or max (handlers 192..233).  Without them the kernel is
 * exactly the reference grammar's. */
template <bool HAS_POW, int QS, bool HAS_FN = false, bool HAS_MINMAX = false>
__device__ __forceinline__ void eval_run(const mcb_program& prog, const EvalLane& L, float (&acc)[kEvalRows], float* sp) {
#pragma unroll
    for (int e = 0; e < kEvalRows; e++) acc[e] = 0.f;
#pragma unroll 1
    for (int pc = 0; pc < prog.n; pc++) {
        const uint32_t insn = prog.code[pc];
        const uint32_t arg = MCB_FINSN_ARG(insn);
        switch (insn & 0xffu) {
            MCB_STEP_LEAF(MCB_F_LOAD)
            MCB_STEP_LEAF(MCB_F_PUSH)
            MCB_STEP_ALL(MCB_F_ADD)
            MCB_STEP_ALL(MCB_F_SUB)
            MCB_STEP_ALL(MCB_F_RSUB)
            MCB_STEP_ALL(MCB_F_MUL)
            MCB_STEP_ALL(MCB_F_DIV)
            MCB_STEP_ALL(MCB_F_RDIV)
#define MCB_STEP_POW(FOP, SRC) \
    case MCB_HANDLER(FOP, SRC): if (HAS_POW) eval_step<FOP, SRC, QS>(acc, sp, arg, prog, L); break;
            MCB_STEP_POW(MCB_F_POW, MCB_SRC_K) MCB_STEP_POW(MCB_F_POW, MCB_SRC_TX) MCB_STEP_POW(MCB_F_POW, MCB_SRC_TY)
            MCB_STEP_POW(MCB_F_POW, MCB_SRC_TZ) MCB_STEP_POW(MCB_F_POW, MCB_SRC_POP)
            MCB_STEP_POW(MCB_F_RPOW, MCB_SRC_K) MCB_STEP_POW(MCB_F_RPOW, MCB_SRC_TX) MCB_STEP_POW(MCB_F_RPOW, MCB_SRC_TY)
            MCB_STEP_POW(MCB_F_RPOW, MCB_SRC_TZ) MCB_STEP_POW(MCB_F_RPOW, MCB_SRC_POP)
#undef MCB_STEP_POW
#define MCB_PAIR(FOP, CA, CB) \
    case MCB_HANDLER_PAIR(FOP, CA, CB): if (HAS_POW || ((FOP) != MCB_F_POW && (FOP) != MCB_F_RPOW)) eval_pair<FOP, CA, CB, QS>(acc, arg, prog.code[++pc], prog, L); break;
#define MCB_PAIR_B(FOP, CA) MCB_PAIR(FOP, CA, 0) MCB_PAIR(FOP, CA, 1) MCB_PAIR(FOP, CA, 2) MCB_PAIR(FOP, CA, 3)
#define MCB_PAIR_AB(FOP) MCB_PAIR_B(FOP, 0) MCB_PAIR_B(FOP, 1) MCB_PAIR_B(FOP, 2) MCB_PAIR_B(FOP, 3)
            MCB_PAIR_AB(MCB_F_ADD) MCB_PAIR_AB(MCB_F_SUB) MCB_PAIR_AB(MCB_F_RSUB) MCB_PAIR_AB(MCB_F_MUL)
            MCB_PAIR_AB(MCB_F_DIV) MCB_PAIR_AB(MCB_F_RDIV) MCB_PAIR_AB(MCB_F_POW) MCB_PAIR_AB(MCB_F_RPOW)
#undef MCB_PAIR
#undef MCB_PAIR_B
#undef MCB_PAIR_AB
            case MCB_HANDLER_SPILL:
#pragma unroll
                for (int e = 0; e < kEvalRows; e++) sp[e * kEvalThreads] = acc[e];
                sp += kEvalLevel;
                break;
            default: /* MCB_F_NEG, and with HAS_FN / HAS_MINMAX the functions; both false compiles to NEG alone */
                if (HAS_MINMAX && (insn & 0xffu) >= MCB_HANDLER_MINMAX_FIRST) { eval_minmax<QS>(acc, sp, insn, prog, L, pc); break; }
                if (HAS_FN && (insn & 0xffu) != MCB_HANDLER_NEG) { eval_fn(acc, insn & 0xffu); break; }
#pragma unroll
                for (int e = 0; e < kEvalRows; e++) acc[e] = -acc[e];
                break;
        }
    }
}
#undef MCB_STEP
#undef MCB_STEP_LEAF
#undef MCB_STEP_ALL
/* MCB_HANDLER* stay defined: mcb_api.cu encodes the launch program with them */

/* K1.  STORE_F = false is the sparse-field mode (mcb_set_field_mode): only the sign bit-plane leaves the kernel and
 * eval_blocks_kernel later writes the field where the surface needs it. */
template <bool HAS_POW, bool STORE_F, bool HAS_FN = false, bool HAS_MINMAX = false> /* programs without `^` (after hoisting) get a
                        kernel without the powf paths: fewer registers; HAS_FN, HAS_MINMAX: with the function grammar's handlers */
__global__ void __launch_bounds__(kEvalThreads, HAS_POW || HAS_FN ? 8 : 10)
eval_field_kernel(const __grid_constant__ mcb_program prog, const Grid g, const float* __restrict__ tables,
                  float* __restrict__ F, uint32_t* __restrict__ S, int row_groups) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    MCB_DYNAMIC_SMEM(float, stack_smem); /* [level][16][kEvalThreads] */
    const int lane = threadIdx.x & 31;
    const int cx = (int)blockIdx.x;                                            /* 128-column tile of the row */
    const int yq = (int)blockIdx.y * (kEvalThreads / 32) + (threadIdx.x >> 5); /* 4-row group */
    const int pz = (int)blockIdx.z;                                            /* plane: vertex kb-1+pz */
    if (yq >= row_groups) return; /* whole warp exits together; the kernel has no block-wide barrier */
    EvalLane L;
    L.tables = tables;
    L.x0 = cx * kEvalTileX + lane;
    L.y0 = yq * kEvalTileY;
    L.zi = pz + g.kb;
    float acc[kEvalRows];
    eval_run<HAS_POW, 32, HAS_FN, HAS_MINMAX>(prog, L, acc, stack_smem + threadIdx.x);

    /* ---- outputs ----
     * A lane's columns are x0 + 32 q: every field store is one fully coalesced 128-byte line per warp, and the warp
     * ballot of (acc > iso) for column group q IS sign word q of the tile row — no bit gathering at all (the kernel
     * was issue-bound in its epilogue).  Strict >, NaN -> 0 (marching.cpp:497-505).  Bits of the padding columns
     * (x >= NV) are unspecified: every reader masks by cube column (column_mask) or addresses a real vertex. */
    const int x0 = L.x0, y0 = L.y0;
    const unsigned row0 = (unsigned)pz * (unsigned)g.NV + (unsigned)y0;
    float* fp = F + (size_t)row0 * g.P + x0;
    /* lane r < 4 stores the four sign words of tile row r; WP is a multiple of 4, so that is one aligned uint4 */
    uint4* sw = reinterpret_cast<uint4*>(S + ((size_t)row0 + (lane & 3)) * g.WP + cx * (kEvalTileX / 32));
#pragma unroll
    for (int r = 0; r < kEvalTileY; r++) {
        if (y0 + r >= g.NV) break; /* uniform per warp */
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int x = x0 + 32 * q;
            if (STORE_F && x < g.P) __stcs(fp + (size_t)r * g.P + 32 * q, acc[4 * r + q]); /* P is a multiple of 32: uniform per warp */
            w[q] = __ballot_sync(0xffffffffu, acc[4 * r + q] > g.iso);
        }
        if (lane == r) *sw = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

/* Sparse-field mode, second half: the field inside the listed 32 x 4 x 4 vertex blocks (x, y, plane), i.e. around
 * the active cubes.  Same interpreter, same arithmetic per vertex as eval_field_kernel, hence the same bits; a lane
 * is one x column and holds 4 rows x 4 planes, so the host swaps the operand classes of the x and z tables when it
 * encodes this kernel's launch program (class 1 = z, stride 1; class 2 = y; class 3 = x, per lane). */
constexpr int kFieldBlockX = 32, kFieldBlockY = 4, kFieldBlockZ = 4;
/* a block on a list: bx | by << 8 | bz << 20 (bx <= 129, by, bz <= 1025 for M <= 4094): no divisions to unpack */
__device__ __forceinline__ uint32_t pack_block(int bx, int by, int bz) { return (uint32_t)bx | ((uint32_t)by << 8) | ((uint32_t)bz << 20); }
struct FieldBlocks {
    int nbx, nby, nbz;            /* blocks per axis: P/32, ceil(NV/4), ceil(NZ/4) */
    uint8_t* flags;               /* [nbz][nby][nbx] */
    uint32_t* list;               /* flagged blocks, any order */
};
template <bool HAS_POW, bool HAS_FN = false, bool HAS_MINMAX = false>
__global__ void __launch_bounds__(kEvalThreads, HAS_POW || HAS_FN ? 8 : 10)
eval_blocks_kernel(const __grid_constant__ mcb_program prog, const Grid g, const float* __restrict__ tables,
                   float* __restrict__ F, uint32_t* __restrict__ S, const uint32_t* __restrict__ list /* pack_block */,
                   const unsigned* __restrict__ count) {
    MCB_DYNAMIC_SMEM(float, stack_smem);
    const int lane = threadIdx.x & 31;
    const unsigned nwarps = gridDim.x * (kEvalThreads / 32);
    const unsigned n = *count;
    for (unsigned b = blockIdx.x * (kEvalThreads / 32) + (threadIdx.x >> 5); b < n; b += nwarps) {
        const uint32_t id = list[b];
        const int bx = (int)(id & 0xFFu), by = (int)((id >> 8) & 0xFFFu), bz = (int)(id >> 20);
        EvalLane L;
        L.tables = tables;
        L.x0 = bz * kFieldBlockZ + g.kb; /* class 1: the z tables, consecutive planes */
        L.y0 = by * kFieldBlockY;        /* class 2: the y tables */
        L.zi = bx * kFieldBlockX + lane; /* class 3: the x tables, this lane's column */
        float acc[kEvalRows];
        eval_run<HAS_POW, 1, HAS_FN, HAS_MINMAX>(prog, L, acc, stack_smem + threadIdx.x);
        uint32_t mine = 0; /* lane 4 r + q keeps the sign word of row r, plane q: bit = this column's value > iso */
#pragma unroll
        for (int e = 0; e < kEvalRows; e++) {
            const uint32_t wv = __ballot_sync(0xffffffffu, acc[e] > g.iso);
            if (lane == e) mine = wv;
        }
        const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
        float* fb = F + (size_t)(bz * kFieldBlockZ) * planep + (size_t)L.y0 * rowp + L.zi;
        const int ny = min(kFieldBlockY, g.NV - L.y0), nz = min(kFieldBlockZ, g.NZ - bz * kFieldBlockZ); /* uniform per warp */
        if (ny == kFieldBlockY && nz == kFieldBlockZ) { /* a whole block: sixteen 128-byte lines */
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int r = 0; r < 4; r++) fb[q * planep + r * rowp] = acc[4 * r + q];
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int r = 0; r < 4; r++)
                    if (q < nz && r < ny) fb[q * planep + r * rowp] = acc[4 * r + q];
        }
        if (lane < kEvalRows && (lane >> 2) < ny && (lane & 3) < nz)
            S[((size_t)(bz * kFieldBlockZ + (lane & 3)) * g.NV + (L.y0 + (lane >> 2))) * g.WP + bx] = mine;
    }
}

/* flags == 1 -> list of the flagged, not yet evaluated block ids (any order).  A thread takes 16 flags (one 16-byte load; the flag array is padded
 * and zero-filled to a multiple of 16), a warp reserves its entries with one atomic. */
__global__ void __launch_bounds__(256)
field_list_kernel(const FieldBlocks fb, unsigned nblocks, Counters* __restrict__ ctr) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const unsigned g16 = blockIdx.x * blockDim.x + threadIdx.x; /* group of 16 flags */
    const int lane = threadIdx.x & 31;
    uint4 f = make_uint4(0u, 0u, 0u, 0u);
    if (g16 * 16u < nblocks) f = __ldg(reinterpret_cast<const uint4*>(fb.flags) + g16);
    const uint32_t w[4] = {f.x, f.y, f.z, f.w};
    uint32_t bits = 0; /* bit i = flag 16 * g16 + i */
#pragma unroll
    for (int q = 0; q < 4; q++)
#pragma unroll
        for (int b = 0; b < 4; b++) bits |= ((w[q] >> (8 * b)) & 0xffu) == 1u ? 1u << (4 * q + b) : 0u;
    const uint32_t mine = (uint32_t)__popc(bits);
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
    const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
    if (total == 0) return;
    unsigned base = 0;
    if (lane == 31) base = atomicAdd(&ctr->field_blocks, total);
    base = __shfl_sync(0xffffffffu, base, 31) + (inc - mine);
    while (bits) {
        const int i = __ffs(bits) - 1;
        bits &= bits - 1;
        const unsigned id = g16 * 16u + (unsigned)i, plane = (unsigned)fb.nbx * (unsigned)fb.nby, bz = id / plane, rem = id - bz * plane;
        fb.list[base++] = pack_block((int)(rem % (unsigned)fb.nbx), (int)(rem / (unsigned)fb.nbx), (int)bz);
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K1 (block-field mode, the default of the drop-in): decide, evaluate, skip.
 *   axis_bounds    minimum and maximum of every axis table over each block of its axis, at two levels: the 32 x 4 x 4
 *                  vertex blocks and the 32 x 16 x 16 super-blocks (1 x 4 x 4 blocks).  A block's range is EXTENDED by
 *                  one vertex at its far end on every axis, so the boxes of neighbouring blocks share vertices: two
 *                  neighbouring blocks that are both decided are decided with the same sign;
 *   super_class    one thread per super-block runs the fused grid program on those intervals (mcb_interval.h: an exact
 *                  proof, rounding included): 1 = no vertex above iso, 2 = every vertex above iso, 0 = undecided;
 *   block_class    one thread per block: the super-block's verdict, or its own interval evaluation when that was
 *                  undecided.  An undecided block goes on the evaluation list (eval_blocks_kernel / mcb_fill_jit turn it
 *                  into field values and sign words) and marks the (up to) eight 32 x 4 x 4 CUBE blocks whose corners
 *                  reach into it as candidates; classify looks nowhere else, because a cube block that touches decided
 *                  blocks only sees one sign (the shared vertices above);
 *   decided_signs  the decided neighbours of the undecided blocks — the only decided blocks classify reads sign words
 *                  of — get their sixteen constant words written.
 * The work of a polygonisation is then proportional to the surface, not to the grid, for any equation — no earlier
 * run of the same configuration is needed to find that out.
 * ------------------------------------------------------------------------------------------------------------- */
struct BlockDims {
    int nbx, nby, nbz; /* vertex blocks per axis: P/32, ceil(NV/4), ceil(NZ/4) */
    int nsy, nsz;      /* super-blocks per axis in y and z: ceil(nby/4), ceil(nbz/4) */
    int nb;            /* max(nbx, nby, nbz): stride of both bounds arrays */
    int spa;           /* table slots per axis */
    int WC, cjb, ckb;  /* cube blocks: words per row, ceil(M/4), ceil(layers/4) */
};
constexpr int kSuper = 4; /* blocks per super-block in y and z */
__global__ void __launch_bounds__(128)
axis_bounds_kernel(const float* __restrict__ tables, const Grid g, const BlockDims bd, int nsx, int nsy, int nsz,
                   mcb_ival* __restrict__ B /* [2][3][spa][nb]: level 0 blocks, level 1 super-blocks */) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int level = blockIdx.y;
    if (idx >= 3 * bd.spa * bd.nb) return;
    const int b = idx % bd.nb, slot = (idx / bd.nb) % bd.spa, axis = idx / (bd.nb * bd.spa);
    const int ns = axis == 0 ? nsx : axis == 1 ? nsy : nsz;
    const int nbk = axis == 0 ? bd.nbx : axis == 1 ? (level ? bd.nsy : bd.nby) : (level ? bd.nsz : bd.nbz);
    if (slot >= ns || b >= nbk) return;
    const int span = axis == 0 ? kFieldBlockX : (level ? kSuper : 1) * (axis == 1 ? kFieldBlockY : kFieldBlockZ);
    const int count = axis == 0 ? g.P : axis == 1 ? g.NV : g.NZ; /* table entries that exist on this axis */
    const int i0 = b * span, i1 = min(i0 + span + 1, count);      /* one past the block: the shared vertex */
    const float* t = tables + ((size_t)axis * bd.spa + slot) * g.P + (axis == 2 ? g.kb : 0); /* plane pz is entry kb + pz */
    float lo = __ldg(t + i0), hi = lo;
    bool ok = mcb_iv_finite(lo) != 0;
    for (int i = i0 + 1; i < i1; i++) {
        const float v = __ldg(t + i);
        ok = ok && mcb_iv_finite(v);
        lo = v < lo ? v : lo;
        hi = v > hi ? v : hi;
    }
    mcb_ival r;
    r.lo = ok ? lo : -INFINITY;
    r.hi = ok ? hi : INFINITY;
    B[(size_t)level * 3 * bd.spa * bd.nb + idx] = r;
}

/* Class of a block as its readers see it: the explicit byte, or — 0xFF, a block of a decided super-block, which the fine
 * pass never visits — the super-block's verdict.  Bit 2 = "its constant sign words are written". */
constexpr uint8_t kClsInherit = 0xFF;
__device__ __forceinline__ int block_class_of(const uint8_t* __restrict__ cls, const uint8_t* __restrict__ scls, const BlockDims& bd,
                                              int bx, int by, int bz) {
    const int c = (int)cls[((size_t)bz * bd.nby + by) * bd.nbx + bx];
    return c != kClsInherit ? c : (int)scls[((size_t)(bz / kSuper) * bd.nsy + by / kSuper) * bd.nbx + bx];
}

__global__ void __launch_bounds__(128)
super_class_kernel(const __grid_constant__ mcb_program prog /* fused grid program, slot numbers as arguments */, const Grid g,
                   const BlockDims bd, const mcb_ival* __restrict__ B, int decide /* 0: everything is "undecided" (tests) */,
                   uint8_t* __restrict__ scls, uint32_t* __restrict__ slist, Counters* __restrict__ ctr) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const unsigned n = (unsigned)bd.nbx * (unsigned)bd.nsy * (unsigned)bd.nsz;
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int c = 0;
    if (idx < n) {
        const int bx = (int)(idx % (unsigned)bd.nbx), sy = (int)(idx / (unsigned)bd.nbx % (unsigned)bd.nsy), sz = (int)(idx / ((unsigned)bd.nbx * (unsigned)bd.nsy));
        if (decide) c = mcb_interval_class(prog.code, prog.n, prog.k, B + (size_t)3 * bd.spa * bd.nb, bd.spa, bd.nb, bx, sy, sz, g.iso, nullptr);
        scls[idx] = (uint8_t)c;
    }
    /* the undecided super-blocks are what the fine pass looks at: a warp reserves its list entries with one atomic */
    const bool undecided = idx < n && c == 0;
    const uint32_t m = __ballot_sync(0xffffffffu, undecided);
    if (m == 0u) return;
    unsigned base = 0;
    if (lane == __ffs(m) - 1) base = atomicAdd(&ctr->eval_supers, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (undecided) slist[base + __popc(m & ((1u << lane) - 1u))] = idx;
}

/* The fine pass: sixteen threads per undecided super-block, one per block. */
__global__ void __launch_bounds__(256)
block_class_kernel(const __grid_constant__ mcb_program prog, const Grid g, const BlockDims bd, const mcb_ival* __restrict__ B,
                   const uint32_t* __restrict__ slist, int decide, uint8_t* __restrict__ cls /* preset to kClsInherit */,
                   uint8_t* __restrict__ flags /* preset to 0 */, uint32_t* __restrict__ list,
                   unsigned long long* __restrict__ cand /* preset to 0: one bit per cube block, cmw words per (layer group, row group) */,
                   Counters* __restrict__ ctr) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const unsigned nsuper = ctr->eval_supers;
    const int lane = threadIdx.x & 31;
    const unsigned stride = gridDim.x * blockDim.x;
    /* neighbouring threads take the same block position in neighbouring super-blocks (the list is close to x-fastest
     * order), so the undecided blocks a warp appends are neighbours in x and the evaluation kernel's warps, which take
     * consecutive list entries, write runs of adjacent 128-byte lines: DRAM pages stay open on dense surfaces */
    const unsigned npad = (nsuper + 31u) & ~31u, total = npad * 16u; /* whole warps stay in the loop: the ballot below needs them */
    const int cmw = (bd.WC + 63) / 64;
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        const unsigned sub = t / npad, si = t - sub * npad;
        bool undecided = false;
        int bx = 0, by = 0, bz = 0;
        if (si < nsuper) {
            const unsigned sidx = slist[si];
            bx = (int)(sidx % (unsigned)bd.nbx);
            by = (int)(sidx / (unsigned)bd.nbx % (unsigned)bd.nsy) * kSuper + (int)(sub & 3u);
            bz = (int)(sidx / ((unsigned)bd.nbx * (unsigned)bd.nsy)) * kSuper + (int)(sub >> 2);
            if (by < bd.nby && bz < bd.nbz) {
                const int c = decide ? mcb_interval_class(prog.code, prog.n, prog.k, B, bd.spa, bd.nb, bx, by, bz, g.iso, nullptr) : 0;
                const size_t id = ((size_t)bz * bd.nby + by) * bd.nbx + bx;
                cls[id] = (uint8_t)c;
                undecided = c == 0;
                if (undecided) flags[id] = 2; /* 2 = on the evaluation list; compact_kernel turns the apron blocks' 0 into 1 */
            }
        }
        const uint32_t m = __ballot_sync(0xffffffffu, undecided);
        if (m == 0u) continue;
        unsigned base = 0;
        if (lane == __ffs(m) - 1) base = atomicAdd(&ctr->eval_blocks, (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (!undecided) continue;
        list[base + __popc(m & ((1u << lane) - 1u))] = pack_block(bx, by, bz);
        /* cube (i, j, kz) reads the stored vertices (i+1..i+2, j+1..j+2, kz+1..kz+2): the cube blocks reaching into this
         * vertex block are (bx-1..bx, by-1..by, bz-1..bz) */
#pragma unroll
        for (int d = 0; d < 4; d++) {
            const int jb = by - (d & 1), kq = bz - (d >> 1);
            if (jb < 0 || kq < 0 || jb >= bd.cjb || kq >= bd.ckb) continue;
            unsigned long long* row = cand + ((size_t)kq * bd.cjb + jb) * cmw;
            /* neighbouring blocks set the same bits: look before the atomic */
            if (bx < bd.WC && !((*(volatile unsigned long long*)(row + (bx >> 6)) >> (bx & 63)) & 1ull)) atomicOr(row + (bx >> 6), 1ull << (bx & 63));
            if (bx >= 1 && bx - 1 < bd.WC && !((*(volatile unsigned long long*)(row + ((bx - 1) >> 6)) >> ((bx - 1) & 63)) & 1ull))
                atomicOr(row + ((bx - 1) >> 6), 1ull << ((bx - 1) & 63));
        }
    }
}

/* sign words of a decided block: sixteen constants, written by sixteen lanes (lane = 4 r + q: row r, plane q) */
__device__ __forceinline__ void write_decided_signs(const Grid& g, uint32_t* __restrict__ S, int bx, int by, int bz, int c, int lane16) {
    const int y = by * kFieldBlockY + (lane16 >> 2), pz = bz * kFieldBlockZ + (lane16 & 3);
    if (y < g.NV && pz < g.NZ) S[((size_t)pz * g.NV + y) * g.WP + bx] = (c & 3) == 2 ? 0xffffffffu : 0u;
}
/* A warp per undecided block: its 26 neighbours are probed by 26 lanes; those that are decided and whose words nobody has
 * written yet (bit 2 of the class byte remembers; two warps racing store the same words) are then written one after the
 * other by sixteen lanes each.  These are all the decided blocks a candidate cube block can reach into. */
__global__ void __launch_bounds__(256)
decided_signs_kernel(const Grid g, const BlockDims bd, const uint32_t* __restrict__ list, const Counters* __restrict__ ctr,
                     uint8_t* __restrict__ cls, const uint8_t* __restrict__ scls, uint32_t* __restrict__ S) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const unsigned n = ctr->eval_blocks;
    const int lane = threadIdx.x & 31;
    const unsigned nwarps = gridDim.x * (blockDim.x >> 5);
    for (unsigned b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); b < n; b += nwarps) {
        const uint32_t id = list[b];
        const int bx = (int)(id & 0xFFu) + lane % 3 - 1, by = (int)((id >> 8) & 0xFFFu) + (lane / 3) % 3 - 1, bz = (int)(id >> 20) + lane / 9 - 1;
        int c = 0;
        if (lane < 27 && lane != 13 && bx >= 0 && by >= 0 && bz >= 0 && bx < bd.nbx && by < bd.nby && bz < bd.nbz) {
            /* claim the block, so that exactly one warp writes its words: its class byte becomes explicit, class | 4, by a
             * compare-and-swap on the 32-bit word that holds it (the byte is kClsInherit, 1 or 2 while unclaimed) */
            const size_t bid = ((size_t)bz * bd.nby + by) * bd.nbx + bx;
            unsigned* word = reinterpret_cast<unsigned*>(cls + (bid & ~(size_t)3));
            const unsigned sh = (unsigned)(bid & 3) * 8u;
            for (;;) {
                const unsigned w = *(volatile unsigned*)word, b8 = (w >> sh) & 0xFFu;
                const int cur = b8 == kClsInherit ? (int)scls[((size_t)(bz / kSuper) * bd.nsy + by / kSuper) * bd.nbx + bx] : (int)b8;
                if (cur == 0 || (b8 != kClsInherit && (b8 & 4u))) { c = 0; break; }   /* undecided, or somebody else has it */
                if (atomicCAS(word, w, (w & ~(0xFFu << sh)) | ((unsigned)(cur | 4) << sh)) == w) { c = cur; break; }
            }
        }
        uint32_t todo = __ballot_sync(0xffffffffu, c != 0);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int nx = __shfl_sync(0xffffffffu, bx, src), ny = __shfl_sync(0xffffffffu, by, src), nz = __shfl_sync(0xffffffffu, bz, src);
            const int nc = __shfl_sync(0xffffffffu, c, src);
            if (lane < 16) write_decided_signs(g, S, nx, ny, nz, nc, lane);
        }
    }
}
/* tri_list of a slab shifted to its place in a mesh assembled from several slabs: index += delta (mcb_set_index_base) */
__global__ void __launch_bounds__(256)
add_index_base_kernel(uint32_t* __restrict__ tri_list, unsigned long long n, uint32_t delta) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) tri_list[q] += delta;
}

/* the parity hook mcb_get_cases reads every sign word: write those of all decided blocks */
__global__ void __launch_bounds__(256)
decided_signs_all_kernel(const Grid g, const BlockDims bd, uint8_t* __restrict__ cls, const uint8_t* __restrict__ scls, uint32_t* __restrict__ S) {
    const unsigned nblocks = (unsigned)bd.nbx * (unsigned)bd.nby * (unsigned)bd.nbz;
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nblocks) return;
    const int bx = (int)(idx % (unsigned)bd.nbx), by = (int)(idx / (unsigned)bd.nbx % (unsigned)bd.nby), bz = (int)(idx / ((unsigned)bd.nbx * (unsigned)bd.nby));
    const int c = block_class_of(cls, scls, bd, bx, by, bz);
    if (c == 0 || (c & 4)) return;
    cls[idx] = (uint8_t)(c | 4);
#pragma unroll
    for (int l = 0; l < 16; l++) write_decided_signs(g, S, bx, by, bz, c, l);
}

/* K1b  constraint validity bit-plane: V &= (lhs(sx*x,sy*y,sz*z) op rhs), one launch per constraint in use. */
__global__ void __launch_bounds__(256)
eval_constraint_kernel(const __grid_constant__ mcb_program prog, const Grid g, const float* __restrict__ cs,
                       int op, float rhs, int first, uint32_t* __restrict__ V, long long total_words) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const int lane = threadIdx.x & 31;
    const long long widx = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (widx >= total_words) return;
    const int w = (int)(widx % g.WP);
    const long long row = widx / g.WP;
    const int y = (int)(row % g.NV);
    const int pz = (int)(row / g.NV);
    const int x = w * 32 + lane;
    bool ok = false;
    if (x < g.NV) {
        float v = mcb_interp_scalar(prog.code, prog.n, prog.k, g.sx * cs[x], g.sy * cs[y], g.sz * cs[pz + g.kb],
                                    nullptr, nullptr, nullptr);
        ok = op == 0 ? v > rhs : op == 1 ? v < rhs : op == 2 ? v >= rhs : v <= rhs;
    }
    unsigned bits = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) V[widx] = first ? bits : (V[widx] & bits);
}

/* ---------------------------------------------------------------------------------------------------------------
 * K2  classify + compact: sign bit-planes -> cube codes -> ambiguity redirect -> per-cube triangle counts ->
 *     device-wide exclusive scan of (active cubes, triangles) -> compacted, loop-ordered active-cube records with
 *     their triangle offsets.
 *
 *     Work item = one 32-cube word of a cube row; items are numbered in the reference's loop order (z slowest,
 *     then y, then x).  A tile is a run of whole cube rows (<= kClsItemCap items).
 *
 *     classify_kernel (one block per tile, no dependency between tiles):
 *       A  every thread walks one word column down a strip of rows, carrying the sign words of the vertex row it
 *          shares with the next cube row (4 loads and ~30 instructions per 32 cubes), and sets a bit in a
 *          shared-memory bitmap for every item that has an active cube.  With the candidate map of the block-field
 *          mode (block_class_kernel) it steps over four cube rows at a time wherever the interval test has already
 *          proven that no sign changes: this is the only work done per voxel, and it is then done per 128 voxels;
 *       B  the bitmap is turned into the list of active items in loop order (popc + block scan);
 *       C1 one lane per ACTIVE item: rebuild its corner words, per cube code -> triangle count.  A cube whose code
 *          has a redirect entry (marching_lookup.h:329-587) is counted with its own row for now and appended to the
 *          ambiguity list.  One 64-bit entry per active item goes to global scratch:
 *              [5:0] active cubes  [13:6] triangles  [26:14] tile-local item  [63:32] redirected cubes (bit per cube)
 *     ambiguity_kernel (one thread per listed cube): the face-centre test of marching.cpp:521-549 — one evaluation of
 *          the field — and, when it redirects, the bit in the item's entry and the triangle-count difference of row
 *          255-code, applied to the entry and to the tile total with atomics.  Dense lanes: a tile with one
 *          ambiguous cube no longer holds up a whole block, and the test is evaluated once, not twice.
 *     compact_kernel (one block per tile; tiles without an active item leave at once, except the last):
 *       C2 the tile's base: the sum of the earlier tiles' totals (final once ambiguity_kernel is done; a few thousand
 *          words from L2); the last tile's block also writes the grand totals to the counters.  Per chunk of 32 list
 *          entries a packed shuffle scan, then one lane per active item writes its cubes' records in loop order at
 *          tile base + chunk base + lane offset.
 * ------------------------------------------------------------------------------------------------------------- */
constexpr int kClsWarps = kClsThreads / 32;
constexpr int kClsItemCap = 8192; /* items per tile: bitmap 1 KB + active-item list 16 KB of shared memory */
constexpr int kClsChunkCap = kClsItemCap / 32;
constexpr size_t kClsSmemBytes = (size_t)kClsChunkCap * 4 + (size_t)kClsItemCap * 2; /* bitmap + list */

struct ClsGeom {
    uint32_t WC;         /* 32-cube words per cube row */
    uint32_t total_rows; /* (ke-kb) * M cube rows in the slab */
    uint32_t tile_rows;  /* cube rows per tile; tile_rows * WC <= kClsItemCap */
    uint32_t nstrips;    /* kClsThreads / WC row strips walked in parallel in phase A */
    uint32_t strip_rows; /* ceil(tile_rows / nstrips) */
    uint32_t inv_wc;     /* ceil(2^32 / WC), 0 when WC == 1 */
    uint32_t inv_m;      /* ceil(2^32 / M),  0 when M == 1 */
};
/* floor(n / d) for n * d < 2^32 (tile-local indices), inv = ceil(2^32 / d) */
__device__ __forceinline__ uint32_t div_small(uint32_t n, uint32_t inv) { return inv ? __umulhi(n, inv) : n; }

struct ClsTables { /* built once per context on the host (mcb_tables.h); read through the read-only path */
    uint64_t tri[256];
    int8_t face[256];
    uint8_t ntri[256];
    uint16_t emask[256]; /* bit e: edge e joins corners on different sides (marching.cpp:563-566), from the raw cube code */
};

/* Sign words of one vertex row as seen by the 32 cubes of an item: the vertex x-index of corner dx of cube i is
 * i+1+dx (apron), hence the funnel shifts by 1 and 2.  r[0], r[1] = corners dx=0,1 on plane z; r[2], r[3] on z+1.
 * All indices fit 32 bits (NZ*NV*WP < 2^32 for M <= 4094). */
__device__ __forceinline__ void vertex_row_words(const uint32_t* __restrict__ B, uint32_t idx, uint32_t plane, uint32_t r[4]) {
    const uint32_t* p0 = B + idx;
    const uint32_t* p1 = B + (idx + plane);
    const uint32_t a0 = __ldg(p0), a1 = __ldg(p0 + 1);
    const uint32_t b0 = __ldg(p1), b1 = __ldg(p1 + 1);
    r[0] = __funnelshift_r(a0, a1, 1); r[1] = __funnelshift_r(a0, a1, 2);
    r[2] = __funnelshift_r(b0, b1, 1); r[3] = __funnelshift_r(b0, b1, 2);
}
/* corner words c[v] (bit b = sign of corner v of cube 32w+b) from the two vertex rows of a cube row */
__device__ __forceinline__ void corner_words(const uint32_t lo[4], const uint32_t hi[4], uint32_t c[8]) {
    c[0] = lo[0]; c[1] = lo[1]; c[4] = lo[2]; c[5] = lo[3];
    c[3] = hi[0]; c[2] = hi[1]; c[7] = hi[2]; c[6] = hi[3];
}

__device__ __forceinline__ int code_of(const uint32_t c[8], int b) {
    int code = 0;
#pragma unroll
    for (int v = 0; v < 8; v++) code |= ((c[v] >> b) & 1u) << v;
    return code;
}

/* Face-centre test of marching.cpp:527-547; returns true when the redirect row 255-code must be used. */
__device__ __noinline__ bool ambiguity_redirects(const mcb_program& prog, const Grid& g, const float* __restrict__ cs,
                                                 int face, int i, int j, int k, float iso) {
    float mx = 0.f, my = 0.f, mz = 0.f;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int ofs = mcb_corner_ofs(mcb_face_corner(face, q));
        mx += cs[i + 1 + (ofs & 1)];
        my += cs[j + 1 + ((ofs >> 1) & 1)];
        mz += cs[k + 1 + ((ofs >> 2) & 1)];
    }
    mx /= 4.0f; my /= 4.0f; mz /= 4.0f;
    const float mid = mcb_interp_scalar(prog.code, prog.n, prog.k, g.sx * mx, g.sy * my, g.sz * mz, nullptr, nullptr, nullptr);
    return mid > iso;
}

__device__ __forceinline__ uint32_t column_mask(const Grid& g, uint32_t w) { /* cubes of word w inside the row */
    const int ncubes = g.M - (int)w * 32;
    return ncubes >= 32 ? 0xffffffffu : ((1u << ncubes) - 1u);
}
__device__ __forceinline__ uint32_t active_mask(const uint32_t c[8], uint32_t colmask) {
    const uint32_t any = c[0] | c[1] | c[2] | c[3] | c[4] | c[5] | c[6] | c[7];
    const uint32_t all = c[0] & c[1] & c[2] & c[3] & c[4] & c[5] & c[6] & c[7];
    return any & ~all & colmask;
}
/* constraints: all 8 corners of a cube must be valid (marching.cpp:475-477) */
__device__ __forceinline__ uint32_t valid_mask(const uint32_t* __restrict__ V, uint32_t idx, uint32_t WP, uint32_t plane) {
    uint32_t lo[4], hi[4];
    vertex_row_words(V, idx, plane, lo);
    vertex_row_words(V, idx + WP, plane, hi);
    return lo[0] & lo[1] & lo[2] & lo[3] & hi[0] & hi[1] & hi[2] & hi[3];
}

/* an active item revisited: position, corner words, active mask */
struct ItemView {
    uint32_t w, j, kz, m;
    uint32_t c[8];
};
/* Repeating-surface mode: a cube's corner signs are relative to ITS iso level, so they cannot be shared through the
 * vertex sign planes; repeat_words_kernel stores the eight corner words of every item instead (Cw[item][8]). */
__device__ __forceinline__ void repeat_item_words(const uint32_t* __restrict__ Cw, size_t item, uint32_t c[8]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(Cw + item * 8)), b = __ldg(reinterpret_cast<const uint4*>(Cw + item * 8 + 4));
    c[0] = a.x; c[1] = a.y; c[2] = a.z; c[3] = a.w; c[4] = b.x; c[5] = b.y; c[6] = b.z; c[7] = b.w;
}
__global__ void __launch_bounds__(256)
repeat_words_kernel(const Grid g, const float* __restrict__ F, uint32_t WC, uint32_t* __restrict__ Cw, unsigned long long items) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const int lane = threadIdx.x & 31;
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    for (unsigned long long item = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); item < items;
         item += (unsigned long long)gridDim.x * (blockDim.x >> 5)) {
        const uint32_t w = (uint32_t)(item % WC);
        const unsigned long long row = item / WC;
        const int j = (int)(row % (unsigned)g.M), kz = (int)(row / (unsigned)g.M), i = (int)w * 32 + lane;
        const bool in = i < g.M;
        float iso = 0.f;
        const float* f0 = F + (size_t)(kz + 1) * planep + (size_t)(j + 1) * rowp + (i + 1);
        if (in) iso = cube_iso(g, F, i, j, kz + g.kb);
        uint32_t mine = 0;
#pragma unroll
        for (int v = 0; v < 8; v++) {
            const int o = mcb_corner_ofs(v);
            const bool up = in && __ldg(f0 + (size_t)(o >> 2) * planep + (size_t)((o >> 1) & 1) * rowp + (o & 1)) > iso; /* marching.cpp:497-505 */
            const uint32_t word = __ballot_sync(0xffffffffu, up);
            if (lane == v) mine = word;
        }
        if (lane < 8) Cw[item * 8 + lane] = mine;
    }
}

template <bool REPEAT>
__device__ __forceinline__ void view_item(ItemView& it, uint32_t item_local, uint32_t j0, uint32_t kz0, const ClsGeom& q,
                                          const Grid& g, const uint32_t* __restrict__ S, const uint32_t* __restrict__ V,
                                          uint32_t plane, const uint32_t* __restrict__ Cw) {
    const uint32_t r = div_small(item_local, q.inv_wc);
    it.w = item_local - r * q.WC;
    const uint32_t jj = j0 + r, dk = div_small(jj, q.inv_m);
    it.j = jj - dk * (uint32_t)g.M;
    it.kz = kz0 + dk;
    const uint32_t idx = ((it.kz + 1u) * (uint32_t)g.NV + (it.j + 1u)) * (uint32_t)g.WP + it.w;
    if (REPEAT) repeat_item_words(Cw, ((size_t)it.kz * (uint32_t)g.M + it.j) * q.WC + it.w, it.c);
    else {
        uint32_t lo[4], hi[4];
        vertex_row_words(S, idx, plane, lo);
        vertex_row_words(S, idx + (uint32_t)g.WP, plane, hi);
        corner_words(lo, hi, it.c);
    }
    it.m = active_mask(it.c, column_mask(g, it.w));
    if (V != nullptr && it.m) it.m &= valid_mask(V, idx, (uint32_t)g.WP, plane);
}

constexpr uint32_t kTileGroupLog = 8, kTileGroup = 1u << kTileGroupLog; /* a group's sums stay below 2^32 */
struct ClsScratch {          /* global scratch handed from classify_kernel to ambiguity / compact */
    unsigned long long* ent; /* [tiles][tile_items]  one entry per active item of the tile, loop order (layout above) */
    uint32_t* nz;            /* [tiles]  number of entries */
    uint32_t* tile_a;        /* [tiles]  active cubes of the tile */
    uint32_t* tile_t;        /* [tiles]  triangles of the tile (ambiguity_kernel corrects it) */
    uint32_t* grp_a;         /* [ceil(tiles / kTileGroup)]  the same sums per group of tiles, zeroed before the pass, */
    uint32_t* grp_t;         /*   so that compact_kernel's base reads a group total per earlier group, not every tile */
    unsigned long long* amb; /* [cap_amb][2]  entry index | bit << 40 | face << 45 | code << 48 ;  i | j << 12 | k << 24 */
    uint32_t cap_amb;
    uint32_t tile_items;     /* tile_rows * WC */
    const unsigned long long* cand; /* [ckb][cjb][cmw] one bit per cube block that may hold an active cube, or nullptr: look everywhere */
    uint32_t cjb;            /* ceil(M / 4) */
    uint32_t cmw;            /* 64-bit words per row group: ceil(WC / 64) */
};
#define MCB_ENT_NA(e) ((uint32_t)(e) & 63u)
#define MCB_ENT_NT(e) (((uint32_t)(e) >> 6) & 255u)
#define MCB_ENT_ITEM(e) (((uint32_t)(e) >> 14) & 8191u)
#define MCB_ENT_RED(e) ((uint32_t)((e) >> 32))

template <bool HAS_V, bool REPEAT /* repeating-surface mode: corner words from Cw instead of the sign planes */>
__global__ void __launch_bounds__(kClsThreads, 4)
classify_kernel(const Grid g, const ClsTables* __restrict__ gtb, const uint32_t* __restrict__ S, const uint32_t* __restrict__ V,
                const ClsGeom q, const ClsScratch sc, Counters* __restrict__ ctr,
                const uint32_t* __restrict__ Cw /* repeating-surface mode: corner words, else nullptr */) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    MCB_DYNAMIC_SMEM(uint32_t, cls_smem);
    uint32_t* bitmap = cls_smem;                                          /* [kClsChunkCap] one bit per item */
    uint16_t* list = reinterpret_cast<uint16_t*>(cls_smem + kClsChunkCap); /* [kClsItemCap] active items, loop order */
    __shared__ uint32_t warp_x[kClsWarps], warp_y[kClsWarps];
    __shared__ uint32_t ncand_s;

    for (int i = threadIdx.x; i < kClsChunkCap; i += kClsThreads) bitmap[i] = 0u;
    __syncthreads();
    const uint32_t tile = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t WP = (uint32_t)g.WP, plane = (uint32_t)g.NV * WP, M = (uint32_t)g.M;
    const uint32_t row0 = tile * q.tile_rows;
    const uint32_t rows = min(q.tile_rows, q.total_rows - row0);
    const uint32_t kz0 = row0 / M, j0 = row0 - kz0 * M;

    /* ---- A: one bit per item -------------------------------------------------------------------------------
     * The tile's rows are taken four at a time: a CELL is one word column of the (up to) four cube rows with the same
     * j / 4 of one layer — the footprint of a cube block of the candidate map.  First the cells worth looking at are
     * listed (all of them without a map), then a thread per listed cell walks its rows, carrying the sign words of the
     * vertex row two cube rows share.  Dense lanes and independent loads: the time goes with the number of candidate
     * cells, not with the volume. */
    {
        const uint32_t cjb = sc.cjb;
        const uint32_t r_last = row0 + rows - 1u, kz1 = r_last / M, j1 = r_last - kz1 * M;
        const uint32_t G0 = kz0 * cjb + (j0 >> 2), G1 = kz1 * cjb + (j1 >> 2);
        const uint32_t ncell = (G1 - G0 + 1u) * q.WC;
        uint16_t* cells = list; /* free until phase B */
        uint32_t ncand = ncell;
        const bool mapped = !REPEAT && sc.cand != nullptr;
        if (mapped) { /* a thread per (row group, 64 word columns): one load says which of its cells are candidates */
            if (threadIdx.x == 0) ncand_s = 0u;
            __syncthreads();
            const uint32_t nG = G1 - G0 + 1u, nmask = nG * sc.cmw;
            for (uint32_t c0 = 0; c0 < nmask; c0 += kClsThreads) {
                const uint32_t mi = c0 + threadIdx.x;
                unsigned long long bits = 0ull;
                uint32_t gq = 0, part = 0;
                if (mi < nmask) {
                    gq = mi / sc.cmw; part = mi - gq * sc.cmw;
                    const uint32_t G = G0 + gq, kz = G / cjb, jb = G - kz * cjb;
                    bits = __ldg(sc.cand + ((size_t)(kz >> 2) * cjb + jb) * sc.cmw + part);
                }
                const uint32_t cnt = (uint32_t)__popcll(bits);
                uint32_t inc = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
                const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
                if (total == 0u) continue;
                uint32_t base = 0;
                if (lane == 31) base = atomicAdd(&ncand_s, total);
                base = __shfl_sync(0xffffffffu, base, 31) + inc - cnt;
                while (bits) {
                    const int w = __ffsll((long long)bits) - 1;
                    bits &= bits - 1ull;
                    cells[base++] = (uint16_t)(gq * q.WC + part * 64u + (uint32_t)w);
                }
            }
            __syncthreads();
            ncand = ncand_s;
        }
        for (uint32_t q2 = threadIdx.x; q2 < ncand; q2 += kClsThreads) {
            const uint32_t c = mapped ? (uint32_t)cells[q2] : q2;
            const uint32_t gq = div_small(c, q.inv_wc), w = c - gq * q.WC, G = G0 + gq, kz = G / cjb, jb = G - kz * cjb;
            uint32_t R_lo = kz * M + 4u * jb, R_hi = kz * M + min(4u * jb + 4u, M); /* slab-local cube rows of the cell */
            R_lo = max(R_lo, row0); R_hi = min(R_hi, row0 + rows);
            if (R_lo >= R_hi) continue;
            const uint32_t n = R_hi - R_lo, j = R_lo - kz * M;
            const uint32_t colmask = column_mask(g, w);
            uint32_t item = (R_lo - row0) * q.WC + w;
            uint32_t idx = ((kz + 1u) * (uint32_t)g.NV + (j + 1u)) * WP + w;
            if (REPEAT) { /* repeating-surface mode: nothing is shared between cube rows */
                for (uint32_t t = 0; t < n; t++) {
                    uint32_t cw8[8];
                    repeat_item_words(Cw, ((size_t)kz * M + (j + t)) * q.WC + w, cw8);
                    uint32_t m = active_mask(cw8, colmask);
                    if (HAS_V && m) m &= valid_mask(V, idx, WP, plane);
                    if (m) atomicOr(&bitmap[item >> 5], 1u << (item & 31u));
                    idx += WP;
                    item += q.WC;
                }
                continue;
            }
            uint32_t lo[4];
            vertex_row_words(S, idx, plane, lo);
            uint32_t any_lo = lo[0] | lo[1] | lo[2] | lo[3], all_lo = lo[0] & lo[1] & lo[2] & lo[3];
#pragma unroll 4
            for (uint32_t t = 0; t < n; t++) {
                uint32_t hi[4];
                vertex_row_words(S, idx + WP, plane, hi);
                const uint32_t any_hi = hi[0] | hi[1] | hi[2] | hi[3], all_hi = hi[0] & hi[1] & hi[2] & hi[3];
                uint32_t m = (any_lo | any_hi) & ~(all_lo & all_hi) & colmask;
                if (HAS_V && m) m &= valid_mask(V, idx, WP, plane);
                if (m) atomicOr(&bitmap[item >> 5], 1u << (item & 31u));
                any_lo = any_hi; all_lo = all_hi;
                idx += WP;
                item += q.WC;
            }
        }
    }
    __syncthreads();

    /* ---- B: bitmap -> list of active items in loop order ------------------------------------------------------ */
    uint32_t nz;
    {
        constexpr int kPer = (kClsChunkCap + kClsThreads - 1) / kClsThreads; /* bitmap words per thread */
        uint32_t wd[kPer], mine = 0;
#pragma unroll
        for (int i = 0; i < kPer; i++) {
            const int wi = threadIdx.x * kPer + i;
            wd[i] = wi < kClsChunkCap ? bitmap[wi] : 0u;
            mine += __popc(wd[i]);
        }
        uint32_t inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) warp_x[warp] = inc;
        __syncthreads();
        uint32_t base = inc - mine;
        nz = 0;
#pragma unroll
        for (int w2 = 0; w2 < kClsWarps; w2++) { if (w2 < warp) base += warp_x[w2]; nz += warp_x[w2]; }
#pragma unroll
        for (int i = 0; i < kPer; i++) {
            uint32_t b = wd[i];
            while (b) {
                const int bit = __ffs(b) - 1;
                b &= b - 1;
                list[base++] = (uint16_t)((threadIdx.x * kPer + i) * 32 + bit);
            }
        }
    }
    __syncthreads();
    if (nz == 0) { /* uniform per block: most tiles of a sparse surface end here */
        if (threadIdx.x == 0) { sc.nz[tile] = 0; sc.tile_a[tile] = 0; sc.tile_t[tile] = 0; }
        return;
    }

    /* ---- C1: per active item: cube codes, triangle counts, the ambiguity list ---------------------------------- */
    unsigned long long* gent = sc.ent + (size_t)tile * sc.tile_items;
    uint32_t sum_a = 0, sum_t = 0;
    for (uint32_t kb = (uint32_t)warp * 32u; kb < nz; kb += kClsThreads) {
        const uint32_t k = kb + (uint32_t)lane;
        if (k < nz) {
            const uint32_t item_local = list[k];
            ItemView it;
            view_item<REPEAT>(it, item_local, j0, kz0, q, g, S, V, plane, Cw);
            const uint32_t na = __popc(it.m);
            uint32_t nt = 0, mm = it.m;
            while (mm) {
                const int b = __ffs(mm) - 1;
                mm &= mm - 1;
                const int code = code_of(it.c, b);
                const int face = (int)(int8_t)__ldg((const signed char*)gtb->face + code);
                if (face >= 0) { /* marching.cpp:521-549: decided by ambiguity_kernel */
                    const uint32_t slot = atomicAdd(&ctr->amb_n, 1u);
                    if (slot < sc.cap_amb) {
                        sc.amb[2 * (size_t)slot] = ((unsigned long long)tile * sc.tile_items + k) | ((unsigned long long)b << 40) |
                                                   ((unsigned long long)face << 45) | ((unsigned long long)code << 48);
                        sc.amb[2 * (size_t)slot + 1] = (unsigned long long)(it.w * 32 + b) | ((unsigned long long)it.j << 12) |
                                                       ((unsigned long long)(it.kz + g.kb) << 24);
                    }
                }
                nt += __ldg(gtb->ntri + code);
            }
            gent[k] = (unsigned long long)(na | (nt << 6) | (item_local << 14)); /* na <= 32, nt <= 160, item < 8192 */
            sum_a += na; sum_t += nt;
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) { sum_a += __shfl_xor_sync(0xffffffffu, sum_a, d); sum_t += __shfl_xor_sync(0xffffffffu, sum_t, d); }
    if (lane == 0) { warp_x[warp] = sum_a; warp_y[warp] = sum_t; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t ta = 0, tt = 0;
#pragma unroll
        for (int w2 = 0; w2 < kClsWarps; w2++) { ta += warp_x[w2]; tt += warp_y[w2]; }
        sc.nz[tile] = nz;
        sc.tile_a[tile] = ta;                  /* < 2^19 cubes */
        sc.tile_t[tile] = tt;                  /* ambiguity_kernel corrects it afterwards */
        atomicAdd(sc.grp_a + (tile >> kTileGroupLog), ta);
        atomicAdd(sc.grp_t + (tile >> kTileGroupLog), tt);
    }
}

/* One thread per ambiguous cube: the face-centre test, evaluated once. */
template <bool REPEAT>
__global__ void __launch_bounds__(128)
ambiguity_kernel(const __grid_constant__ mcb_program point_prog, const Grid g, const float* __restrict__ cs,
                 const ClsTables* __restrict__ gtb, const ClsScratch sc, Counters* __restrict__ ctr, const float* __restrict__ F) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const uint32_t n = min(ctr->amb_n, sc.cap_amb);
    uint32_t redirected = 0;
    for (uint32_t a = blockIdx.x * blockDim.x + threadIdx.x; a < n; a += gridDim.x * blockDim.x) {
        const unsigned long long e0 = sc.amb[2 * (size_t)a], e1 = sc.amb[2 * (size_t)a + 1];
        const unsigned long long entry = e0 & ((1ull << 40) - 1ull);
        const int b = (int)((e0 >> 40) & 31u), face = (int)((e0 >> 45) & 7u), code = (int)((e0 >> 48) & 255u);
        const int ci = (int)(e1 & 0xFFFu), cj = (int)((e1 >> 12) & 0xFFFu), ck = (int)((e1 >> 24) & 0xFFFu);
        if (!ambiguity_redirects(point_prog, g, cs, face, ci, cj, ck, REPEAT ? cube_level(g, F, ci, cj, ck) : g.iso)) continue;
        redirected++;
        const int delta = (int)__ldg(gtb->ntri + (255 - code)) - (int)__ldg(gtb->ntri + code);
        /* one atomic sets the cube's redirect bit and moves the item's triangle count: the count field cannot underflow,
         * every partial sum of corrections is at least minus the triangles counted for those cubes */
        atomicAdd(sc.ent + entry, (1ull << (32 + b)) + (unsigned long long)((long long)delta * 64));
        if (delta) {
            const uint32_t t = (uint32_t)(entry / sc.tile_items);
            atomicAdd(sc.tile_t + t, (uint32_t)delta);
            atomicAdd(sc.grp_t + (t >> kTileGroupLog), (uint32_t)delta);
        }
    }
    if (redirected) atomicAdd(&ctr->redirected, (unsigned long long)redirected);
}

template <bool REPEAT>
__global__ void __launch_bounds__(kClsThreads, 5) /* 48 registers, as before the tile bases moved in: no spill */
compact_kernel(const Grid g, const ClsTables* __restrict__ gtb, const uint32_t* __restrict__ S, const uint32_t* __restrict__ V,
               const ClsGeom q, const ClsScratch sc, Counters* __restrict__ ctr, unsigned long long* __restrict__ rec,
               uint32_t* __restrict__ trioff, unsigned long long cap_active, unsigned long long* __restrict__ item_info /* nullptr unless the weld needs it */,
               const uint32_t* __restrict__ Cw /* repeating-surface mode, else nullptr */,
               const FieldBlocks fb /* block-field mode: flags != nullptr, the apron blocks are marked here */) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    __shared__ uint32_t chunk_a[kClsChunkCap], chunk_t[kClsChunkCap]; /* per 32 list entries */
    __shared__ uint32_t warp_x[kClsWarps], warp_y[kClsWarps];
    __shared__ unsigned long long warp_ba[kClsWarps], warp_bt[kClsWarps], base_s[2];

    const uint32_t tile = blockIdx.x;
    const uint32_t nz = sc.nz[tile];
    const bool last = tile == gridDim.x - 1u; /* the grid is one block per tile */
    if (nz == 0 && !last) return; /* uniform per block */
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    /* the tile's exclusive bases (read back from base_s in C2): every tile and group total is final once ambiguity_kernel
     * is done; the earlier groups' totals, then the earlier tiles of this tile's group */
    {
        unsigned long long sa = 0, st = 0;
        const uint32_t g0 = tile >> kTileGroupLog;
        for (uint32_t i = threadIdx.x; i < g0; i += kClsThreads) { sa += sc.grp_a[i]; st += sc.grp_t[i]; }
        for (uint32_t i = (g0 << kTileGroupLog) + threadIdx.x; i < tile; i += kClsThreads) { sa += sc.tile_a[i]; st += sc.tile_t[i]; }
#pragma unroll
        for (int d = 16; d; d >>= 1) { sa += __shfl_xor_sync(0xffffffffu, sa, d); st += __shfl_xor_sync(0xffffffffu, st, d); }
        if (lane == 0) { warp_ba[warp] = sa; warp_bt[warp] = st; }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long ba = 0, bt = 0;
#pragma unroll
            for (int w2 = 0; w2 < kClsWarps; w2++) { ba += warp_ba[w2]; bt += warp_bt[w2]; }
            base_s[0] = ba; base_s[1] = bt;
            if (last) {
                const unsigned long long total_t = bt + sc.tile_t[tile];
                ctr->active = ba + sc.tile_a[tile];
                ctr->triangles = total_t;
                ctr->ambiguous = ctr->amb_n;
                if (total_t >= (1ull << 31)) ctr->error = 2u; /* >= 2^31 triangles in one slab: beyond any output buffer */
            }
        }
    }
    if (nz == 0) return; /* the last tile's block, done with the totals */
    const unsigned long long* __restrict__ gent = sc.ent + (size_t)tile * sc.tile_items;
    const uint32_t row0 = tile * q.tile_rows;

    for (uint32_t kb = (uint32_t)warp * 32u; kb < nz; kb += kClsThreads) {
        const uint32_t k = kb + (uint32_t)lane;
        const unsigned long long e = k < nz ? gent[k] : 0ull;
        uint32_t na = MCB_ENT_NA(e), nt = MCB_ENT_NT(e);
#pragma unroll
        for (int d = 16; d; d >>= 1) { na += __shfl_xor_sync(0xffffffffu, na, d); nt += __shfl_xor_sync(0xffffffffu, nt, d); }
        if (lane == 0) { chunk_a[kb >> 5] = na; chunk_t[kb >> 5] = nt; }
    }
    __syncthreads();
    { /* exclusive scan of the chunk totals, in place */
        constexpr int kPer = (kClsChunkCap + kClsThreads - 1) / kClsThreads;
        const uint32_t nchunks = (nz + 31u) >> 5;
        uint32_t a[kPer], t[kPer], sa = 0, st = 0;
#pragma unroll
        for (int i = 0; i < kPer; i++) {
            const uint32_t c = threadIdx.x * kPer + i;
            a[i] = c < nchunks ? chunk_a[c] : 0u;
            t[i] = c < nchunks ? chunk_t[c] : 0u;
            sa += a[i]; st += t[i];
        }
        uint32_t ia = sa, it = st;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t ua = __shfl_up_sync(0xffffffffu, ia, d), ut = __shfl_up_sync(0xffffffffu, it, d);
            if (lane >= d) { ia += ua; it += ut; }
        }
        if (lane == 31) { warp_x[warp] = ia; warp_y[warp] = it; }
        __syncthreads();
        uint32_t ba = ia - sa, bt = it - st;
#pragma unroll
        for (int w2 = 0; w2 < kClsWarps; w2++)
            if (w2 < warp) { ba += warp_x[w2]; bt += warp_y[w2]; }
#pragma unroll
        for (int i = 0; i < kPer; i++) {
            const uint32_t c = threadIdx.x * kPer + i;
            if (c < nchunks) { chunk_a[c] = ba; chunk_t[c] = bt; }
            ba += a[i]; bt += t[i];
        }
    }
    __syncthreads();

    /* ---- C2: write the compacted records in loop order -------------------------------------------------------- */
    const uint32_t WP = (uint32_t)g.WP, plane = (uint32_t)g.NV * WP, M = (uint32_t)g.M;
    const uint32_t kz0 = row0 / M, j0 = row0 - kz0 * M;
    const unsigned long long tile_a = base_s[0], tile_t = base_s[1];
    for (uint32_t kb = (uint32_t)warp * 32u; kb < nz; kb += kClsThreads) {
        const uint32_t k = kb + (uint32_t)lane;
        const unsigned long long e = k < nz ? gent[k] : 0ull;
        const uint32_t mine = MCB_ENT_NA(e) | (MCB_ENT_NT(e) << 16);
        uint32_t inc = mine; /* <= 32 | 160 << 16 per lane: a chunk's sum stays below 2^16 per field */
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (k >= nz) continue;
        unsigned long long oa = tile_a + chunk_a[kb >> 5] + ((inc - mine) & 0xffffu);
        unsigned long long ot = tile_t + chunk_t[kb >> 5] + ((inc - mine) >> 16);
        ItemView it;
        const uint32_t item_local = MCB_ENT_ITEM(e), red = MCB_ENT_RED(e);
        view_item<REPEAT>(it, item_local, j0, kz0, q, g, S, V, plane, Cw);
        uint32_t m = it.m;
        if (item_info != nullptr) /* cube -> record look-up of the weld: first record of the word | its active mask */
            item_info[(size_t)tile * sc.tile_items + item_local] = (oa & 0xFFFFFFFFull) | ((unsigned long long)m << 32);
        if (fb.flags != nullptr) {
            /* the mesh stages read the field at the corners of the active cubes and their +-1 neighbours: stored vertices
             * [i, i+3] x [j, j+3] x [kz, kz+3].  Blocks of that range the evaluation skipped (flag 0) are marked for the
             * apron refill.  Per item: the cubes of a word share j and kz, and span at most two blocks in x. */
            const int bx0 = (int)it.w, bx1 = (m >> 29) ? min((int)it.w + 1, fb.nbx - 1) : (int)it.w; /* a cube with i % 32 >= 29 reaches x + 3 in the next block */
            const int by0 = (int)it.j >> 2, by1 = ((int)it.j + 3) >> 2, bz0 = (int)it.kz >> 2, bz1 = ((int)it.kz + 3) >> 2;
            for (int bz = bz0; bz <= bz1; bz++)
                for (int by = by0; by <= by1; by++)
                    for (int bx = bx0; bx <= bx1; bx++) {
                        uint8_t* f = fb.flags + ((size_t)bz * fb.nby + by) * fb.nbx + bx;
                        if (*f == 0) *f = 1; /* 2 = already evaluated; racing writers all store 1 */
                    }
        }
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            const int code = code_of(it.c, b);
            const int tidx = ((red >> b) & 1u) ? 255 - code : code; /* marching.cpp:545-547 */
            if (oa < cap_active) {
                rec[oa] = (unsigned long long)(it.w * 32 + b) | ((unsigned long long)it.j << 12) |
                          ((unsigned long long)(it.kz + g.kb) << 24) | ((unsigned long long)code << 36) |
                          ((unsigned long long)tidx << 44);
                trioff[oa] = (uint32_t)ot;
            }
            oa++;
            ot += __ldg(gtb->ntri + tidx);
        }
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K3  emit: a block of kEmitThreads threads takes kEmitCubes consecutive active cubes.
 *       1  one thread per cube reads its record, looks up the crossing-edge set of its raw cube code
 *          (marching.cpp:563-566) in a table and appends one work entry per crossing edge to a shared-memory list
 *          (block scan);
 *       2  one thread per crossing EDGE (dense lanes, no divergence over which edges cross): the two corner values,
 *          Marching::interp for the position, central-difference gradients at both corners blended along the edge
 *          for the normal -> a float4 in shared memory (its coordinate + the normal), in compact slots: first slot
 *          of the cube + rank of the edge among the cube's crossing edges;
 *       3  the block writes the chunk's contiguous output range, one float4 position (+ one float4 normal) per
 *          thread per step: fully coalesced 16-byte stores in the reference's emission order, with chunk-local
 *          32-bit arithmetic.
 *     An edge is parallel to an axis, so Marching::interp (marching.cpp:437-446) changes ONE coordinate; for the other
 *     two, t * 0 is 0 or NaN and both the sum and the fallback return the end point's own grid coordinate exactly: one
 *     interp per edge, the positions bit for bit the reference's.
 *     The gradient normals are the product's own definition, checked to 1e-5 (north_star), not bit for bit: central
 *     differences multiply by a per-coordinate table of 1 / (c[v+1] - c[v-1]) (built once per grid on the host) instead
 *     of six IEEE divisions per edge, and the normalisation is rsqrtf.
 *     A chunk whose crossing edges exceed the kEmitSlots slots (never on a surface; a degenerate field can: 64 cubes
 *     of 12 crossing edges need 768) is emitted in several runs of whole cubes.
 *     The tiling (kEmitCubes, kEmitSlots, kEmitBlocksPerSM) was measured fastest on every workload against the
 *     alternatives in profiles/r02_ab_variants*.jsonl and profiles/r02_ab_emit_grid.jsonl (DESIGN.md §5).
 * ------------------------------------------------------------------------------------------------------------- */
/* The gradient normal of a crossing point is defined on the GRID EDGE, not on the cube that looks at it: blended from the
 * lower end point to the upper one with t = (iso - f_lo) / (f_hi - f_lo) (0.5 when that is not finite).  A cube whose edge
 * runs the other way (corner a is the upper end point) swaps the roles; fwd = corner a is the lower end point. */
__device__ __forceinline__ void blend_edge_normal(bool fwd, float iso, float f1, float f2, float tq, float gxa, float gya, float gza, float gxb,
                                                  float gyb, float gzb, float& nx, float& ny, float& nz) {
    float tt = fwd ? tq : (iso - f2) / (f1 - f2);
    if (isinf(tt) || isnan(tt)) tt = 0.5f;
    const float lx = fwd ? gxa : gxb, ly = fwd ? gya : gyb, lz = fwd ? gza : gzb;
    const float hx = fwd ? gxb : gxa, hy = fwd ? gyb : gya, hz = fwd ? gzb : gza;
    nx = lx + tt * (hx - lx);
    ny = ly + tt * (hy - ly);
    nz = lz + tt * (hz - lz);
}

template <bool NORMALS, bool IDX32 /* the slab's field has fewer than 2^32 values: 32-bit offsets, one IMAD.WIDE per load address */>
__global__ void __launch_bounds__(kEmitThreads, kEmitBlocksPerSM)
emit2_kernel(const Grid g, const float* __restrict__ cs, const float* __restrict__ rinv, const float* __restrict__ F,
             const ClsTables* __restrict__ gtb, const unsigned long long* __restrict__ rec, const uint32_t* __restrict__ trioff,
             Counters* ctr, unsigned long long cap_active, unsigned long long cap_tris,
             float4* __restrict__ pos, float4* __restrict__ nrm) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    static_assert(kEmitSlots >= 12 && kEmitCubes <= 256 && kEmitCubes <= kEmitThreads, "a cube's edges fit one run; a thread per cube in phase 1");
    __shared__ float4 eslot[NORMALS ? kEmitSlots : 1];    /* crossing edge: coordinate along its axis, normal */
    __shared__ float epos_only[NORMALS ? 1 : kEmitSlots];
    __shared__ float ccoord[kEmitCubes * 6];              /* x0 x1 y0 y1 z0 z1 of the cube */
    __shared__ float crinv[NORMALS ? kEmitCubes * 6 : 1]; /* 1 / (c[v+1] - c[v-1]) at the same six coordinates */
    typedef typename std::conditional<IDX32, uint32_t, unsigned long long>::type off_t; /* offsets into F */
    __shared__ off_t cbase_s[kEmitCubes];                 /* offset of the cube's corner 0 in F */
    __shared__ uint32_t off_s[kEmitCubes + 1];            /* first triangle of the cube */
    __shared__ uint64_t triw_s[kEmitCubes];
    __shared__ uint16_t emask_s[kEmitCubes];
    __shared__ uint16_t ebase_s[kEmitCubes + 1];          /* exclusive prefix of the crossing-edge counts */
    __shared__ uint16_t work_s[kEmitCubes * 12];          /* local cube << 4 | edge, one per crossing edge, (cube, edge) order */
    __shared__ uint8_t tri2cube[kEmitCubes * 5];          /* chunk-local triangle -> local cube (a cube has at most 5) */
    __shared__ uint32_t warp_s[kEmitThreads / 32];

    unsigned long long A = ctr->active;
    const unsigned long long T = ctr->triangles;
    const bool whole = A <= cap_active;
    if (!whole) A = cap_active; /* the host re-runs with larger buffers when counts exceed capacity */
    const unsigned long long nchunks = (A + kEmitCubes - 1) / kEmitCubes;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const off_t rowp = (off_t)g.P, planep = (off_t)g.NV * (off_t)g.P;

    /* Chunks are handed out by an atomic counter: a chunk's work varies with its crossing edges, and the grid is one
     * resident wave (a static stride leaves the blocks of a partial last wave running alone).  The last block to finish
     * resets the counters, so a repeated launch within the call starts from zero again. */
    __shared__ unsigned int chunk_s;
    for (;;) {
        __syncthreads();
        if (t == 0) chunk_s = atomicAdd(&ctr->emit_next, 1u);
        __syncthreads();
        const unsigned long long chunk = chunk_s;
        if (chunk >= nchunks) break;
        const unsigned long long c0 = chunk * kEmitCubes;
        const int n = (int)((A - c0) < (unsigned long long)kEmitCubes ? (A - c0) : kEmitCubes);

        /* ---- 1: records -> per-cube state and the edge work list ---- */
        uint32_t emask = 0;
        if (t < n) {
            const unsigned long long r = rec[c0 + t];
            const int code = (int)((r >> 36) & 0xFF), tidx = (int)((r >> 44) & 0xFF);
            const int i = (int)(r & 0xFFF), j = (int)((r >> 12) & 0xFFF), k = (int)((r >> 24) & 0xFFF);
            off_s[t] = trioff[c0 + t];
            triw_s[t] = mcb_tri_word(tidx);
            emask = __ldg(gtb->emask + code);
            emask_s[t] = (uint16_t)emask;
            ccoord[6 * t + 0] = __ldg(cs + i + 1); ccoord[6 * t + 1] = __ldg(cs + i + 2);
            ccoord[6 * t + 2] = __ldg(cs + j + 1); ccoord[6 * t + 3] = __ldg(cs + j + 2);
            ccoord[6 * t + 4] = __ldg(cs + k + 1); ccoord[6 * t + 5] = __ldg(cs + k + 2);
            if (NORMALS) {
                crinv[6 * t + 0] = __ldg(rinv + i + 1); crinv[6 * t + 1] = __ldg(rinv + i + 2);
                crinv[6 * t + 2] = __ldg(rinv + j + 1); crinv[6 * t + 3] = __ldg(rinv + j + 2);
                crinv[6 * t + 4] = __ldg(rinv + k + 1); crinv[6 * t + 5] = __ldg(rinv + k + 2);
            }
            cbase_s[t] = (off_t)(k - g.kb + 1) * planep + (off_t)(j + 1) * rowp + (off_t)(i + 1);
        }
        const uint32_t nv = __popc(emask);
        uint32_t inc = nv;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) warp_s[warp] = inc;
        __syncthreads();
        uint32_t wbase = inc - nv;
#pragma unroll
        for (int w2 = 0; w2 < kEmitThreads / 32; w2++) if (w2 < warp) wbase += warp_s[w2];
        if (t < n) ebase_s[t] = (uint16_t)wbase;
        if (t == n - 1) ebase_s[n] = (uint16_t)(wbase + nv);
        while (emask) {
            const int e = __ffs(emask) - 1;
            emask &= emask - 1;
            work_s[wbase++] = (uint16_t)((t << 4) | e);
        }
        if (t == 0) /* end of the chunk's output range; a capacity-truncated run is repeated by the host anyway */
            off_s[n] = (c0 + n < A) ? trioff[c0 + n] : (whole ? (uint32_t)T : off_s[n - 1]);
        __syncthreads();
        if (t < n) { /* off_s is complete here */
            const uint32_t first = off_s[t] - off_s[0], cnt = off_s[t + 1] - off_s[t];
            for (uint32_t q2 = 0; q2 < cnt && q2 < 5u; q2++) tri2cube[first + q2] = (uint8_t)t;
        }

        /* runs of whole cubes whose crossing edges fit the slots (one run, except on degenerate fields) */
        for (int cb = 0; cb < n;) {
            int ce = n;
            if ((int)ebase_s[n] - (int)ebase_s[cb] > kEmitSlots) { /* uniform: everyone reads the same prefix array */
                ce = cb + 1;
                while (ce < n && (int)ebase_s[ce + 1] - (int)ebase_s[cb] <= kEmitSlots) ce++;
            }
            const uint32_t q0 = ebase_s[cb], q1 = ebase_s[ce];

            /* ---- 2: one thread per crossing edge ---- */
            for (uint32_t q = q0 + t; q < q1; q += kEmitThreads) {
                const uint32_t wk = work_s[q];
                const int lc = (int)(wk >> 4), e = (int)(wk & 15u);
                const int a = mcb_edge_a(e), b = mcb_edge_b(e);
                const int oa = mcb_corner_ofs(a), ob = mcb_corner_ofs(b);
                const int axis = e >= 8 ? 2 : (e & 1);
                const off_t c0f = cbase_s[lc]; /* corner 0 of the cube; the end points are at most one step away on each axis */
                const off_t ia = c0f + (off_t)(oa & 1) + (((oa >> 1) & 1) ? rowp : (off_t)0) + ((oa >> 2) ? planep : (off_t)0);
                const off_t ib = c0f + (off_t)(ob & 1) + (((ob >> 1) & 1) ? rowp : (off_t)0) + ((ob >> 2) ? planep : (off_t)0);
                const float* cc = ccoord + 6 * lc + 2 * axis;
                const float ca = cc[(oa >> axis) & 1], cb2 = cc[(ob >> axis) & 1];
                const float f1 = __ldg(F + ia), f2 = __ldg(F + ib);
                const float tq = (g.iso - f1) / (f2 - f1); /* Marching::interp uses the surface constant itself, also in repeating-surface mode */
                const float p = mcb_interp_ref(ca, cb2, tq);
                if (NORMALS) { /* central differences times the reciprocals kept in shared memory, blended along the grid edge */
                    const float* ri = crinv + 6 * lc;
                    const float gxa = (__ldg(F + ia + 1) - __ldg(F + ia - 1)) * ri[oa & 1];
                    const float gya = (__ldg(F + (ia + rowp)) - __ldg(F + (ia - rowp))) * ri[2 + ((oa >> 1) & 1)];
                    const float gza = (__ldg(F + (ia + planep)) - __ldg(F + (ia - planep))) * ri[4 + (oa >> 2)];
                    const float gxb = (__ldg(F + ib + 1) - __ldg(F + ib - 1)) * ri[ob & 1];
                    const float gyb = (__ldg(F + (ib + rowp)) - __ldg(F + (ib - rowp))) * ri[2 + ((ob >> 1) & 1)];
                    const float gzb = (__ldg(F + (ib + planep)) - __ldg(F + (ib - planep))) * ri[4 + (ob >> 2)];
                    float nx, ny, nz;
                    blend_edge_normal(oa < ob, g.iso, f1, f2, tq, gxa, gya, gza, gxb, gyb, gzb, nx, ny, nz);
                    const float inv = rsqrtf(nx * nx + ny * ny + nz * nz);
                    eslot[q - q0] = make_float4(p, nx * inv, ny * inv, nz * inv);
                } else epos_only[q - q0] = p;
            }
            __syncthreads();

            /* ---- 3: coalesced float4 emission of the cubes [cb, ce) ---- */
            const uint32_t tri0 = off_s[0];
            const uint32_t lv_begin = 3u * (off_s[cb] - tri0), lv_end = 3u * (off_s[ce] - tri0);
            for (uint32_t lv = lv_begin + t; lv < lv_end; lv += kEmitThreads) {
                const uint32_t ltri = lv / 3u;
                const int corner = (int)(lv - 3u * ltri);
                const int lo = (int)tri2cube[ltri];
                const int lt = (int)(ltri - (off_s[lo] - tri0));
                const int e = (int)((triw_s[lo] >> (4 * (3 * lt + corner))) & 0xF);
                const uint32_t slot = (uint32_t)ebase_s[lo] - q0 + (uint32_t)__popc((uint32_t)emask_s[lo] & ((1u << e) - 1u));
                const int oa = mcb_corner_ofs(mcb_edge_a(e));
                const int axis = e >= 8 ? 2 : (e & 1);
                const float* cc = ccoord + 6 * lo;
                float x = cc[oa & 1], y = cc[2 + ((oa >> 1) & 1)], z = cc[4 + ((oa >> 2) & 1)];
                float4 en = make_float4(0.f, 0.f, 0.f, 0.f);
                float p;
                if (NORMALS) { en = eslot[slot]; p = en.x; } else p = epos_only[slot];
                if (axis == 0) x = p; else if (axis == 1) y = p; else z = p;
                const unsigned long long ov = 3ull * tri0 + lv;
                if ((unsigned long long)tri0 + ltri < cap_tris) {
                    __stcs(pos + ov, make_float4(x, y, z, 1.0f));
                    if (NORMALS) __stcs(nrm + ov, make_float4(en.y, en.z, en.w, 0.0f));
                }
            }
            cb = ce;
            if (cb < n) __syncthreads(); /* the slots are reused by the next run */
        }
    }
    if (t == 0) {
        __threadfence();
        if (atomicAdd(&ctr->emit_done, 1u) == gridDim.x - 1u) { ctr->emit_next = 0u; ctr->emit_done = 0u; }
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K4  weld: the reference's indexed mesh — Poly_Data::vertex_list / tri_list as add_step_to_poly_data / add_point
 *     build them (marching.cpp:599-654) — produced on the GPU without a std::set.
 *
 *     What the reference's tolerance set amounts to (marching.h:38-54: per-axis |d| < 1e-6 counts as equal; first
 *     inserted coordinates win; vertices are numbered by first insertion):
 *       - the up to four cubes sharing a grid edge compute the same crossing point to within an ulp, so they share
 *         one vertex, numbered and positioned by the FIRST of those cubes in loop order — the edge's owner;
 *       - two different grid edges can only yield points within 1e-6 of each other around a grid vertex they share,
 *         i.e. when both crossing points lie within the tolerance of that vertex (the surface passes through a grid
 *         corner: `x+y` on a dyadic grid does it everywhere).  All such points around one grid vertex form one
 *         cluster whose representative is the member inserted first.
 *         corner: `x+y` on a dyadic grid does it everywhere).  There the comparator is not even transitive, so the
 *         outcome of an insert depends on the insertion history: weld_replay re-enacts the (at most 24) insertions
 *         around that grid vertex with libstdc++'s unique-insert rule.
 *     So (cube, edge) -> welded vertex is a pure, local function of the grid: the edge's owner, or the replay's
 *     answer when the owner's point sits on a grid vertex.
 *     weld_count marks, per active cube, the edges for which the cube inserts a NEW vertex; an exclusive scan of
 *     those counts in loop order is the reference's vertex numbering; weld_emit writes vertex_list (the inserting
 *     cube's own interpolation), tri_list and, optionally, gradient normals per welded vertex.
 * ------------------------------------------------------------------------------------------------------------- */
/* REPEAT = repeating-surface mode: only then a cube's level has to be looked at (cube_level); the plain instantiation
 * carries none of it. */
template <bool REPEAT>
struct WeldViewT {
    static constexpr bool kRepeat = REPEAT;
    Grid g;
    const float* __restrict__ cs;
    const float* __restrict__ F;
    const uint32_t* __restrict__ V; /* constraint validity planes or nullptr */
    /* seed mode: only the kept cubes insert vertices.  Per 32-cube word `first record | kept mask << 32` (zero for
     * words without a kept cube), or nullptr when every active cube is present. */
    const unsigned long long* __restrict__ present;
    uint32_t WC;
};
using WeldView = WeldViewT<false>;
template <class WV>
__device__ __forceinline__ float weld_level(const WV& W, int i, int j, int k) { return WV::kRepeat ? cube_level(W.g, W.F, i, j, k) : W.g.iso; }

struct CubeEdge { /* an edge of a cube: who inserts a vertex, and as which of its edges */
    int i, j, k, e;
};
struct GridEdge { /* axis 0..2 and the lower end point in cube-vertex coordinates (0..M per axis) */
    int axis, vx, vy, vz;
};

__device__ __forceinline__ GridEdge grid_edge_of(int i, int j, int k, int e) {
    const int oa = mcb_corner_ofs(mcb_edge_a(e)), ob = mcb_corner_ofs(mcb_edge_b(e));
    const int lo = oa & ob, d = oa ^ ob; /* the end points differ in exactly one axis */
    GridEdge E;
    E.axis = d == 1 ? 0 : d == 2 ? 1 : 2;
    E.vx = i + (lo & 1); E.vy = j + ((lo >> 1) & 1); E.vz = k + ((lo >> 2) & 1);
    return E;
}
/* `level`: repeating-surface mode only — the iso level of the cube that asks.  A neighbour polygonised with another level
 * puts no point on the shared grid edge at this level, so for this edge it does not exist. */
template <class WV>
__device__ __forceinline__ bool weld_cube_ok(const WV& W, int i, int j, int k, float level = 0.f) {
    const Grid& g = W.g;
    if (i < 0 || j < 0 || i >= g.M || j >= g.M || k < g.kb || k >= g.ke) return false;
    if (WV::kRepeat && !(cube_level(g, W.F, i, j, k) == level)) return false;
    if (W.present != nullptr &&
        !(((uint32_t)(W.present[((size_t)(k - g.kb) * g.M + j) * W.WC + (i >> 5)] >> 32) >> (i & 31)) & 1u)) return false;
    if (W.V == nullptr) return true;
    bool ok = true; /* all 8 corners must satisfy the constraints (marching.cpp:475-477) */
#pragma unroll
    for (int v = 0; v < 8; v++) {
        const int x = i + 1 + (v & 1), y = j + 1 + ((v >> 1) & 1), z = k - g.kb + 1 + (v >> 2);
        ok = ok && ((W.V[((size_t)z * g.NV + y) * g.WP + (x >> 5)] >> (x & 31)) & 1u);
    }
    return ok;
}
/* first cube in loop order (z slowest, then y, then x) that contains the grid edge and is visited by the loop */
template <class WV>
__device__ __forceinline__ bool weld_owner(const WV& W, const GridEdge& E, CubeEdge& o, float level) {
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int hi = 1 - (q >> 1), lo = 1 - (q & 1); /* offsets in the slower / faster of the two other axes */
        if (E.axis == 0) { o.i = E.vx; o.j = E.vy - lo; o.k = E.vz - hi; o.e = 2 * lo + 4 * hi; }
        else if (E.axis == 1) { o.i = E.vx - lo; o.j = E.vy; o.k = E.vz - hi; o.e = (lo ? 1 : 3) + 4 * hi; }
        else { o.i = E.vx - lo; o.j = E.vy - hi; o.k = E.vz; o.e = 8 + (hi ? (lo ? 2 : 3) : (lo ? 1 : 0)); }
        if (weld_cube_ok(W, o.i, o.j, o.k, level)) return true;
    }
    return false;
}
/* crossing point of edge e of cube (i,j,k) along the edge's axis, interpolated in that cube's edge direction
 * (marching.cpp:557-583); crossing = the end points lie on different sides of iso */
template <class WV>
__device__ __forceinline__ float weld_edge_point(const WV& W, const CubeEdge& c, int axis, bool& crossing) {
    const Grid& g = W.g;
    const int oa = mcb_corner_ofs(mcb_edge_a(c.e)), ob = mcb_corner_ofs(mcb_edge_b(c.e));
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    const float* f0 = W.F + (size_t)(c.k - g.kb + 1) * planep + (size_t)(c.j + 1) * rowp + (c.i + 1);
    const float f1 = __ldg(f0 + (oa >> 2) * planep + ((oa >> 1) & 1) * rowp + (oa & 1));
    const float f2 = __ldg(f0 + (ob >> 2) * planep + ((ob >> 1) & 1) * rowp + (ob & 1));
    const float level = weld_level(W, c.i, c.j, c.k);
    crossing = (f1 > level) != (f2 > level);
    const int base = (axis == 0 ? c.i : axis == 1 ? c.j : c.k) + 1;
    const float ca = W.cs[base + ((oa >> axis) & 1)], cb = W.cs[base + ((ob >> axis) & 1)];
    return mcb_interp_ref(ca, cb, (g.iso - f1) / (f2 - f1)); /* Marching::interp (marching.cpp:437-446) always uses the surface constant */
}
__device__ __forceinline__ bool weld_close(float a, float b) { return (double)fabsf(a - b) < 0.000001; } /* marching.h:41 */
__device__ __forceinline__ unsigned long long weld_key(const Grid& g, const CubeEdge& c) {
    return ((((unsigned long long)c.k * g.M + c.j) * g.M + c.i) << 4) | (unsigned)c.e;
}

/* the reference's comparator, marching.h:38-54 */
__device__ __forceinline__ bool weld_less(const float a[3], const float b[3]) {
    if (!weld_close(a[0], b[0])) return a[0] < b[0];
    if (!weld_close(a[1], b[1])) return a[1] < b[1];
    if (!weld_close(a[2], b[2])) return a[2] < b[2];
    return false;
}
__device__ __forceinline__ CubeEdge weld_unkey(const Grid& g, unsigned long long key) {
    CubeEdge c;
    c.e = (int)(key & 15u);
    unsigned long long q = key >> 4;
    c.i = (int)(q % (unsigned)g.M); q /= (unsigned)g.M;
    c.j = (int)(q % (unsigned)g.M);
    c.k = (int)(q / (unsigned)g.M);
    return c;
}

/* Around a grid vertex G the tolerance comparator is not an equivalence relation (two collinear crossing points on
 * opposite sides of G can each be within 1e-6 of G yet 1e-6 apart, while a point on another axis is "equal" to
 * both), so what std::set::insert returns depends on what was inserted before.  This replays exactly that: every
 * insertion of a point near G — each cube sharing one of the six grid edges at G inserts its own interpolation of
 * the crossing point, in loop order — against the elements inserted so far, with libstdc++'s unique-insert rule:
 * the element found is the last one in order that is not greater than the new point; the new point is dropped when
 * that element is not less than it either.  At most 24 insertions, a handful of elements; only taken when the
 * owner's point lies within 1.5e-6 of an end point (the extra half tolerance covers the ulp-level differences
 * between the sharing cubes' interpolations). */
template <class WV>
__device__ __noinline__ CubeEdge weld_replay(const WV& W, const int G[3], unsigned long long target) {
    const Grid& g = W.g;
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    unsigned long long ekey[24];
    float ept[24]; /* coordinate along the edge's own axis; the other two are G's */
    int n = 0;
    const CubeEdge asking = weld_unkey(g, target);
    const float iso = weld_level(W, asking.i, asking.j, asking.k); /* repeating-surface mode: only this level's points can meet here */
    for (int ax = 0; ax < 3; ax++)
        for (int side = 0; side < 2; side++) { /* side 0: G is the edge's upper end point, 1: its lower end point */
            GridEdge E2{ax, G[0], G[1], G[2]};
            if (ax == 0) E2.vx -= 1 - side; else if (ax == 1) E2.vy -= 1 - side; else E2.vz -= 1 - side;
            if (E2.vx < 0 || E2.vy < 0 || E2.vz < g.kb) continue; /* the upper bounds fall out of weld_cube_ok */
            const int lo_idx = (ax == 0 ? E2.vx : ax == 1 ? E2.vy : E2.vz) + 1;
            if (lo_idx + 1 > g.M + 1) continue;
            const float* fp = W.F + (size_t)(E2.vz - g.kb + 1) * planep + (size_t)(E2.vy + 1) * rowp + (E2.vx + 1);
            const float fl = __ldg(fp), fu = __ldg(fp + (ax == 0 ? (size_t)1 : ax == 1 ? rowp : planep));
            if ((fl > iso) == (fu > iso)) continue;
            const float cl = W.cs[lo_idx], cu = W.cs[lo_idx + 1];
            const float pf = mcb_interp_ref(cl, cu, (g.iso - fl) / (fu - fl)); /* cube edge running lower -> upper */
            const float pb = mcb_interp_ref(cu, cl, (g.iso - fu) / (fl - fu)); /* cube edge running upper -> lower */
            for (int q = 0; q < 4; q++) {
                const int hi = 1 - (q >> 1), lo = 1 - (q & 1);
                CubeEdge o;
                if (ax == 0) { o.i = E2.vx; o.j = E2.vy - lo; o.k = E2.vz - hi; o.e = 2 * lo + 4 * hi; }
                else if (ax == 1) { o.i = E2.vx - lo; o.j = E2.vy; o.k = E2.vz - hi; o.e = (lo ? 1 : 3) + 4 * hi; }
                else { o.i = E2.vx - lo; o.j = E2.vy - hi; o.k = E2.vz; o.e = 8 + (hi ? (lo ? 2 : 3) : (lo ? 1 : 0)); }
                if (!weld_cube_ok(W, o.i, o.j, o.k, iso)) continue;
                const unsigned long long key = weld_key(g, o);
                if (key > target) continue; /* inserted after the point we are resolving */
                const bool forward = ((mcb_corner_ofs(mcb_edge_a(o.e)) >> ax) & 1) == 0;
                const float pt = forward ? pf : pb;
                if (!((double)fabsf(pt - W.cs[G[ax] + 1]) < 0.000002)) continue; /* cannot interact with anything at G */
                ekey[n] = key; ept[n] = pt; n++;
            }
        }
    /* insertion order */
    for (int a2 = 1; a2 < n; a2++) {
        const unsigned long long kk = ekey[a2];
        const float pp = ept[a2];
        int b2 = a2 - 1;
        while (b2 >= 0 && ekey[b2] > kk) { ekey[b2 + 1] = ekey[b2]; ept[b2 + 1] = ept[b2]; b2--; }
        ekey[b2 + 1] = kk; ept[b2 + 1] = pp;
    }
    const float gc[3] = {W.cs[G[0] + 1], W.cs[G[1] + 1], W.cs[G[2] + 1]};
    float sp[8][3];
    unsigned long long stok[8];
    int ns = 0;
    unsigned long long result = target;
    for (int ev = 0; ev < n; ev++) {
        const CubeEdge ce = weld_unkey(g, ekey[ev]);
        const int ax = ce.e >= 8 ? 2 : (ce.e & 1);
        float kpt[3] = {gc[0], gc[1], gc[2]};
        kpt[ax] = ept[ev];
        int j = -1;
        for (int q = 0; q < ns; q++)
            if (!weld_less(kpt, sp[q]) && (j < 0 || weld_less(sp[j], sp[q]))) j = q;
        unsigned long long tok;
        if (j >= 0 && !weld_less(sp[j], kpt)) tok = stok[j];
        else {
            tok = ekey[ev];
            if (ns < 8) { sp[ns][0] = kpt[0]; sp[ns][1] = kpt[1]; sp[ns][2] = kpt[2]; stok[ns] = tok; ns++; }
        }
        if (ekey[ev] == target) result = tok;
    }
    return weld_unkey(g, result);
}

/* Owner of a grid edge, closed form for the unconstrained grid: the first cube in loop order is the one furthest
 * back in the two other axes that still exists ((i,j) >= 0, k >= kb); with constraints, the candidate loop. */
template <class WV>
__device__ __forceinline__ void weld_owner_fast(const WV& W, const GridEdge& E, CubeEdge& o) {
    if (W.V != nullptr || W.present != nullptr || WV::kRepeat) { /* o comes in as the asking (cube, edge) */
        weld_owner(W, E, o, weld_level(W, o.i, o.j, o.k));
        return;
    }
    const int kb = W.g.kb;
    if (E.axis == 0) {
        const int lo = E.vy >= 1, hi = E.vz >= kb + 1;
        o.i = E.vx; o.j = E.vy - lo; o.k = E.vz - hi; o.e = 2 * lo + 4 * hi;
    } else if (E.axis == 1) {
        const int lo = E.vx >= 1, hi = E.vz >= kb + 1;
        o.i = E.vx - lo; o.j = E.vy; o.k = E.vz - hi; o.e = (lo ? 1 : 3) + 4 * hi;
    } else {
        const int lo = E.vx >= 1, hi = E.vy >= 1;
        o.i = E.vx - lo; o.j = E.vy - hi; o.k = E.vz; o.e = 8 + (hi ? (lo ? 2 : 3) : (lo ? 1 : 0));
    }
}

/* Does the crossing point of (cube, edge), as this cube interpolates it, sit on a grid vertex?  The sharing cubes'
 * interpolations differ by an ulp or two (< 2.5e-7), so 1.5e-6 catches every edge any of whose versions is within
 * the reference's 1e-6.  Returns 0 (no), 1 (lower end point) or 2 (upper end point). */
template <class WV>
__device__ __forceinline__ int weld_on_vertex(const WV& W, int i, int j, int k, int e) {
    const GridEdge E = grid_edge_of(i, j, k, e);
    bool cr;
    const CubeEdge me{i, j, k, e};
    const float p = weld_edge_point(W, me, E.axis, cr);
    const int base = (E.axis == 0 ? E.vx : E.axis == 1 ? E.vy : E.vz) + 1;
    if ((double)fabsf(p - W.cs[base]) < 0.0000015) return 1;
    if ((double)fabsf(p - W.cs[base + 1]) < 0.0000015) return 2;
    return 0;
}

/* (cube, crossing edge) -> the (cube, edge) whose insertion created the welded vertex the reference uses there.
 * on_vertex = weld_on_vertex() of this pair (computed once, in weld_count, and handed on in the vinfo words). */
template <class WV>
__device__ __forceinline__ CubeEdge weld_resolve(const WV& W, int i, int j, int k, int e, int on_vertex) {
    const GridEdge E = grid_edge_of(i, j, k, e);
    if (on_vertex == 0) { /* the up-to-four sharing cubes agree to within an ulp: the first inserter wins */
        CubeEdge own{i, j, k, e};
        weld_owner_fast(W, E, own);
        return own;
    }
    int G[3] = {E.vx, E.vy, E.vz};
    if (on_vertex == 2) G[E.axis] += 1; /* the grid vertex the point sits on */
    const CubeEdge me{i, j, k, e};
    return weld_replay(W, G, weld_key(W.g, me));
}

constexpr int kWeldCubes = 128;   /* active cubes per chunk */
constexpr int kWeldThreads = 256;

/* vinfo word per active cube: [31:0] index of its first new vertex, [43:32] edges for which the cube inserts a new
 * vertex, [55:44] edges whose crossing point sits on a grid vertex (which end point is recomputed on that rare path) */
struct WeldBuffers {
    const unsigned long long* __restrict__ rec;  /* [A] loop-ordered active cubes (compact_kernel) */
    const uint32_t* __restrict__ trioff;         /* [A] */
    const unsigned long long* __restrict__ item; /* [items] per 32-cube word: first record | active mask << 32 (compact_kernel) */
    unsigned long long* vinfo;                   /* [A] see above */
    uint32_t* chunk_new;                         /* [chunks] new vertices per chunk, then their exclusive scan */
    uint32_t WC;                                 /* 32-cube words per cube row */
};
#define MCB_VINFO_BASE(v) ((uint32_t)(v))
#define MCB_VINFO_NEW(v) ((uint32_t)((v) >> 32) & 0xFFFu)
#define MCB_VINFO_ONV(v) ((uint32_t)((v) >> 44) & 0xFFFu)

/* record index of an ACTIVE cube: first record of its 32-cube word + rank of the cube among the word's active cubes */
__device__ __forceinline__ uint32_t weld_find_cube(const WeldBuffers& B, const Grid& g, int i, int j, int k) {
    const size_t item = ((size_t)(k - g.kb) * g.M + j) * B.WC + (i >> 5);
    const unsigned long long w = B.item[item];
    return (uint32_t)w + (uint32_t)__popc((uint32_t)(w >> 32) & ((1u << (i & 31)) - 1u));
}

/* chunk prologue shared by weld_count and weld_emit: records -> shared memory, crossing-edge work list */
struct WeldChunk {
    uint32_t ijk[kWeldCubes];       /* i | j << 12 */
    uint16_t k[kWeldCubes];
    uint32_t mask[kWeldCubes];      /* new-vertex edges | on-vertex edges << 12 */
    uint16_t work[kWeldCubes * 12]; /* local cube << 4 | edge */
    uint32_t warp[kWeldThreads / 32];
};
__device__ __forceinline__ uint32_t weld_load_chunk(WeldChunk& sh, const unsigned long long* __restrict__ rec,
                                                    unsigned long long c0, int n, unsigned long long* rec_out) {
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    uint32_t emask = 0;
    unsigned long long r = 0;
    if (t < n) {
        r = rec[c0 + t];
        const int code = (int)((r >> 36) & 0xFF);
        sh.ijk[t] = (uint32_t)(r & 0xFFFFFF);
        sh.k[t] = (uint16_t)((r >> 24) & 0xFFF);
#pragma unroll
        for (int e = 0; e < 12; e++)
            emask |= (uint32_t)(((code >> mcb_edge_a(e)) ^ (code >> mcb_edge_b(e))) & 1) << e;
    }
    if (rec_out) *rec_out = r;
    const uint32_t nv = __popc(emask);
    uint32_t inc = nv;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
    if (lane == 31) sh.warp[warp] = inc;
    __syncthreads();
    uint32_t wbase = inc - nv, total = 0;
#pragma unroll
    for (int w2 = 0; w2 < kWeldThreads / 32; w2++) { if (w2 < warp) wbase += sh.warp[w2]; total += sh.warp[w2]; }
    while (emask) {
        const int e = __ffs(emask) - 1;
        emask &= emask - 1;
        sh.work[wbase++] = (uint16_t)((t << 4) | e);
    }
    return total;
}

/* marks, per active cube, the edges for which it inserts a new vertex and those whose point sits on a grid vertex */
template <class WV>
__global__ void __launch_bounds__(kWeldThreads)
weld_count_kernel(const WV W, const WeldBuffers B, const Counters* __restrict__ ctr, unsigned long long cap_active) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    __shared__ WeldChunk sh;
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    const unsigned long long nchunks = (A + kWeldCubes - 1) / kWeldCubes;
    const int t = threadIdx.x;
    for (unsigned long long chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        __syncthreads();
        const unsigned long long c0 = chunk * kWeldCubes;
        const int n = (int)((A - c0) < (unsigned long long)kWeldCubes ? (A - c0) : kWeldCubes);
        if (t < kWeldCubes) sh.mask[t] = 0;
        const uint32_t total_v = weld_load_chunk(sh, B.rec, c0, n, nullptr);
        __syncthreads();
        for (uint32_t q = t; q < total_v; q += kWeldThreads) {
            const uint32_t wk = sh.work[q];
            const int lc = (int)(wk >> 4), e = (int)(wk & 15u);
            const int i = (int)(sh.ijk[lc] & 0xFFF), j = (int)(sh.ijk[lc] >> 12), k = (int)sh.k[lc];
            const int onv = weld_on_vertex(W, i, j, k, e);
            const CubeEdge v = weld_resolve(W, i, j, k, e, onv);
            uint32_t bits = onv ? (1u << (12 + e)) : 0u;
            if (v.i == i && v.j == j && v.k == k && v.e == e) bits |= 1u << e;
            if (bits) atomicOr(&sh.mask[lc], bits);
        }
        __syncthreads();
        uint32_t mine = 0;
        if (t < n) { B.vinfo[c0 + t] = (unsigned long long)sh.mask[t] << 32; mine = __popc(sh.mask[t] & 0xFFFu); }
#pragma unroll
        for (int d = 16; d; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
        if ((t & 31) == 0) sh.warp[t >> 5] = mine;
        __syncthreads();
        if (t == 0) {
            uint32_t s2 = 0;
#pragma unroll
            for (int w2 = 0; w2 < kWeldThreads / 32; w2++) s2 += sh.warp[w2];
            B.chunk_new[chunk] = s2;
        }
    }
}

/* The same marks for the plain grid (no constraints, no seed mode, no per-cube levels), a thread per CUBE instead of a
 * thread per crossing edge.  There the owner of a grid edge has a closed form (weld_owner_fast): a cube is the first in
 * loop order to contain the edges on its far faces, and those on its near faces only where the grid or the slab begins —
 * pure index arithmetic.  What needs field values is the rare case of a crossing point sitting on a grid vertex, where
 * the replay decides: a multiplication-only test on the cube's eight corner values rules it out for nearly every edge
 * (a point within 1.5e-6 of an end point has |t| h or |1 - t| h below 3e-6, with t = (iso - f_a) / (f_b - f_a)), and only
 * the edges it cannot rule out take the exact functions above.  Same vinfo words, a fraction of the work. */
__global__ void __launch_bounds__(kWeldCubes, 12)
weld_count_fast_kernel(const WeldView W, const WeldBuffers B, const ClsTables* __restrict__ gtb, const Counters* __restrict__ ctr,
                       unsigned long long cap_active) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    __shared__ uint32_t warp_s[kWeldCubes / 32];
    const Grid& g = W.g;
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    const unsigned long long nchunks = (A + kWeldCubes - 1) / kWeldCubes;
    const int t = threadIdx.x;
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    for (unsigned long long chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        __syncthreads();
        const unsigned long long a = chunk * kWeldCubes + t;
        uint32_t bits = 0;
        if (a < A) {
            const unsigned long long r = B.rec[a];
            const int i = (int)(r & 0xFFF), j = (int)((r >> 12) & 0xFFF), k = (int)((r >> 24) & 0xFFF), code = (int)((r >> 36) & 0xFF);
            const uint32_t emask = __ldg(gtb->emask + code);
            const uint32_t X0 = i == 0, Y0 = j == 0, Z0 = k == g.kb;
            /* edges 5, 6, 10 lie on the far faces; the others need the cube to be first along the axes they are near on */
            uint32_t own = (1u << 5) | (1u << 6) | (1u << 10) | ((Y0 & Z0) << 0) | (Z0 << 2) | (Y0 << 4) | (Z0 << 1) | ((X0 & Z0) << 3) |
                           (X0 << 7) | ((X0 & Y0) << 8) | (Y0 << 9) | (X0 << 11);
            const float* f0 = W.F + (size_t)(k - g.kb + 1) * planep + (size_t)(j + 1) * rowp + (i + 1);
            float f[8];
#pragma unroll
            for (int v = 0; v < 8; v++) {
                const int o = mcb_corner_ofs(v);
                f[v] = __ldg(f0 + (size_t)(o >> 2) * planep + (size_t)((o >> 1) & 1) * rowp + (o & 1));
            }
            const float hx = W.cs[i + 2] - W.cs[i + 1], hy = W.cs[j + 2] - W.cs[j + 1], hz = W.cs[k + 2] - W.cs[k + 1];
            uint32_t maybe = 0; /* crossing edges whose point may sit on a grid vertex */
#pragma unroll
            for (int e = 0; e < 12; e++) {
                const float fa = f[mcb_edge_a(e)], fb = f[mcb_edge_b(e)];
                const float h = fabsf(e >= 8 ? hz : (e & 1) ? hy : hx);
                const float d1 = fabsf(g.iso - fa), d2 = fabsf(fb - fa), d3 = fabsf(fb - g.iso);
                const bool clear = d1 * h > 3e-6f * d2 && d3 * h > 3e-6f * d2; /* NaN / inf / zero denominators compare false */
                maybe |= clear ? 0u : 1u << e;
            }
            maybe &= emask;
            bits = emask & own;
            while (maybe) { /* rare: the exact path of weld_count_kernel for this edge */
                const int e = __ffs(maybe) - 1;
                maybe &= maybe - 1;
                const int onv = weld_on_vertex(W, i, j, k, e);
                if (onv == 0) continue;
                const CubeEdge v = weld_resolve(W, i, j, k, e, onv);
                bits |= 1u << (12 + e);
                if (v.i == i && v.j == j && v.k == k && v.e == e) bits |= 1u << e; else bits &= ~(1u << e);
            }
            B.vinfo[a] = (unsigned long long)bits << 32;
        }
        uint32_t mine = __popc(bits & 0xFFFu);
#pragma unroll
        for (int d = 16; d; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
        if ((t & 31) == 0) warp_s[t >> 5] = mine;
        __syncthreads();
        if (t == 0) {
            uint32_t s2 = 0;
#pragma unroll
            for (int w2 = 0; w2 < kWeldCubes / 32; w2++) s2 += warp_s[w2];
            B.chunk_new[chunk] = s2;
        }
    }
}

/* exclusive scan of the per-chunk new-vertex counts (one block; a thread takes kWeldScanPer consecutive chunks, so the
 * 19 000 chunks of a 1024^3 sphere are four rounds of the block) */
constexpr int kWeldScanPer = 8;
__global__ void __launch_bounds__(1024)
weld_scan_kernel(uint32_t* __restrict__ chunk_new, Counters* __restrict__ ctr, unsigned long long cap_active) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry_s;
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    const unsigned long long nchunks = (A + kWeldCubes - 1) / kWeldCubes;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (unsigned long long b0 = 0; b0 < nchunks; b0 += 1024ull * kWeldScanPer) {
        const unsigned long long c0 = b0 + (unsigned long long)t * kWeldScanPer;
        uint32_t v[kWeldScanPer];
        unsigned long long mine = 0;
#pragma unroll
        for (int q = 0; q < kWeldScanPer; q++) { v[q] = c0 + q < nchunks ? chunk_new[c0 + q] : 0u; mine += v[q]; }
        unsigned long long inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const unsigned long long u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) warp_tot[warp] = inc;
        __syncthreads();
        unsigned long long base = carry_s;
        for (int w2 = 0; w2 < warp; w2++) base += warp_tot[w2];
        unsigned long long run = base + inc - mine;
#pragma unroll
        for (int q = 0; q < kWeldScanPer; q++) { if (c0 + q < nchunks) chunk_new[c0 + q] = (uint32_t)run; run += v[q]; }
        __syncthreads();
        if (t == 1023) carry_s = base + inc;
        __syncthreads();
    }
    if (t == 0) ctr->vertices = carry_s;
}

/* per-cube first vertex index: chunk base + exclusive scan of the new-vertex counts inside the chunk */
__global__ void __launch_bounds__(kWeldCubes)
weld_base_kernel(const WeldBuffers B, const Counters* __restrict__ ctr, unsigned long long cap_active) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    __shared__ uint32_t warp_s[kWeldCubes / 32];
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    const unsigned long long nchunks = (A + kWeldCubes - 1) / kWeldCubes;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (unsigned long long chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        __syncthreads();
        const unsigned long long c = chunk * kWeldCubes + t;
        const unsigned long long vi = c < A ? B.vinfo[c] : 0ull;
        const uint32_t nv = (uint32_t)__popc(MCB_VINFO_NEW(vi));
        uint32_t inc = nv;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) warp_s[warp] = inc;
        __syncthreads();
        uint32_t base = B.chunk_new[chunk] + inc - nv;
        for (int w2 = 0; w2 < warp; w2++) base += warp_s[w2];
        if (c < A) B.vinfo[c] = (vi & 0xFFFFFFFF00000000ull) | base;
    }
}

/* first vertex and first triangle of K+1 chunk boundaries (boundary j = chunk j * nchunks / K): what the host needs
 * to stream the mesh out in K ranges while weld_emit is still producing the later ones */
__global__ void weld_bounds_kernel(const WeldBuffers B, const Counters* __restrict__ ctr, unsigned long long cap_active, int K,
                                   unsigned long long* __restrict__ out /* [3 * (K + 1)]: chunk, vertex, triangle */) {
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    const unsigned long long nchunks = (A + kWeldCubes - 1) / kWeldCubes;
    const int j = threadIdx.x;
    if (j > K) return;
    const unsigned long long c = j == K ? nchunks : nchunks * (unsigned long long)j / (unsigned long long)K;
    out[3 * j] = c;
    out[3 * j + 1] = c < nchunks ? (unsigned long long)B.chunk_new[c] : ctr->vertices;
    out[3 * j + 2] = c < nchunks ? (unsigned long long)B.trioff[c * kWeldCubes] : ctr->triangles;
}

template <bool NORMALS, class WV>
__global__ void __launch_bounds__(kWeldThreads)
weld_emit_kernel(const WV W, const WeldBuffers B, const Counters* __restrict__ ctr, unsigned long long cap_active,
                 unsigned long long cap_verts, unsigned long long cap_tris, float* __restrict__ vertex_list,
                 float* __restrict__ vertex_nrm, uint32_t* __restrict__ tri_list, unsigned long long chunk_begin,
                 unsigned long long chunk_end /* chunks [begin,end) of kWeldCubes cubes: the host streams the mesh out range by range */) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    __shared__ WeldChunk sh;
    __shared__ uint32_t eidx[kWeldCubes * 12]; /* welded vertex index of [cube][edge] */
    __shared__ uint8_t tri2cube[kWeldCubes * 5]; /* chunk-local triangle -> local cube (a cube has at most 5) */
    __shared__ uint32_t off_s[kWeldCubes + 1];
    __shared__ uint64_t triw_s[kWeldCubes];
    __shared__ uint32_t vb_s[kWeldCubes];
    const Grid& g = W.g;
    unsigned long long A = ctr->active, T = ctr->triangles;
    if (A > cap_active) A = cap_active;
    unsigned long long nchunks = (A + kWeldCubes - 1) / kWeldCubes;
    if (nchunks > chunk_end) nchunks = chunk_end;
    const int t = threadIdx.x;
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    for (unsigned long long chunk = chunk_begin + blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        __syncthreads();
        const unsigned long long c0 = chunk * kWeldCubes;
        const int n = (int)((A - c0) < (unsigned long long)kWeldCubes ? (A - c0) : kWeldCubes);
        unsigned long long r;
        const uint32_t total_v = weld_load_chunk(sh, B.rec, c0, n, &r);
        if (t < n) {
            const unsigned long long vi = B.vinfo[c0 + t];
            off_s[t] = B.trioff[c0 + t];
            triw_s[t] = mcb_tri_word((int)((r >> 44) & 0xFF));
            sh.mask[t] = (uint32_t)(vi >> 32);
            vb_s[t] = MCB_VINFO_BASE(vi);
        }
        /* end of the chunk's output range.  In a pass with too small buffers (repeated by the host) the last cube gets no
         * output; its offset is read from global memory, NOT from off_s[n - 1], which another warp is writing right now */
        if (t == 0) off_s[n] = (c0 + n < A) ? B.trioff[c0 + n] : (A == ctr->active ? (uint32_t)T : B.trioff[c0 + n - 1]);
        __syncthreads();
        for (uint32_t q = t; q < total_v; q += kWeldThreads) {
            const uint32_t wk = sh.work[q];
            const int lc = (int)(wk >> 4), e = (int)(wk & 15u);
            const int i = (int)(sh.ijk[lc] & 0xFFF), j = (int)(sh.ijk[lc] >> 12), k = (int)sh.k[lc];
            const uint32_t m = sh.mask[lc];
            uint32_t idx;
            if ((m >> e) & 1u) { /* this cube inserts the vertex of this edge: write it (add_point, marching.cpp:627-643) */
                idx = vb_s[lc] + (uint32_t)__popc(m & ((1u << e) - 1u));
                if (idx < cap_verts) {
                    const int oa = mcb_corner_ofs(mcb_edge_a(e)), ob = mcb_corner_ofs(mcb_edge_b(e));
                    const int xa = i + 1 + (oa & 1), ya = j + 1 + ((oa >> 1) & 1), za = k + 1 + ((oa >> 2) & 1);
                    const int xb = i + 1 + (ob & 1), yb = j + 1 + ((ob >> 1) & 1), zb = k + 1 + ((ob >> 2) & 1);
                    const float* pa = W.F + (size_t)(za - g.kb) * planep + (size_t)ya * rowp + xa;
                    const float* pb = W.F + (size_t)(zb - g.kb) * planep + (size_t)yb * rowp + xb;
                    const float f1 = __ldg(pa), f2 = __ldg(pb);
                    const float tq = (g.iso - f1) / (f2 - f1);
                    float* out = vertex_list + 3ull * idx;
                    out[0] = mcb_interp_ref(W.cs[xa], W.cs[xb], tq);
                    out[1] = mcb_interp_ref(W.cs[ya], W.cs[yb], tq);
                    out[2] = mcb_interp_ref(W.cs[za], W.cs[zb], tq);
                    if (NORMALS) { /* central differences with IEEE divisions, blended along the grid edge, normalised by 1 / sqrtf */
                        const float* cs = W.cs;
                        const float gxa = (__ldg(pa + 1) - __ldg(pa - 1)) / (cs[xa + 1] - cs[xa - 1]);
                        const float gya = (__ldg(pa + rowp) - __ldg(pa - rowp)) / (cs[ya + 1] - cs[ya - 1]);
                        const float gza = (__ldg(pa + planep) - __ldg(pa - planep)) / (cs[za + 1] - cs[za - 1]);
                        const float gxb = (__ldg(pb + 1) - __ldg(pb - 1)) / (cs[xb + 1] - cs[xb - 1]);
                        const float gyb = (__ldg(pb + rowp) - __ldg(pb - rowp)) / (cs[yb + 1] - cs[yb - 1]);
                        const float gzb = (__ldg(pb + planep) - __ldg(pb - planep)) / (cs[zb + 1] - cs[zb - 1]);
                        float nx, ny, nz;
                        blend_edge_normal(oa < ob, g.iso, f1, f2, tq, gxa, gya, gza, gxb, gyb, gzb, nx, ny, nz);
                        const float inv = 1.0f / sqrtf(nx * nx + ny * ny + nz * nz);
                        float* on = vertex_nrm + 3ull * idx;
                        on[0] = nx * inv; on[1] = ny * inv; on[2] = nz * inv;
                    }
                }
            } else { /* somebody else inserted it: the edge's owner, or the replay's answer on a grid vertex */
                const int onv = ((m >> (12 + e)) & 1u) ? weld_on_vertex(W, i, j, k, e) : 0;
                const CubeEdge v = weld_resolve(W, i, j, k, e, onv);
                unsigned long long vi;
                if (v.i == i && v.j == j && v.k == k) vi = ((unsigned long long)m << 32) | vb_s[lc];
                else { /* the owner's record; beyond the (too small) buffers of a pass the host is about to repeat there is nothing to read */
                    const uint32_t owner = weld_find_cube(B, g, v.i, v.j, v.k);
                    vi = owner < A ? B.vinfo[owner] : 0ull;
                }
                idx = MCB_VINFO_BASE(vi) + (uint32_t)__popc(MCB_VINFO_NEW(vi) & ((1u << v.e) - 1u));
            }
            eidx[lc * 12 + e] = idx;
        }
        if (t < n) {
            const uint32_t first = off_s[t] - off_s[0], cnt = off_s[t + 1] - off_s[t];
            for (uint32_t q2 = 0; q2 < cnt && q2 < 5u; q2++) tri2cube[first + q2] = (uint8_t)t;
        }
        __syncthreads();
        const unsigned long long v_begin = 3ull * off_s[0], v_end = 3ull * off_s[n];
        for (unsigned long long ov = v_begin + t; ov < v_end; ov += kWeldThreads) {
            const uint32_t tri = (uint32_t)(ov / 3);
            const int corner = (int)(ov - 3ull * tri);
            const int lo = (int)tri2cube[tri - off_s[0]]; /* local cube this triangle belongs to */
            const int lt = (int)(tri - off_s[lo]);
            const int e = (int)((triw_s[lo] >> (4 * (3 * lt + corner))) & 0xF);
            if (tri < cap_tris) tri_list[ov] = eidx[lo * 12 + e];
        }
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K5  normal.h normals (mcb_set_normals(ctx, 2)): CalculateNormal, normal.h:3-42, on the indexed mesh — bit-exact.
 *     The reference walks the triangles in order and does vNormal[i] = faceNormal + vNormal[i] for the three corners
 *     of each, then glm::normalize.  fp32 addition is not associative, so the result depends on that order: per
 *     vertex the additions happen in ascending (triangle, corner) order, a repeated index accumulating twice.
 *     Here: face normals once per triangle (glm::cross of B-A and C-A, no FMA contraction); a CSR list of the
 *     corners referencing each vertex (count, scan, fill by atomic cursor), sorted per vertex so that the sum runs in
 *     the reference's order; x * (1.0f / sqrt(dot)) like glm 0.9.5.3 (func_geometric.inl:257-267,
 *     func_exponential.inl:226-229).
 * ------------------------------------------------------------------------------------------------------------- */
/* A welded mesh that did not fit its buffers is incomplete (indices point past the vertex list); the host grows the
 * buffers and repeats the pass, and until then this stage must not touch it. */
__global__ void nh_gate_kernel(Counters* __restrict__ ctr, unsigned long long cap_active, unsigned long long cap_verts, unsigned long long cap_tris) {
    const bool fits = ctr->active <= cap_active && ctr->vertices <= cap_verts && ctr->triangles <= cap_tris;
    ctr->nh_vertices = fits ? ctr->vertices : 0ull;
    ctr->nh_triangles = fits ? ctr->triangles : 0ull;
}
__global__ void __launch_bounds__(256)
nh_face_normals_kernel(const float* __restrict__ vl, const uint32_t* __restrict__ tl, const Counters* __restrict__ ctr,
                       unsigned long long cap_tris, float* __restrict__ fn, uint32_t* __restrict__ count) {
    unsigned long long T = ctr->nh_triangles;
    if (T > cap_tris) T = cap_tris;
    for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t i1 = tl[3 * t], i2 = tl[3 * t + 1], i3 = tl[3 * t + 2];
        const float ax = vl[3ull * i1], ay = vl[3ull * i1 + 1], az = vl[3ull * i1 + 2];
        const float bx = vl[3ull * i2] - ax, by = vl[3ull * i2 + 1] - ay, bz = vl[3ull * i2 + 2] - az;
        const float cx = vl[3ull * i3] - ax, cy = vl[3ull * i3 + 1] - ay, cz = vl[3ull * i3 + 2] - az;
        fn[3 * t] = by * cz - cy * bz;
        fn[3 * t + 1] = bz * cx - cz * bx;
        fn[3 * t + 2] = bx * cy - cx * by;
        atomicAdd(count + i1, 1u); atomicAdd(count + i2, 1u); atomicAdd(count + i3, 1u);
    }
}

/* exclusive scan of n counters in three steps (n read from the device): block sums, one-block scan, local scan */
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock)
scan_block_sums_kernel(const uint32_t* __restrict__ in, const unsigned long long* __restrict__ n_ptr, uint32_t* __restrict__ sums) {
    __shared__ uint32_t warp_s[32];
    const unsigned long long n = *n_ptr;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (unsigned long long b0 = (unsigned long long)blockIdx.x * kScanBlock; b0 < n; b0 += (unsigned long long)gridDim.x * kScanBlock) {
        uint32_t v = b0 + t < n ? in[b0 + t] : 0u;
#pragma unroll
        for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if (lane == 0) warp_s[warp] = v;
        __syncthreads();
        if (warp == 0) {
            uint32_t s = warp_s[lane];
#pragma unroll
            for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
            if (lane == 0) sums[b0 / kScanBlock] = s;
        }
        __syncthreads();
    }
}
__global__ void __launch_bounds__(kScanBlock)
scan_sums_kernel(uint32_t* __restrict__ sums, const unsigned long long* __restrict__ n_ptr) {
    __shared__ uint32_t warp_s[32];
    __shared__ uint32_t carry_s;
    const unsigned long long nb = (*n_ptr + kScanBlock - 1) / kScanBlock;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (unsigned long long b0 = 0; b0 < nb; b0 += kScanBlock) {
        const uint32_t v = b0 + t < nb ? sums[b0 + t] : 0u;
        uint32_t inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) warp_s[warp] = inc;
        __syncthreads();
        uint32_t base = carry_s;
        for (int w2 = 0; w2 < warp; w2++) base += warp_s[w2];
        if (b0 + t < nb) sums[b0 + t] = base + inc - v;
        __syncthreads();
        if (t == kScanBlock - 1) carry_s = base + inc;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(kScanBlock)
scan_apply_kernel(const uint32_t* __restrict__ in, const uint32_t* __restrict__ sums, const unsigned long long* __restrict__ n_ptr,
                  uint32_t* __restrict__ out) {
    __shared__ uint32_t warp_s[32];
    const unsigned long long n = *n_ptr;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (unsigned long long b0 = (unsigned long long)blockIdx.x * kScanBlock; b0 < n; b0 += (unsigned long long)gridDim.x * kScanBlock) {
        const uint32_t v = b0 + t < n ? in[b0 + t] : 0u;
        uint32_t inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) warp_s[warp] = inc;
        __syncthreads();
        uint32_t base = sums[b0 / kScanBlock];
        for (int w2 = 0; w2 < warp; w2++) base += warp_s[w2];
        if (b0 + t < n) out[b0 + t] = base + inc - v;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
nh_fill_kernel(const uint32_t* __restrict__ tl, const Counters* __restrict__ ctr, unsigned long long cap_tris,
               const uint32_t* __restrict__ start, uint32_t* __restrict__ cursor, uint32_t* __restrict__ adj) {
    unsigned long long T = ctr->nh_triangles;
    if (T > cap_tris) T = cap_tris;
    const unsigned long long n = 3 * T;
    for (unsigned long long c = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t v = tl[c];
        adj[start[v] + atomicAdd(cursor + v, 1u)] = (uint32_t)c;
    }
}

__global__ void __launch_bounds__(128)
nh_accumulate_kernel(const float* __restrict__ fn, const uint32_t* __restrict__ start, const uint32_t* __restrict__ count,
                     uint32_t* __restrict__ adj, const Counters* __restrict__ ctr, unsigned long long cap_verts,
                     float* __restrict__ vnrm) {
    unsigned long long Vn = ctr->nh_vertices;
    if (Vn > cap_verts) Vn = cap_verts;
    for (unsigned long long v = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; v < Vn; v += (unsigned long long)gridDim.x * blockDim.x) {
        uint32_t* a = adj + start[v];
        const uint32_t n = count[v];
        for (uint32_t i = 1; i < n; i++) { /* ascending corner order = the order of the reference's triangle loop */
            const uint32_t key = a[i];
            uint32_t j = i;
            while (j > 0 && a[j - 1] > key) { a[j] = a[j - 1]; j--; }
            a[j] = key;
        }
        float ox = 0.f, oy = 0.f, oz = 0.f; /* vNormal.resize(): zero-initialised glm::vec3 */
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t t = a[i] / 3u;
            ox = fn[3ull * t] + ox; oy = fn[3ull * t + 1] + oy; oz = fn[3ull * t + 2] + oz;
        }
        const float inv = 1.0f / sqrtf(ox * ox + oy * oy + oz * oz);
        vnrm[3 * v] = ox * inv; vnrm[3 * v + 1] = oy * inv; vnrm[3 * v + 2] = oz * inv;
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K6  seed mode (Marching::seed_mode / set_seed, marching.cpp:42-137, 310-331): keep only the cubes reachable from
 *     the cube containing the seed point by stepping across cube faces that carry a crossing edge
 *     (find_cubes_for_seeding: a face is crossed when its four corner signs are not all equal; the neighbour must lie
 *     inside the reference's bound check and, with constraints, be a cube the loop would not skip).  The reference
 *     does this as a BFS and emits in BFS order; here it is a monotone marking over the compacted active-cube list
 *     (0 = untouched, 1 = reached, 2 = reached and expanded) repeated until nothing changes, followed by a scan that
 *     compacts the reached cubes — so the same SET of cubes and triangles comes out, in the full-grid loop order.
 * ------------------------------------------------------------------------------------------------------------- */
struct SeedBuffers {
    const unsigned long long* __restrict__ rec;
    const unsigned long long* __restrict__ item; /* per 32-cube word: first record | active mask << 32 */
    uint32_t WC;
    uint8_t* mark;      /* [A] */
    uint32_t* changed;  /* [1] */
};
__device__ __forceinline__ bool seed_lookup(const SeedBuffers& B, const Grid& g, int i, int j, int k, uint32_t* idx) {
    const size_t item = ((size_t)(k - g.kb) * g.M + j) * B.WC + (i >> 5);
    const unsigned long long w = B.item[item];
    const uint32_t mask = (uint32_t)(w >> 32);
    if (!((mask >> (i & 31)) & 1u)) return false; /* note: words without any active cube are never read (see caller) */
    *idx = (uint32_t)w + (uint32_t)__popc(mask & ((1u << (i & 31)) - 1u));
    return true;
}
/* the seed cube: Marching::get_starting_seed_grid (marching.cpp:104-113) gives its index per axis on the host */
__global__ void seed_init_kernel(const SeedBuffers B, const Grid g, const Counters* __restrict__ ctr, unsigned long long cap_active,
                                 int si, int sj, int sk) {
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    /* the seed cube's word may hold no active cube at all, in which case its item word was never written: find the
     * record by bisection over the loop-ordered list instead */
    const unsigned long long key = (unsigned long long)si | ((unsigned long long)sj << 12) | ((unsigned long long)sk << 24);
    unsigned long long lo = 0, hi = A;
    while (lo < hi) {
        const unsigned long long mid = (lo + hi) >> 1;
        if ((B.rec[mid] & 0xFFFFFFFFFull) < key) lo = mid + 1; else hi = mid;
    }
    if (lo < A && (B.rec[lo] & 0xFFFFFFFFFull) == key) { B.mark[lo] = 1; *B.changed = 1u; }
}
__global__ void __launch_bounds__(256)
seed_sweep_kernel(const SeedBuffers B, const WeldView W, const Counters* __restrict__ ctr, unsigned long long cap_active, double half_step) {
    const Grid& g = W.g;
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    for (unsigned long long c = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; c < A; c += (unsigned long long)gridDim.x * blockDim.x) {
        if (*(volatile uint8_t*)(B.mark + c) != 1) continue;
        B.mark[c] = 2;
        const unsigned long long r = B.rec[c];
        const int i = (int)(r & 0xFFF), j = (int)((r >> 12) & 0xFFF), k = (int)((r >> 24) & 0xFFF), code = (int)((r >> 36) & 0xFF);
#pragma unroll
        for (int f = 0; f < 6; f++) {
            const int b0 = (code >> mcb_face_corner(f, 0)) & 1, b1 = (code >> mcb_face_corner(f, 1)) & 1;
            const int b2 = (code >> mcb_face_corner(f, 2)) & 1, b3 = (code >> mcb_face_corner(f, 3)) & 1;
            if (b0 == b1 && b1 == b2 && b2 == b3) continue; /* no edge of this face is crossed */
            /* cube_face_normal, marching_lookup.h:43-50 */
            const int ni = i + (f == 1 ? 1 : f == 3 ? -1 : 0), nj = j + (f == 4 ? 1 : f == 5 ? -1 : 0), nk = k + (f == 2 ? 1 : f == 0 ? -1 : 0);
            if (!weld_cube_ok(W, ni, nj, nk)) continue;
            /* marching.cpp:81-84: origin >= -1 - h/2 and origin + h/2 <= 1 on every axis, evaluated in double */
            const double ox = (double)W.cs[ni + 1], oy = (double)W.cs[nj + 1], oz = (double)W.cs[nk + 1];
            if (!(ox >= -1.0 - half_step && ox + half_step <= 1.0 && oy >= -1.0 - half_step && oy + half_step <= 1.0 &&
                  oz >= -1.0 - half_step && oz + half_step <= 1.0)) continue;
            uint32_t n;
            if (!seed_lookup(B, g, ni, nj, nk, &n)) continue; /* the neighbour shares the crossed face, so it is active */
            if (*(volatile uint8_t*)(B.mark + n) == 0) { B.mark[n] = 1; *B.changed = 1u; }
        }
    }
}
/* keep[c], kept triangle count -> two u32 arrays for the scans */
__global__ void __launch_bounds__(256)
seed_flags_kernel(const SeedBuffers B, const ClsTables* __restrict__ gtb, const Counters* __restrict__ ctr, unsigned long long cap_active,
                  uint32_t* __restrict__ keep, uint32_t* __restrict__ ktri) {
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    for (unsigned long long c = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; c < A; c += (unsigned long long)gridDim.x * blockDim.x) {
        const bool k = B.mark[c] != 0;
        keep[c] = k ? 1u : 0u;
        ktri[c] = k ? (uint32_t)__ldg(gtb->ntri + (int)((B.rec[c] >> 44) & 0xFF)) : 0u;
    }
}
__global__ void __launch_bounds__(256)
seed_scatter_kernel(const SeedBuffers B, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ ktri,
                    const uint32_t* __restrict__ pa, const uint32_t* __restrict__ pt, Counters* __restrict__ ctr,
                    unsigned long long cap_active, unsigned long long* __restrict__ rec2, uint32_t* __restrict__ trioff2) {
    unsigned long long A = ctr->active;
    if (A > cap_active) A = cap_active;
    for (unsigned long long c = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; c < A; c += (unsigned long long)gridDim.x * blockDim.x) {
        if (keep[c]) { rec2[pa[c]] = B.rec[c]; trioff2[pa[c]] = pt[c]; }
        if (c == A - 1) { ctr->seed_active = (unsigned long long)pa[c] + keep[c]; ctr->seed_triangles = (unsigned long long)pt[c] + ktri[c]; }
    }
}
/* the counters switch over to the kept set once every reader of the old count is done */
__global__ void seed_commit_kernel(Counters* __restrict__ ctr) {
    ctr->active = ctr->seed_active;
    ctr->triangles = ctr->seed_triangles;
}
/* rebuild the per-word look-up (first record | mask) for the kept, compacted list */
__global__ void __launch_bounds__(256)
seed_items_kernel(const unsigned long long* __restrict__ rec2, const Grid g, uint32_t WC, const Counters* __restrict__ ctr,
                  unsigned long long* __restrict__ item) {
    const unsigned long long A = ctr->active;
    for (unsigned long long c = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; c < A; c += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long wkey = rec2[c] & 0xFFFFFFFE0ull; /* k : j : i / 32 */
        if (c > 0 && (rec2[c - 1] & 0xFFFFFFFE0ull) == wkey) continue; /* not the first kept cube of its word */
        uint32_t mask = 0;
        for (unsigned long long d = c; d < A && (rec2[d] & 0xFFFFFFFE0ull) == wkey; d++) mask |= 1u << (uint32_t)(rec2[d] & 31u);
        const int i = (int)(rec2[c] & 0xFFF), j = (int)((rec2[c] >> 12) & 0xFFF), k = (int)((rec2[c] >> 24) & 0xFFF);
        item[((size_t)(k - g.kb) * g.M + j) * WC + (i >> 5)] = (c & 0xFFFFFFFFull) | ((unsigned long long)mask << 32);
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K7  inspect: Marching::calculate_step(x_0, y_0, z_0) (marching.cpp:456-595) for ONE cube at an arbitrary origin —
 *     what the GUI's step-by-step / movie mode shows per cube (Step_Data, marching.h:15-23).  One thread; the point
 *     programs of the surface and of the constraints in use.
 * ------------------------------------------------------------------------------------------------------------- */
struct StepOut { /* mirrors mcb_step_data (include/mcb.h) */
    float corner_coords[24];
    float corner_values[8];
    float intersect_coord[36];
    int32_t edge_list[12];
    int32_t tri_vlist[15];
    int32_t n_edges, n_tri_idx, cube_code, table_idx, skipped;
    float surf_constant;
};
struct InspectCons {
    int n;            /* constraints in use */
    int op[3];        /* 0 '>', 1 '<', 2 '>=', 3 '<=' */
    float rhs[3];
};
__global__ void inspect_cube_kernel(const mcb_program* __restrict__ progs /* [0] surface, [1..3] constraint lhs */, const InspectCons cons,
                                    const int cons_slot0, const int cons_slot1, const int cons_slot2,
                                    float x0, float y0, float z0, float step, float sx, float sy, float sz, float iso_in,
                                    int repeat, float rstep, const ClsTables* __restrict__ gtb, StepOut* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    StepOut o;
    const float x1 = x0 + step, y1 = y0 + step, z1 = z0 + step; /* marching.cpp:458-460 */
    const float cc[24] = {x0, y0, z0, x1, y0, z0, x1, y1, z0, x0, y1, z0, x0, y0, z1, x1, y0, z1, x1, y1, z1, x0, y1, z1};
    for (int q = 0; q < 24; q++) o.corner_coords[q] = cc[q];
    for (int q = 0; q < 8; q++) o.corner_values[q] = 0.f;
    o.n_edges = 0; o.n_tri_idx = 0; o.cube_code = 0; o.table_idx = 0; o.skipped = 0;
    const int slots[3] = {cons_slot0, cons_slot1, cons_slot2};
    for (int v = 0; v < 8 && !o.skipped; v++) {
        const float X = sx * cc[3 * v], Y = sy * cc[3 * v + 1], Z = sz * cc[3 * v + 2]; /* Marching::evaluate, marching.cpp:211 */
        for (int c = 0; c < cons.n; c++) { /* check_constraints, marching.cpp:255-280 */
            const mcb_program& p = progs[slots[c]];
            const float lhs = mcb_interp_scalar(p.code, p.n, p.k, X, Y, Z, nullptr, nullptr, nullptr);
            const int op = cons.op[c];
            const bool ok = op == 0 ? lhs > cons.rhs[c] : op == 1 ? lhs < cons.rhs[c] : op == 2 ? lhs >= cons.rhs[c] : lhs <= cons.rhs[c];
            if (!ok) o.skipped = 1;
        }
        if (o.skipped) break;
        o.corner_values[v] = mcb_interp_scalar(progs[0].code, progs[0].n, progs[0].k, X, Y, Z, nullptr, nullptr, nullptr);
    }
    float iso = iso_in;
    if (!o.skipped && repeat) { /* marching.cpp:481-494 */
        float mx = o.corner_values[0];
        for (int v = 1; v < 8; v++)
            if (mx < o.corner_values[v]) mx = o.corner_values[v];
        float a = (mx - iso_in) / rstep;
        a = floorf(a);
        iso = iso_in + rstep * a;
    }
    o.surf_constant = iso;
    if (!o.skipped) {
        int code = 0;
        for (int v = 0; v < 8; v++) code |= (o.corner_values[v] > iso ? 1 : 0) << v;
        o.cube_code = code;
        o.table_idx = code;
        if (code != 0 && code != 255) {
            const int face = (int)gtb->face[code];
            if (face >= 0) { /* marching.cpp:521-549 */
                float mx = 0.f, my = 0.f, mz = 0.f;
                for (int q = 0; q < 4; q++) {
                    const int cv = mcb_face_corner(face, q);
                    mx += cc[3 * cv]; my += cc[3 * cv + 1]; mz += cc[3 * cv + 2];
                }
                mx /= 4.0f; my /= 4.0f; mz /= 4.0f;
                const float mid = mcb_interp_scalar(progs[0].code, progs[0].n, progs[0].k, sx * mx, sy * my, sz * mz, nullptr, nullptr, nullptr);
                if (mid > iso) o.table_idx = 255 - code;
            }
            int mapper[12];
            for (int e = 0; e < 12; e++) {
                mapper[e] = 12;
                const int a = mcb_edge_a(e), b = mcb_edge_b(e);
                if ((((code >> a) ^ (code >> b)) & 1) == 0) continue;
                const float t = (iso - o.corner_values[a]) / (o.corner_values[b] - o.corner_values[a]);
                mapper[e] = o.n_edges;
                o.edge_list[o.n_edges] = e;
                o.intersect_coord[3 * o.n_edges] = mcb_interp_ref(cc[3 * a], cc[3 * b], t);
                o.intersect_coord[3 * o.n_edges + 1] = mcb_interp_ref(cc[3 * a + 1], cc[3 * b + 1], t);
                o.intersect_coord[3 * o.n_edges + 2] = mcb_interp_ref(cc[3 * a + 2], cc[3 * b + 2], t);
                o.n_edges++;
            }
            const uint64_t row = gtb->tri[o.table_idx];
            for (int f = 0; f < 15; f++) {
                const int e = (int)((row >> (4 * f)) & 0xF);
                if (e == 0xF) break;
                o.tri_vlist[o.n_tri_idx++] = mapper[e];
            }
        }
    }
    *out = o;
}

/* ---------------------------------------------------------------------------------------------------------------
 * Slab balancing (SURVEY §8e "optionally by measured active count"): triangles per cube layer of the last
 * polygonisation.  The records are in loop order, so a warp's 32 cubes nearly always share their layer: one atomic
 * per warp then.
 * ------------------------------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(256)
layer_hist_kernel(const unsigned long long* __restrict__ rec, const uint32_t* __restrict__ trioff, const Counters* __restrict__ ctr,
                  unsigned long long cap_active, uint32_t* __restrict__ hist /* [M], indexed by the global layer */) {
    unsigned long long A = ctr->active;
    const unsigned long long T = ctr->triangles;
    if (A > cap_active) A = cap_active;
    const int lane = threadIdx.x & 31;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x, a0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (unsigned long long base = a0 - lane; base < A; base += stride) { /* whole warps stay in the loop together */
        const unsigned long long a = base + lane;
        int layer = -1;
        uint32_t cnt = 0;
        if (a < A) {
            layer = (int)((rec[a] >> 24) & 0xFFFu);
            cnt = (a + 1 < A ? trioff[a + 1] : (uint32_t)T) - trioff[a];
        }
        const int first = __shfl_sync(0xffffffffu, layer, 0);
        if (__all_sync(0xffffffffu, layer == first || layer < 0)) {
#pragma unroll
            for (int d = 16; d; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
            if (lane == 0 && first >= 0) atomicAdd(hist + first, cnt);
        } else if (layer >= 0) atomicAdd(hist + layer, cnt);
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * Parity hooks (not on the hot path).
 * ------------------------------------------------------------------------------------------------------------- */
__global__ void dense_codes_kernel(const Grid g, const uint32_t* __restrict__ S, const uint32_t* __restrict__ V,
                                   uint8_t* __restrict__ code_out, uint8_t* __restrict__ tidx_out, long long ncubes,
                                   const uint32_t* __restrict__ Cw, uint32_t WC) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ncubes) return;
    const int i = (int)(idx % g.M);
    const long long r = idx / g.M;
    const int j = (int)(r % g.M), kz = (int)(r / g.M);
    int code = 0;
    bool ok = true;
#pragma unroll
    for (int v = 0; v < 8; v++) {
        const int o = mcb_corner_ofs(v);
        const int x = i + 1 + (o & 1), y = j + 1 + ((o >> 1) & 1), z = kz + 1 + ((o >> 2) & 1);
        const size_t widx = ((size_t)z * g.NV + y) * g.WP + (x >> 5);
        if (Cw != nullptr) code |= (int)((Cw[(((size_t)kz * g.M + j) * WC + (i >> 5)) * 8 + v] >> (i & 31)) & 1u) << v;
        else code |= (int)((S[widx] >> (x & 31)) & 1u) << v;
        if (V) ok = ok && ((V[widx] >> (x & 31)) & 1u);
    }
    if (!ok) code = 0;
    if (code_out) code_out[idx] = (uint8_t)code;
    if (tidx_out) tidx_out[idx] = (uint8_t)code; /* redirects are patched in by scatter_tidx_kernel */
}

__global__ void scatter_tidx_kernel(const Grid g, const unsigned long long* __restrict__ rec, unsigned long long A,
                                    uint8_t* __restrict__ tidx_out) {
    const unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= A) return;
    const unsigned long long r = rec[q];
    const long long i = (long long)(r & 0xFFF), j = (long long)((r >> 12) & 0xFFF), k = (long long)((r >> 24) & 0xFFF);
    tidx_out[((k - g.kb) * g.M + j) * g.M + i] = (uint8_t)((r >> 44) & 0xFF);
}

__global__ void eval_points_kernel(const __grid_constant__ mcb_program prog, const float* __restrict__ xyz,
                                   float* __restrict__ out, long long n, float sx, float sy, float sz) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    out[q] = mcb_interp_scalar(prog.code, prog.n, prog.k, sx * xyz[3 * q], sy * xyz[3 * q + 1], sz * xyz[3 * q + 2],
                               nullptr, nullptr, nullptr);
}

__global__ void eval_gradients_kernel(const __grid_constant__ mcb_program prog, const float* __restrict__ xyz,
                                      float* __restrict__ grad, long long n, float sx, float sy, float sz) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    float gr[3];
    mcb_interp_grad_scalar(prog.code, prog.n, prog.k, sx * xyz[3 * q], sy * xyz[3 * q + 1], sz * xyz[3 * q + 2], sx, sy, sz, gr);
    grad[3 * q] = gr[0]; grad[3 * q + 1] = gr[1]; grad[3 * q + 2] = gr[2];
}

/* Analytic normals (mcb_set_normals 3): the normalised gradient of the surface's point program at every output vertex,
 * after the emitter (SOUP: float4 (x,y,z,1) -> (nx,ny,nz,0), 3 per triangle) or the weld (float3 -> float3).  A normal is
 * a function of the position bits, the equation and the scale only.  The element count comes from the device counters,
 * capped by the buffer, so the pass needs no host synchronisation and runs again in a repeated pass. */
template <bool SOUP>
__global__ void __launch_bounds__(256)
grad_normals_kernel(const __grid_constant__ mcb_program prog, float sx, float sy, float sz, const Counters* __restrict__ ctr,
                    unsigned long long cap, const float* __restrict__ pos, float* __restrict__ nrm) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    unsigned long long n = SOUP ? ctr->triangles : ctr->vertices;
    if (n > cap) n = cap;
    if (SOUP) n *= 3;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
        float p[3], gr[3], o[3];
        if (SOUP) {
            const float4 v = reinterpret_cast<const float4*>(pos)[q];
            p[0] = v.x; p[1] = v.y; p[2] = v.z;
        } else {
            p[0] = pos[3 * q]; p[1] = pos[3 * q + 1]; p[2] = pos[3 * q + 2];
        }
        mcb_interp_grad_scalar(prog.code, prog.n, prog.k, sx * p[0], sy * p[1], sz * p[2], sx, sy, sz, gr);
        mcb_grad_normalise(gr, o);
        if (SOUP) reinterpret_cast<float4*>(nrm)[q] = make_float4(o[0], o[1], o[2], 0.f);
        else { nrm[3 * q] = o[0]; nrm[3 * q + 1] = o[1]; nrm[3 * q + 2] = o[2]; }
    }
}

/* Refined vertices (mcb_set_refine_vertices): every output vertex strictly inside a grid edge moves, in place, to the root
 * of the point program along that edge (mcb_refine_vertex, mcb_refine.h), after the emitter (SOUP: float4 (x,y,z,1), 3
 * per triangle, w kept) or the weld (float3).  cs = the coordinate table c[0..M].  The element count comes from the device
 * counters, capped by the buffer, so the pass needs no host synchronisation and runs again in a repeated pass. */
template <bool SOUP>
__global__ void __launch_bounds__(256)
refine_vertices_kernel(const __grid_constant__ mcb_program prog, float sx, float sy, float sz, float iso, const float* __restrict__ cs,
                       int M, const Counters* __restrict__ ctr, unsigned long long cap, float* __restrict__ pos) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    unsigned long long n = SOUP ? ctr->triangles : ctr->vertices;
    if (n > cap) n = cap;
    if (SOUP) n *= 3;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
        float p[3];
        if (SOUP) {
            const float4 v = reinterpret_cast<const float4*>(pos)[q];
            p[0] = v.x; p[1] = v.y; p[2] = v.z;
        } else {
            p[0] = pos[3 * q]; p[1] = pos[3 * q + 1]; p[2] = pos[3 * q + 2];
        }
        if (mcb_refine_vertex(prog.code, prog.n, prog.k, cs, M, iso, sx, sy, sz, p, nullptr) <= 0) continue;
        if (SOUP) reinterpret_cast<float4*>(pos)[q] = make_float4(p[0], p[1], p[2], 1.f);
        else { pos[3 * q] = p[0]; pos[3 * q + 1] = p[1]; pos[3 * q + 2] = p[2]; }
    }
}

/* ---------------------------------------------------------------------------------------------------------------
 * K8  dual contouring (MCB_MESH_DC, mcb_qef.h, DESIGN.md §14), after compact in place of the soup and the weld.  One
 *     vertex per active cube, numbered like the record list; a cube is found through the weld's per-word look-up
 *     (compact_kernel's item words: first record | active mask).  A cube that contains a crossing edge is active exactly
 *     when it lies in the grid and passes the constraints (weld_cube_ok), so no sign has to be read outside the cube
 *     that asks.
 *       dc_edges   per active cube: Hermite data (refined coordinate, unit normal; one float4) of every crossing edge it is
 *                  the first cube in loop order to contain, into slot 12 * record + local edge
 *       dc_vertex  per active cube: its crossing edges' Hermite data from their computing cubes, the QEF vertex, and two
 *                  triangles for each of its three quad edges (through its corner (i+1, j+1, k+1)) whose cubes are active
 *       scan       exclusive scan of those counts (scan_block_sums / scan_sums / scan_apply)
 *       dc_emit    the triangles, split along the quad's shorter diagonal
 *     Sizes come from the device counters (dc_n = active capped by the records), so nothing waits for the host; a pass
 *     whose buffers were too small writes what fits and is repeated.
 * ------------------------------------------------------------------------------------------------------------- */
__device__ __forceinline__ void dc_corners(const Grid& g, const float* __restrict__ F, int i, int j, int k, float f[8]) {
    const size_t rowp = (size_t)g.P, planep = (size_t)g.NV * g.P;
    const float* f0 = F + (size_t)(k - g.kb + 1) * planep + (size_t)(j + 1) * rowp + (i + 1);
#pragma unroll
    for (int v = 0; v < 8; v++) {
        const int o = mcb_corner_ofs(v);
        f[v] = __ldg(f0 + (size_t)(o >> 2) * planep + (size_t)((o >> 1) & 1) * rowp + (o & 1));
    }
}
/* field value at the lower end of edge e (the end with the smaller coordinate) */
__device__ __forceinline__ float dc_lower_value(const float f[8], int e) {
    const int a = mcb_edge_a(e), b = mcb_edge_b(e);
    return mcb_corner_ofs(a) < mcb_corner_ofs(b) ? f[a] : f[b];
}
/* the first cube in loop order that contains the grid edge and is active */
__device__ __forceinline__ CubeEdge dc_computing_cube(const WeldView& W, int i, int j, int k, int e, const GridEdge& E) {
    CubeEdge o{i, j, k, e};
    weld_owner_fast(W, E, o);
    return o;
}

__global__ void __launch_bounds__(256)
dc_edges_kernel(const __grid_constant__ mcb_program prog, const WeldView W, const unsigned long long* __restrict__ rec,
                Counters* __restrict__ ctr, unsigned long long cap_active, float4* __restrict__ slots) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const Grid& g = W.g;
    const unsigned long long A = ctr->active, n = A < cap_active ? A : cap_active;
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctr->vertices = A; ctr->triangles = 0ull; ctr->dc_n = n; }
    const float* c = W.cs + 1; /* c[v] = cs[v+1] */
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
        const unsigned long long r = rec[q];
        const int i = (int)(r & 0xFFF), j = (int)((r >> 12) & 0xFFF), k = (int)((r >> 24) & 0xFFF);
        float f[8];
        dc_corners(g, W.F, i, j, k, f);
        for (int e = 0; e < 12; e++) {
            if ((f[mcb_edge_a(e)] > g.iso) == (f[mcb_edge_b(e)] > g.iso)) continue;
            const GridEdge E = grid_edge_of(i, j, k, e);
            const CubeEdge o = dc_computing_cube(W, i, j, k, e, E);
            if (o.i != i || o.j != j || o.k != k) continue;
            const float lo[3] = {c[E.vx], c[E.vy], c[E.vz]};
            const int ia = E.axis == 0 ? E.vx : E.axis == 1 ? E.vy : E.vz;
            const bool a_low = mcb_corner_ofs(mcb_edge_a(e)) < mcb_corner_ofs(mcb_edge_b(e));
            const float flo = a_low ? f[mcb_edge_a(e)] : f[mcb_edge_b(e)], fhi = a_low ? f[mcb_edge_b(e)] : f[mcb_edge_a(e)];
            float h[4];
            mcb_dc_edge(prog.code, prog.n, prog.k, c, g.M, g.iso, g.sx, g.sy, g.sz, lo, E.axis, ia, flo, fhi, h);
            slots[12 * q + e] = make_float4(h[0], h[1], h[2], h[3]);
        }
    }
}

__global__ void __launch_bounds__(256)
dc_vertex_kernel(const WeldView W, const WeldBuffers B, const Counters* __restrict__ ctr, unsigned long long cap_verts,
                 const float4* __restrict__ slots, float* __restrict__ vlist, uint32_t* __restrict__ tcount) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const Grid& g = W.g;
    const unsigned long long n = ctr->dc_n;
    const float* c = W.cs + 1;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
        const unsigned long long r = B.rec[q];
        const int i = (int)(r & 0xFFF), j = (int)((r >> 12) & 0xFFF), k = (int)((r >> 24) & 0xFFF);
        float f[8];
        dc_corners(g, W.F, i, j, k, f);
        float pts[12][3], nrm[12][3];
        int m = 0;
        for (int e = 0; e < 12; e++) {
            if ((f[mcb_edge_a(e)] > g.iso) == (f[mcb_edge_b(e)] > g.iso)) continue;
            const GridEdge E = grid_edge_of(i, j, k, e);
            const CubeEdge o = dc_computing_cube(W, i, j, k, e, E);
            const uint32_t idx = weld_find_cube(B, g, o.i, o.j, o.k);
            const float4 h = idx < n ? slots[12ull * idx + o.e] : make_float4(0.f, 0.f, 0.f, 0.f); /* else: truncated records, repeated */
            pts[m][0] = c[E.vx]; pts[m][1] = c[E.vy]; pts[m][2] = c[E.vz];
            pts[m][E.axis] = h.x;
            nrm[m][0] = h.y; nrm[m][1] = h.z; nrm[m][2] = h.w;
            m++;
        }
        const float lo[3] = {c[i], c[j], c[k]}, hi[3] = {c[i + 1], c[j + 1], c[k + 1]};
        float x[3];
        mcb_qef_vertex(pts, nrm, m, lo, hi, x, nullptr);
        if (q < cap_verts) { vlist[3 * q] = x[0]; vlist[3 * q + 1] = x[1]; vlist[3 * q + 2] = x[2]; }
        uint32_t t = 0;
        for (int axis = 0; axis < 3; axis++) {
            const int e = mcb_dc_quad_edge(axis);
            if ((f[mcb_edge_a(e)] > g.iso) == (f[mcb_edge_b(e)] > g.iso)) continue;
            int cb[4][3];
            mcb_dc_quad_cubes(i, j, k, axis, false, cb);
            bool ok = true;
            for (int s = 1; s < 4; s++) ok = ok && weld_cube_ok(W, cb[s][0], cb[s][1], cb[s][2]);
            if (ok) t += 2;
        }
        tcount[q] = t;
    }
}

__global__ void __launch_bounds__(256)
dc_emit_kernel(const WeldView W, const WeldBuffers B, Counters* __restrict__ ctr, unsigned long long cap_verts, unsigned long long cap_tris,
               const float* __restrict__ vlist, const uint32_t* __restrict__ tcount, const uint32_t* __restrict__ toff,
               uint32_t* __restrict__ tlist) {
    MCB_GRID_WAIT();
    MCB_GRID_DEPENDENTS();
    const Grid& g = W.g;
    const unsigned long long n = ctr->dc_n;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
        if (q == n - 1) ctr->triangles = (unsigned long long)toff[q] + tcount[q];
        if (tcount[q] == 0) continue;
        const unsigned long long r = B.rec[q];
        const int i = (int)(r & 0xFFF), j = (int)((r >> 12) & 0xFFF), k = (int)((r >> 24) & 0xFFF);
        float f[8];
        dc_corners(g, W.F, i, j, k, f);
        unsigned long long t = toff[q];
        for (int axis = 0; axis < 3; axis++) {
            const int e = mcb_dc_quad_edge(axis);
            if ((f[mcb_edge_a(e)] > g.iso) == (f[mcb_edge_b(e)] > g.iso)) continue;
            int cb[4][3];
            mcb_dc_quad_cubes(i, j, k, axis, dc_lower_value(f, e) > g.iso, cb);
            bool ok = true;
            for (int s = 0; s < 4; s++) ok = ok && weld_cube_ok(W, cb[s][0], cb[s][1], cb[s][2]);
            if (!ok) continue;
            uint32_t w[4];
            float p[4][3];
            for (int s = 0; s < 4; s++) {
                w[s] = weld_find_cube(B, g, cb[s][0], cb[s][1], cb[s][2]);
                const unsigned long long v = w[s] < cap_verts ? w[s] : 0ull; /* else: the pass is repeated with room */
                p[s][0] = vlist[3 * v]; p[s][1] = vlist[3 * v + 1]; p[s][2] = vlist[3 * v + 2];
            }
            const bool d02 = mcb_dc_split02(p[0], p[1], p[2], p[3]);
            const uint32_t tri[6] = {w[0], w[1], d02 ? w[2] : w[3], d02 ? w[0] : w[1], w[2], w[3]};
            for (int h = 0; h < 2; h++, t++)
                if (t < cap_tris) { tlist[3 * t] = tri[3 * h]; tlist[3 * t + 1] = tri[3 * h + 1]; tlist[3 * t + 2] = tri[3 * h + 2]; }
        }
    }
}

} /* namespace mcbk */
