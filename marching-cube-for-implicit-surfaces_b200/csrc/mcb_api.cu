/* libmcb200.so — C ABI (include/mcb.h) over the sm_100a kernels in mcb_kernels.cuh.
 *
 * One mcb_ctx owns the device buffers of one z-slab on one GPU and a CUDA stream; every entry point makes the
 * context's device current, enqueues on that stream and reports failures as negative status codes.  No entry point
 * computes field values, cases or triangles on the host.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <future>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/mcb.h"
#include "mcb_kernels.cuh"
#include "mcb_jit.h"
#include "mcb_lower.h"

using namespace mcbk;

namespace {

struct EqSlot {
    bool valid = false;
    mcb::Compiled c;
    mcb_program point; /* full expression at an arbitrary point */
    mcb_program grid;  /* full expression on the grid, hoisted subtrees as table operands, fused accumulator form */
    uint32_t* d_slot_code = nullptr;
    SlotDesc* d_slots = nullptr;
    float* d_kpool = nullptr;
    int n_const = 0, n_axis = 0, max_per_axis = 1;
};

struct Constraint {
    int op = 0;
    float rhs = 0.f;
    bool in_use = false;
};

} /* namespace */

struct mcb_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::string err;

    EqSlot eq[4];
    int grammar = MCB_GRAMMAR_REFERENCE; /* mcb_set_grammar: how later mcb_set_equation calls parse */
    Constraint cons[3];
    float step = 0.25f;
    int M = 0;
    std::vector<float> axis; /* c[0..M] of the reference loop */
    int kb = 0, ke = 0;
    float iso = 0.f;
    float scale[3] = {1.f, 1.f, 1.f};
    int normals = 1;

    Grid g{};
    bool grid_dirty = true;
    float* d_cs = nullptr;
    size_t rinv_ofs = 0; /* d_cs + rinv_ofs: 1 / (c[v+1] - c[v-1]) per stored coordinate */
    float* d_F = nullptr;
    uint32_t* d_S = nullptr;
    uint32_t* d_V = nullptr;
    float* d_tables = nullptr;
    size_t cap_F = 0, cap_S = 0, cap_V = 0, cap_tables = 0, cap_cs = 0;
    ClsTables* d_cls = nullptr;
    Counters* d_ctr = nullptr;
    Counters* h_ctr = nullptr; /* pinned */
    unsigned long long* d_ent = nullptr;    /* classify -> compact scratch: one entry per active item of every tile */
    uint32_t* d_tile_u32 = nullptr;         /* [5][cap_tiles]: entries, active cubes, triangles, and the two exclusive prefixes */
    unsigned long long* d_amb = nullptr;    /* [cap_amb][2] ambiguous cubes awaiting the face-centre test */
    uint32_t cap_amb = 0;
    size_t cap_tile_entries = 0;
    size_t cap_tiles = 0;
    unsigned long long* d_rec = nullptr;
    uint32_t* d_trioff = nullptr;
    unsigned long long cap_active = 0;
    float4* d_pos = nullptr;
    float4* d_nrm = nullptr;
    unsigned long long cap_tris = 0;
    bool nrm_allocated = false;
    int mesh_mode = MCB_MESH_SOUP;
    /* welded, indexed mesh (Poly_Data layout) */
    float* d_vlist = nullptr;      /* [3 * cap_verts] */
    float* d_vnrm = nullptr;       /* [3 * cap_verts] */
    uint32_t* d_tlist = nullptr;   /* [3 * cap_itris] */
    unsigned long long cap_verts = 0, cap_itris = 0;
    bool vnrm_allocated = false;
    /* host output registered with mcb_set_host_output: the indexed mesh is streamed out while it is produced */
    float* h_out_v = nullptr;
    uint32_t* h_out_t = nullptr;
    float* h_out_n = nullptr;
    unsigned long long h_cap_v = 0, h_cap_t = 0;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t seg_ev[9] = {};
    cudaEvent_t fork_ev[2] = {};    /* evaluation stage: decided_signs runs on copy_stream next to the block evaluation */
    unsigned long long* d_bounds = nullptr;
    unsigned long long* h_bounds = nullptr; /* pinned */
    bool streamed = false;                  /* the last polygonise delivered the mesh to the registered buffers */
    /* seed mode (mcb_set_seed) */
    bool seed_on = false;
    /* run-time specialised evaluator (mcb_set_jit): one cubin per distinct generated source, i.e. per equation */
    int jit = MCB_JIT_AUTO;
    std::string jit_note;          /* why MCB_JIT_AUTO stayed with the interpreter, if it did */
    struct JitKernel { cudaLibrary_t lib = nullptr; cudaKernel_t kernel = nullptr, signs = nullptr, fill = nullptr; };
    const JitKernel* jit_cur = nullptr; /* the module the last evaluation used */
    std::map<std::string, JitKernel> jit_cache;
    /* MCB_JIT_AUTO compiles in the background: the calls made meanwhile interpret (same results), the first call after
     * the compile has finished loads the module.  Keyed by the generated source, like the cache. */
    struct JitBuilt { std::string err; std::vector<char> cubin; float ms = 0.f; };
    std::map<std::string, std::future<JitBuilt>> jit_pending;
    std::map<std::string, std::string> jit_failed; /* source -> why its compile failed: not tried again */
    bool jit_sync = false;         /* $MCB_JIT_SYNC=1: MCB_JIT_AUTO compiles inside the call, like MCB_JIT_ON */
    bool jit_used = false;         /* the last polygonisation ran the specialised kernel */
    float ms_compile = 0.f;        /* host time of the NVRTC compile it had to do (0 when cached) */
    bool repeat_on = false;        /* repeating-surface mode (mcb_set_repeat) */
    float repeat_step = 0.f;
    uint32_t* d_cw = nullptr;      /* [items][8] corner words of every 32-cube item, repeating-surface mode only */
    size_t cap_cw = 0;
    float seed[3] = {0.f, 0.f, 0.f};
    /* z-slabs over several GPUs (mcb_comm_*): the NCCL communicator and the device-side placement of this slab */
    void* nccl_comm = nullptr;
    int comm_rank = 0, comm_nranks = 1;
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t comm_ready = nullptr, comm_done = nullptr;
    unsigned long long* d_comm = nullptr;   /* [2 + nranks]: two staging slots for this slab's count, then the gathered counts */
    unsigned long long* h_comm = nullptr;   /* pinned copy of the gathered counts */
    int comm_flip = 0;
    bool comm_pending = false;
    std::vector<double> layer_cost;         /* [M] cost of every cube layer as the last (re)balance saw it */
    std::vector<int> comm_cuts;             /* [nranks + 1] the slabs of the last (re)balance */
    bool comm_auto = false;                 /* mcb_comm_set_auto: mcb_polygonise enqueues the exchange itself, as soon as the count is final */
    uint32_t* d_layer_hist = nullptr;       /* [cap_layer_hist] triangles per global cube layer */
    size_t cap_layer_hist = 0;
    uint8_t* d_mark = nullptr;
    uint32_t* d_changed = nullptr;
    uint32_t* d_seed_u32 = nullptr; /* keep | ktri | pa | pt, cap_seed entries each, then the block sums */
    unsigned long long* d_rec2 = nullptr;
    uint32_t* d_trioff2 = nullptr;
    unsigned long long cap_seed = 0;
    /* normal.h normals (mcb_set_normals 2): face normals, vertex -> corner CSR */
    float* d_fn = nullptr;
    uint32_t* d_nh_count = nullptr;
    uint32_t* d_nh_start = nullptr;
    uint32_t* d_nh_cursor = nullptr;
    uint32_t* d_nh_sums = nullptr;
    uint32_t* d_nh_adj = nullptr;
    unsigned long long cap_nh_verts = 0, cap_nh_tris = 0;
    unsigned long long* d_item = nullptr;  /* per 32-cube word: first record | active mask << 32 (compact -> weld) */
    size_t cap_items = 0;
    unsigned long long* d_vinfo = nullptr; /* per active cube: first new vertex | new-edge mask | on-vertex mask */
    uint32_t* d_chunk_new = nullptr;
    unsigned long long cap_weld = 0;       /* cubes the two arrays above are sized for */
    cudaEvent_t ev[9] = {};
    /* sparse-field mode (mcb_set_field_mode): the field is only written in 32 x 4 x 4 vertex blocks around the surface */
    int field_mode = MCB_FIELD_DENSE;
    bool field_is_sparse = false;  /* what the last polygonisation left in d_F: only the blocks around the surface */
    bool poison_field = false;     /* $MCB_POISON_FIELD: NaN-fill d_F first, so a read outside the blocks shows (tests) */
    bool decide_blocks = true;     /* $MCB_NO_INTERVAL=1: treat every block as undecided, i.e. evaluate them all (tests) */
    bool stage_timing = true;      /* mcb_set_stage_timing: CUDA events around the stages (mcb_counts::ms_*) */
    uint32_t index_base = 0;        /* mcb_set_index_base: added to every index mcb_get_indexed_mesh delivers */
    uint32_t index_base_applied = 0; /* what d_tlist currently carries (0 after every polygonisation) */
    uint8_t* d_fflags = nullptr;   /* [cap_fblocks] 2 = evaluated (undecided block), 1 = apron block to refill, 0 = untouched */
    uint8_t* d_bcls = nullptr;     /* [cap_fblocks] interval class of every 32 x 4 x 4 vertex block */
    uint32_t* d_flist = nullptr;   /* [cap_fblocks] apron blocks */
    uint32_t* d_elist = nullptr;   /* [cap_fblocks] undecided blocks */
    unsigned long long* d_cand = nullptr; /* [cap_cand] one bit per cube block that may hold an active cube */
    uint32_t* d_slist = nullptr;   /* [cap_scls] undecided super-blocks */
    uint8_t* d_scls = nullptr;     /* [cap_scls] interval class of every 32 x 16 x 16 super-block */
    size_t cap_scls = 0;
    BlockDims bd{};                /* block geometry of the last block-field run (mcb_get_cases completes the sign words with it) */
    mcb_ival* d_bounds_iv = nullptr; /* [3][slots][nb] table bounds per block of each axis */
    size_t cap_fblocks = 0, cap_cand = 0, cap_bounds_iv = 0;
    mcb_counts last{};
    bool have_result = false;
};

namespace {

#define MCB_CK(call)                                                                                         \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess) {                                                                             \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                   \
            return e_ == cudaErrorMemoryAllocation ? MCB_E_NOMEM : MCB_E_CUDA;                               \
        }                                                                                                    \
    } while (0)

int comm_enqueue(mcb_ctx* ctx); /* below, with the rest of the multi-GPU exchange */

int fail(mcb_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    return code;
}

template <class T>
int ensure(mcb_ctx* ctx, T** p, size_t* cap, size_t need) {
    if (*cap >= need && *p) return MCB_OK;
    if (*p) { cudaFree(*p); *p = nullptr; *cap = 0; }
    MCB_CK(cudaMalloc((void**)p, need * sizeof(T)));
    *cap = need;
    return MCB_OK;
}

/* The reference's grid loop, marching.cpp:372-377: fp32 accumulation, bound rounded from a double expression. */
std::vector<float> reference_axis(float step) {
    std::vector<float> c;
    float lower = -1.0f;
    float upper = (float)(1.0 + 0.5 * (double)step);
    for (float v = lower; v <= upper; v += step) {
        c.push_back(v);
        if (c.size() > 8192) break;
    }
    c.push_back(c.back() + step); /* far corner of the last cube: x_1 = x_0 + step (marching.cpp:458) */
    return c;
}

void fill_program(mcb_program& p, const std::vector<uint32_t>& code, const std::vector<float>& k) {
    std::memset(&p, 0, sizeof p);
    p.n = (int)code.size();
    std::copy(code.begin(), code.end(), p.code);
    std::copy(k.begin(), k.end(), p.k);
}

void free_slot(EqSlot& s) {
    if (s.d_slot_code) cudaFree(s.d_slot_code);
    if (s.d_slots) cudaFree(s.d_slots);
    if (s.d_kpool) cudaFree(s.d_kpool);
    s.d_slot_code = nullptr; s.d_slots = nullptr; s.d_kpool = nullptr;
}

int install_equation(mcb_ctx* ctx, int slot, const char* equation) {
    mcb::Compiled c;
    std::string err;
    int rc = mcb::compile(equation ? equation : "", c, &err, ctx->grammar);
    if (rc != MCB_OK) return fail(ctx, rc, err);

    EqSlot ns;
    struct Guard { /* frees the new slot's device memory on every early return */
        EqSlot* s;
        ~Guard() { if (s) free_slot(*s); }
    } guard{&ns};
    ns.c = c;
    ns.valid = true;
    std::vector<SlotDesc> descs;
    for (const mcb::Slot& s : c.slots) {
        SlotDesc d{s.code_begin, s.code_len, s.axis, s.kindex};
        descs.push_back(d);
        if (s.axis < 0) ns.n_const++; else ns.n_axis++;
    }
    ns.max_per_axis = std::max(1, std::max(c.n_axis_slots[0], std::max(c.n_axis_slots[1], c.n_axis_slots[2])));
    if (!descs.empty()) {
        MCB_CK(cudaMalloc((void**)&ns.d_slot_code, std::max<size_t>(1, c.slot_code.size()) * sizeof(uint32_t)));
        MCB_CK(cudaMalloc((void**)&ns.d_slots, descs.size() * sizeof(SlotDesc)));
        MCB_CK(cudaMemcpyAsync(ns.d_slot_code, c.slot_code.data(), c.slot_code.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        MCB_CK(cudaMemcpyAsync(ns.d_slots, descs.data(), descs.size() * sizeof(SlotDesc), cudaMemcpyHostToDevice, ctx->stream));
    }
    MCB_CK(cudaMalloc((void**)&ns.d_kpool, MCB_MAX_K * sizeof(float)));
    MCB_CK(cudaMemcpyAsync(ns.d_kpool, c.kpool.data(), c.kpool.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (ns.n_const > 0) {
        /* constant subtrees are folded ON THE DEVICE by the same interpreter that evaluates the field */
        MCB_LAUNCH((fold_constants_kernel), 1, 128, 0, ctx->stream, ns.d_slot_code, ns.d_slots, (int)descs.size(), ns.d_kpool, ns.d_kpool);
        MCB_CK(cudaGetLastError());
        MCB_CK(cudaMemcpyAsync(ns.c.kpool.data(), ns.d_kpool, ns.c.kpool.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    }
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    fill_program(ns.point, ns.c.point_code, ns.c.kpool);
    fill_program(ns.grid, ns.c.grid_fused, ns.c.kpool);
    free_slot(ctx->eq[slot]);
    ctx->eq[slot] = ns;
    guard.s = nullptr; /* the slot owns the allocations now */
    ctx->have_result = false;
    return MCB_OK;
}

/* Tiling of the classify pass: runs of whole cube rows, at most kClsItemCap items, at least ~4 tiles per SM
 * (DESIGN.md, classify). */
ClsGeom classify_geometry(const mcb_ctx* ctx, const Grid& g, unsigned* tiles) {
    ClsGeom cg;
    cg.WC = (uint32_t)((g.M + 31) / 32);
    cg.total_rows = (uint32_t)(g.ke - g.kb) * (uint32_t)g.M;
    const uint32_t cap_rows = (uint32_t)kClsItemCap / cg.WC;
    const uint32_t target = (uint32_t)ctx->sm_count * 4u;
    cg.tile_rows = std::min(cap_rows, std::max(1u, (cg.total_rows + target - 1) / target));
    cg.nstrips = std::max(1u, (uint32_t)kClsThreads / cg.WC);
    cg.strip_rows = (cg.tile_rows + cg.nstrips - 1) / cg.nstrips;
    cg.inv_wc = cg.WC == 1 ? 0u : (uint32_t)((1ull << 32) / cg.WC + ((1ull << 32) % cg.WC ? 1 : 0));
    cg.inv_m = g.M == 1 ? 0u : (uint32_t)((1ull << 32) / (unsigned)g.M + ((1ull << 32) % (unsigned)g.M ? 1 : 0));
    *tiles = (cg.total_rows + cg.tile_rows - 1) / cg.tile_rows;
    return cg;
}

int setup_grid(mcb_ctx* ctx) {
    if (!ctx->grid_dirty) return MCB_OK;
    Grid& g = ctx->g;
    g.M = ctx->M;
    g.NV = ctx->M + 3;
    g.P = (g.NV + 31) / 32 * 32;
    g.WP = (g.P / 32 + 3) / 4 * 4; /* whole 128-column eval tiles: a tile row's 4 sign words are one aligned 16-byte store */
    g.kb = ctx->kb;
    g.ke = ctx->ke;
    g.NZ = (g.ke - g.kb) + 3;
    /* coordinates with the apron: cs[v+1] = c[v]; c[-1] = c[0]-step, c[M+1] = c[M]+step (fp32, like the loop) */
    const size_t ncs = (size_t)g.P + 64;
    std::vector<float> cs(2 * ncs, 0.f); /* coordinates, then 1 / (c[v+1] - c[v-1]): the central-difference denominators */
    cs[0] = ctx->axis[0] - ctx->step;
    for (int v = 0; v <= g.M; v++) cs[v + 1] = ctx->axis[v];
    cs[g.M + 2] = ctx->axis[g.M] + ctx->step;
    for (size_t q = g.NV; q < ncs; q++) cs[q] = cs[g.NV - 1];
    for (int v = 1; v + 1 < g.NV; v++) cs[ncs + v] = 1.0f / (cs[v + 1] - cs[v - 1]);
    ctx->rinv_ofs = ncs;
    int rc;
    if ((rc = ensure(ctx, &ctx->d_cs, &ctx->cap_cs, cs.size())) != MCB_OK) return rc;
    MCB_CK(cudaMemcpyAsync(ctx->d_cs, cs.data(), cs.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream)); /* cs is a stack vector */
    const size_t nF = (size_t)g.NZ * g.NV * g.P + 64;
    const size_t nS = (size_t)g.NZ * g.NV * g.WP + 64;
    if ((rc = ensure(ctx, &ctx->d_F, &ctx->cap_F, nF)) != MCB_OK) return rc;
    if ((rc = ensure(ctx, &ctx->d_S, &ctx->cap_S, nS)) != MCB_OK) return rc;
    unsigned tiles_now = 0;
    const ClsGeom cg0 = classify_geometry(ctx, g, &tiles_now);
    const size_t tiles = (size_t)tiles_now + 1;
    if (tiles > ctx->cap_tiles) {
        if (ctx->d_tile_u32) cudaFree(ctx->d_tile_u32);
        ctx->d_tile_u32 = nullptr;
        ctx->cap_tiles = 0;
        MCB_CK(cudaMalloc((void**)&ctx->d_tile_u32, 5 * tiles * 4));
        ctx->cap_tiles = tiles;
    }
    const size_t entries = tiles * (size_t)cg0.tile_rows * cg0.WC; /* worst case: every item active */
    if (entries > ctx->cap_tile_entries) {
        if (ctx->d_ent) cudaFree(ctx->d_ent);
        ctx->d_ent = nullptr;
        ctx->cap_tile_entries = 0;
        MCB_CK(cudaMalloc((void**)&ctx->d_ent, entries * 8));
        ctx->cap_tile_entries = entries;
    }
    if (!ctx->d_amb) {
        ctx->cap_amb = 1u << 18;
        MCB_CK(cudaMalloc((void**)&ctx->d_amb, (size_t)ctx->cap_amb * 16));
    }
    ctx->grid_dirty = false;
    return MCB_OK;
}

int ensure_records(mcb_ctx* ctx, unsigned long long need) {
    if (ctx->cap_active >= need) return MCB_OK;
    if (ctx->d_rec) cudaFree(ctx->d_rec);
    if (ctx->d_trioff) cudaFree(ctx->d_trioff);
    ctx->d_rec = nullptr; ctx->d_trioff = nullptr; ctx->cap_active = 0;
    MCB_CK(cudaMalloc((void**)&ctx->d_rec, need * 8));
    MCB_CK(cudaMalloc((void**)&ctx->d_trioff, need * 4));
    ctx->cap_active = need;
    return MCB_OK;
}

int ensure_soup(mcb_ctx* ctx, unsigned long long need, bool normals) {
    if (ctx->cap_tris >= need && (!normals || ctx->nrm_allocated)) return MCB_OK;
    need = std::max(need, ctx->cap_tris);
    if (ctx->d_pos) cudaFree(ctx->d_pos);
    if (ctx->d_nrm) cudaFree(ctx->d_nrm);
    ctx->d_pos = nullptr; ctx->d_nrm = nullptr; ctx->cap_tris = 0; ctx->nrm_allocated = false;
    MCB_CK(cudaMalloc((void**)&ctx->d_pos, need * 3 * sizeof(float4)));
    if (normals) {
        MCB_CK(cudaMalloc((void**)&ctx->d_nrm, need * 3 * sizeof(float4)));
        ctx->nrm_allocated = true;
    }
    ctx->cap_tris = need;
    return MCB_OK;
}

int ensure_weld_scratch(mcb_ctx* ctx, const Grid& g) {
    const size_t items = (size_t)(g.ke - g.kb) * g.M * ((g.M + 31) / 32);
    int rc;
    if ((rc = ensure(ctx, &ctx->d_item, &ctx->cap_items, items)) != MCB_OK) return rc;
    if (ctx->cap_weld >= ctx->cap_active && ctx->d_vinfo) return MCB_OK;
    if (ctx->d_vinfo) cudaFree(ctx->d_vinfo);
    if (ctx->d_chunk_new) cudaFree(ctx->d_chunk_new);
    ctx->d_vinfo = nullptr; ctx->d_chunk_new = nullptr; ctx->cap_weld = 0;
    MCB_CK(cudaMalloc((void**)&ctx->d_vinfo, ctx->cap_active * 8));
    MCB_CK(cudaMalloc((void**)&ctx->d_chunk_new, (ctx->cap_active / kWeldCubes + 2) * 4));
    ctx->cap_weld = ctx->cap_active;
    return MCB_OK;
}

int ensure_seed_scratch(mcb_ctx* ctx) {
    if (ctx->cap_seed >= ctx->cap_active && ctx->d_mark) return MCB_OK;
    cudaFree(ctx->d_mark); cudaFree(ctx->d_seed_u32); cudaFree(ctx->d_rec2); cudaFree(ctx->d_trioff2);
    ctx->d_mark = nullptr; ctx->d_seed_u32 = nullptr; ctx->d_rec2 = nullptr; ctx->d_trioff2 = nullptr; ctx->cap_seed = 0;
    const unsigned long long n = ctx->cap_active;
    MCB_CK(cudaMalloc((void**)&ctx->d_mark, n));
    MCB_CK(cudaMalloc((void**)&ctx->d_seed_u32, (4 * n + n / kScanBlock + 2) * 4));
    MCB_CK(cudaMalloc((void**)&ctx->d_rec2, n * 8));
    MCB_CK(cudaMalloc((void**)&ctx->d_trioff2, n * 4));
    if (!ctx->d_changed) MCB_CK(cudaMalloc((void**)&ctx->d_changed, 4));
    ctx->cap_seed = n;
    return MCB_OK;
}

/* Marching::get_starting_seed_grid (marching.cpp:104-113), as cube indices: floor(((seed/scale) - (-1)) / step), fp32 */
void seed_cube(const mcb_ctx* ctx, int out[3]) {
    for (int a = 0; a < 3; a++) {
        const float d = ((ctx->seed[a] / ctx->scale[a] - (-1.0f)) / ctx->step);
        out[a] = (int)std::floor(d);
    }
}

int ensure_normal_h_scratch(mcb_ctx* ctx) {
    if (ctx->cap_nh_verts < ctx->cap_verts || !ctx->d_nh_count) {
        cudaFree(ctx->d_nh_count); cudaFree(ctx->d_nh_start); cudaFree(ctx->d_nh_cursor); cudaFree(ctx->d_nh_sums);
        ctx->d_nh_count = ctx->d_nh_start = ctx->d_nh_cursor = ctx->d_nh_sums = nullptr; ctx->cap_nh_verts = 0;
        MCB_CK(cudaMalloc((void**)&ctx->d_nh_count, ctx->cap_verts * 4));
        MCB_CK(cudaMalloc((void**)&ctx->d_nh_start, ctx->cap_verts * 4));
        MCB_CK(cudaMalloc((void**)&ctx->d_nh_cursor, ctx->cap_verts * 4));
        MCB_CK(cudaMalloc((void**)&ctx->d_nh_sums, (ctx->cap_verts / kScanBlock + 2) * 4));
        ctx->cap_nh_verts = ctx->cap_verts;
    }
    if (ctx->cap_nh_tris < ctx->cap_itris || !ctx->d_fn) {
        cudaFree(ctx->d_fn); cudaFree(ctx->d_nh_adj);
        ctx->d_fn = nullptr; ctx->d_nh_adj = nullptr; ctx->cap_nh_tris = 0;
        MCB_CK(cudaMalloc((void**)&ctx->d_fn, ctx->cap_itris * 3 * sizeof(float)));
        MCB_CK(cudaMalloc((void**)&ctx->d_nh_adj, ctx->cap_itris * 3 * sizeof(uint32_t)));
        ctx->cap_nh_tris = ctx->cap_itris;
    }
    return MCB_OK;
}

int ensure_indexed(mcb_ctx* ctx, unsigned long long verts, unsigned long long tris, bool normals) {
    if (ctx->cap_verts < verts || !ctx->d_vlist || (normals && !ctx->vnrm_allocated)) {
        verts = std::max(verts, ctx->cap_verts);
        if (ctx->d_vlist) cudaFree(ctx->d_vlist);
        if (ctx->d_vnrm) cudaFree(ctx->d_vnrm);
        ctx->d_vlist = nullptr; ctx->d_vnrm = nullptr; ctx->cap_verts = 0; ctx->vnrm_allocated = false;
        MCB_CK(cudaMalloc((void**)&ctx->d_vlist, verts * 3 * sizeof(float)));
        if (normals) {
            MCB_CK(cudaMalloc((void**)&ctx->d_vnrm, verts * 3 * sizeof(float)));
            ctx->vnrm_allocated = true;
        }
        ctx->cap_verts = verts;
    }
    if (ctx->cap_itris < tris || !ctx->d_tlist) {
        if (ctx->d_tlist) cudaFree(ctx->d_tlist);
        ctx->d_tlist = nullptr; ctx->cap_itris = 0;
        MCB_CK(cudaMalloc((void**)&ctx->d_tlist, tris * 3 * sizeof(uint32_t)));
        ctx->cap_itris = tris;
    }
    return MCB_OK;
}

int enter(mcb_ctx* ctx) {
    if (!ctx) return MCB_E_ARG;
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return fail(ctx, MCB_E_NODEVICE, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return MCB_OK;
}

int copy_text(const std::string& s, char* out, size_t cap) {
    if (!out || cap < s.size() + 1) return MCB_E_CAPACITY;
    std::memcpy(out, s.c_str(), s.size() + 1);
    return MCB_OK;
}

} /* namespace */

extern "C" {

int mcb_abi_version(void) { return MCB_ABI_VERSION; }

const char* mcb_build_stamp(void) {
    return
#include "mcb_build_stamp.inc" /* sha256 over the sources this library was built from, written by build.py */
        ;
}

int mcb_struct_size(int which) { return which == 0 ? (int)sizeof(mcb_counts) : which == 1 ? (int)sizeof(mcb_step_data) : MCB_E_ARG; }

const char* mcb_status_string(int s) {
    switch (s) {
        case MCB_OK: return "ok";
        case MCB_E_PARSE: return "equation rejected";
        case MCB_E_ARG: return "argument out of range";
        case MCB_E_CUDA: return "CUDA failure";
        case MCB_E_NOMEM: return "out of memory";
        case MCB_E_STATE: return "call out of order";
        case MCB_E_CAPACITY: return "capacity exceeded";
        case MCB_E_NODEVICE: return "no CUDA device (there is no CPU fallback)";
        default: return "unknown status";
    }
}

int mcb_parse(const char* equation) { return mcb_grammar_text(equation, MCB_GRAMMAR_REFERENCE, -1, nullptr, 0); }

int mcb_tokens(const char* equation, char* out, size_t cap) { return mcb_grammar_text(equation, MCB_GRAMMAR_REFERENCE, 0, out, cap); }

int mcb_postfix(const char* equation, char* out, size_t cap) { return mcb_grammar_text(equation, MCB_GRAMMAR_REFERENCE, 1, out, cap); }

int mcb_disassemble(const char* equation, int which, char* out, size_t cap) {
    return mcb_grammar_text(equation, MCB_GRAMMAR_REFERENCE, 2 + (which == 0 || which == 1 || which == 3 ? which : 2), out, cap);
}

int mcb_grammar_text(const char* equation, int grammar, int what, char* out, size_t cap) {
    if (grammar != MCB_GRAMMAR_REFERENCE && grammar != MCB_GRAMMAR_FUNCTIONS) return MCB_E_ARG;
    if (what == 0) {
        std::vector<mcb::Token> t;
        if (!mcb::tokenize(equation ? equation : "", t, nullptr, grammar)) return MCB_E_PARSE;
        std::string s;
        for (size_t i = 0; i < t.size(); i++) { if (i) s += ' '; s += t[i].text; }
        return copy_text(s, out, cap);
    }
    mcb::Compiled c;
    int rc = mcb::compile(equation ? equation : "", c, nullptr, grammar);
    if (rc != MCB_OK || what < 0) return rc;
    std::string s;
    if (what == 1) s = mcb::postfix_text(c.expr);
    else if (what == 2) s = mcb::disassemble(c.point_code);
    else if (what == 3) s = mcb::disassemble(c.grid_code);
    else if (what == 5) s = mcb::disassemble_fused(c.grid_fused);
    else {
        for (const mcb::Slot& sl : c.slots) {
            std::vector<uint32_t> code(c.slot_code.begin() + sl.code_begin, c.slot_code.begin() + sl.code_begin + sl.code_len);
            char head[64];
            std::snprintf(head, sizeof head, "%s%d: ", sl.axis < 0 ? "K" : sl.axis == 0 ? "TX" : sl.axis == 1 ? "TY" : "TZ", sl.kindex);
            s += head + mcb::disassemble(code) + "\n";
        }
    }
    return copy_text(s, out, cap);
}

int mcb_grid_axis(float step, float* coords, int cap) {
    if (!(step > 0.f) || !(step <= 1.0f) || !std::isfinite(step)) return MCB_E_ARG;
    if (2.0 / (double)step > 4094.0) return MCB_E_ARG;
    std::vector<float> c = reference_axis(step);
    int M = (int)c.size() - 1;
    if (M > 4094) return MCB_E_ARG;
    if (coords && cap >= M + 1) std::copy(c.begin(), c.end(), coords);
    return M;
}

uint64_t mcb_tri_row(int table_idx) { return (table_idx >= 0 && table_idx < 256) ? MCB_TRI_WORDS[table_idx] : ~0ull; }

int mcb_slab_range(int M, int rank, int nranks, int* k_begin, int* k_end) {
    if (M <= 0 || nranks <= 0 || rank < 0 || rank >= nranks || !k_begin || !k_end) return MCB_E_ARG;
    *k_begin = (int)((long long)M * rank / nranks);
    *k_end = (int)((long long)M * (rank + 1) / nranks);
    return MCB_OK;
}

int mcb_create(int device, mcb_ctx** out) {
    if (!out) return MCB_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return MCB_E_NODEVICE;
    mcb_ctx* ctx = new (std::nothrow) mcb_ctx();
    if (!ctx) return MCB_E_NOMEM;
    ctx->device = device;
    auto bail = [&](int code) { mcb_destroy(ctx); return code; };
    if (cudaSetDevice(device) != cudaSuccess) return bail(MCB_E_NODEVICE);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(MCB_E_NODEVICE);
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MCB_E_CUDA);
    ctx->stream = ctx->own_stream;
    for (auto& e : ctx->ev)
        if (cudaEventCreate(&e) != cudaSuccess) return bail(MCB_E_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MCB_E_CUDA);
    for (auto& e : ctx->seg_ev)
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(MCB_E_CUDA);
    for (auto& e : ctx->fork_ev)
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(MCB_E_CUDA);
    if (cudaMalloc((void**)&ctx->d_bounds, 3 * 9 * 8) != cudaSuccess) return bail(MCB_E_NOMEM);
    if (cudaMallocHost((void**)&ctx->h_bounds, 3 * 9 * 8) != cudaSuccess) return bail(MCB_E_NOMEM);
    if (cudaMalloc((void**)&ctx->d_ctr, sizeof(Counters)) != cudaSuccess) return bail(MCB_E_NOMEM);
    if (cudaMallocHost((void**)&ctx->h_ctr, sizeof(Counters)) != cudaSuccess) return bail(MCB_E_NOMEM);
    ClsTables tb;
    int8_t face[256];
    mcb_build_ambiguity_faces(face);
    for (int q = 0; q < 256; q++) {
        tb.tri[q] = MCB_TRI_WORDS[q];
        tb.face[q] = face[q];
        tb.ntri[q] = (uint8_t)mcb_tri_count(MCB_TRI_WORDS[q]);
        tb.emask[q] = 0;
        for (int e = 0; e < 12; e++) tb.emask[q] |= (uint16_t)((((q >> mcb_edge_a(e)) ^ (q >> mcb_edge_b(e))) & 1) << e);
    }
    if (cudaMalloc((void**)&ctx->d_cls, sizeof(ClsTables)) != cudaSuccess) return bail(MCB_E_NOMEM);
    if (cudaMemcpy(ctx->d_cls, &tb, sizeof tb, cudaMemcpyHostToDevice) != cudaSuccess) return bail(MCB_E_CUDA);
    {
        const int stack_bytes = MCB_MAX_STACK * kEvalRows * kEvalThreads * (int)sizeof(float);
        const void* evals[] = {(const void*)eval_field_kernel<true, true>, (const void*)eval_field_kernel<false, true>,
                               (const void*)eval_blocks_kernel<true>,      (const void*)eval_blocks_kernel<false>,
                               (const void*)eval_field_kernel<true, true, true>, (const void*)eval_blocks_kernel<true, true>,
                               (const void*)eval_field_kernel<true, true, true, true>, (const void*)eval_field_kernel<false, true, false, true>,
                               (const void*)eval_blocks_kernel<true, true, true>, (const void*)eval_blocks_kernel<false, false, true>};
        for (const void* k : evals)
            if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, stack_bytes) != cudaSuccess) return bail(MCB_E_CUDA);
        const char* poison = std::getenv("MCB_POISON_FIELD");
        ctx->poison_field = poison && poison[0] == '1';
        const char* js = std::getenv("MCB_JIT_SYNC");
        ctx->jit_sync = js && js[0] == '1';
        const char* noiv = std::getenv("MCB_NO_INTERVAL");
        ctx->decide_blocks = !(noiv && noiv[0] == '1');
    }
    int rc = install_equation(ctx, 0, "x+y"); /* Evaluator::Evaluator(), evaluator.cpp:6-8 */
    if (rc != MCB_OK) return bail(rc);
    rc = mcb_set_grid_step(ctx, 0.25f); /* Marching::Marching(), marching.cpp:24 */
    if (rc < 0) return bail(rc);
    *out = ctx;
    return MCB_OK;
}

void mcb_destroy(mcb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto& s : ctx->eq) free_slot(s);
    for (auto& kv : ctx->jit_cache) if (kv.second.lib) cudaLibraryUnload(kv.second.lib);
    cudaFree(ctx->d_fflags); cudaFree(ctx->d_flist); cudaFree(ctx->d_cw); cudaFree(ctx->d_bcls); cudaFree(ctx->d_elist); cudaFree(ctx->d_cand); cudaFree(ctx->d_scls); cudaFree(ctx->d_slist);
    cudaFree(ctx->d_bounds_iv); cudaFree(ctx->d_ent); cudaFree(ctx->d_tile_u32); cudaFree(ctx->d_amb);
    cudaFree(ctx->d_cs); cudaFree(ctx->d_F); cudaFree(ctx->d_S); cudaFree(ctx->d_V); cudaFree(ctx->d_tables);
    cudaFree(ctx->d_cls); cudaFree(ctx->d_ctr);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    cudaFree(ctx->d_rec); cudaFree(ctx->d_trioff); cudaFree(ctx->d_pos); cudaFree(ctx->d_nrm);
    cudaFree(ctx->d_vlist); cudaFree(ctx->d_vnrm); cudaFree(ctx->d_tlist); cudaFree(ctx->d_item); cudaFree(ctx->d_vinfo);
    cudaFree(ctx->d_chunk_new); cudaFree(ctx->d_fn); cudaFree(ctx->d_nh_count); cudaFree(ctx->d_nh_start); cudaFree(ctx->d_nh_cursor);
    cudaFree(ctx->d_nh_sums); cudaFree(ctx->d_nh_adj);
    cudaFree(ctx->d_mark); cudaFree(ctx->d_changed); cudaFree(ctx->d_seed_u32); cudaFree(ctx->d_rec2); cudaFree(ctx->d_trioff2);
    for (auto& e : ctx->ev) if (e) cudaEventDestroy(e);
    for (auto& e : ctx->seg_ev) if (e) cudaEventDestroy(e);
    for (auto& e : ctx->fork_ev) if (e) cudaEventDestroy(e);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    mcb_comm_finalize(ctx);
    cudaFree(ctx->d_layer_hist);
    cudaFree(ctx->d_bounds);
    if (ctx->h_bounds) cudaFreeHost(ctx->h_bounds);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char* mcb_last_error(const mcb_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int mcb_set_stream(mcb_ctx* ctx, void* s) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return MCB_OK;
}

int mcb_set_equation(mcb_ctx* ctx, int slot, const char* equation) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (slot < 0 || slot > 3) return fail(ctx, MCB_E_ARG, "slot must be 0..3");
    return install_equation(ctx, slot, equation);
}

int mcb_set_grammar(mcb_ctx* ctx, int grammar) {
    if (!ctx) return MCB_E_ARG;
    if (grammar != MCB_GRAMMAR_REFERENCE && grammar != MCB_GRAMMAR_FUNCTIONS) return fail(ctx, MCB_E_ARG, "grammar must be MCB_GRAMMAR_REFERENCE or MCB_GRAMMAR_FUNCTIONS");
    ctx->grammar = grammar;
    return MCB_OK;
}

int mcb_eval_points(mcb_ctx* ctx, int slot, const float* xyz, float* out, size_t n, int apply_scale) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (slot < 0 || slot > 3 || !ctx->eq[slot].valid) return fail(ctx, MCB_E_STATE, "no equation in that slot");
    if (n == 0) return MCB_OK;
    if (!xyz || !out) return fail(ctx, MCB_E_ARG, "null buffer");
    float *d_in = nullptr, *d_out = nullptr;
    MCB_CK(cudaMalloc((void**)&d_in, n * 3 * sizeof(float)));
    cudaError_t e = cudaMalloc((void**)&d_out, n * sizeof(float));
    if (e != cudaSuccess) { cudaFree(d_in); return fail(ctx, MCB_E_NOMEM, "cudaMalloc"); }
    float sx = apply_scale ? ctx->scale[0] : 1.f, sy = apply_scale ? ctx->scale[1] : 1.f, sz = apply_scale ? ctx->scale[2] : 1.f;
    cudaMemcpyAsync(d_in, xyz, n * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    MCB_LAUNCH((eval_points_kernel), (unsigned)((n + 127) / 128), 128, 0, ctx->stream, ctx->eq[slot].point, d_in, d_out, (long long)n, sx, sy, sz);
    cudaMemcpyAsync(out, d_out, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    e = cudaStreamSynchronize(ctx->stream);
    cudaError_t e2 = cudaGetLastError();
    cudaFree(d_in); cudaFree(d_out);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, MCB_E_CUDA, std::string("eval_points: ") + cudaGetErrorString(e != cudaSuccess ? e : e2));
    return MCB_OK;
}

int mcb_eval_gradients(mcb_ctx* ctx, int slot, const float* xyz, float* grad, size_t n, int apply_scale) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (slot < 0 || slot > 3 || !ctx->eq[slot].valid) return fail(ctx, MCB_E_STATE, "no equation in that slot");
    if (n == 0) return MCB_OK;
    if (!xyz || !grad) return fail(ctx, MCB_E_ARG, "null buffer");
    float *d_in = nullptr, *d_out = nullptr;
    MCB_CK(cudaMalloc((void**)&d_in, n * 3 * sizeof(float)));
    cudaError_t e = cudaMalloc((void**)&d_out, n * 3 * sizeof(float));
    if (e != cudaSuccess) { cudaFree(d_in); return fail(ctx, MCB_E_NOMEM, "cudaMalloc"); }
    float sx = apply_scale ? ctx->scale[0] : 1.f, sy = apply_scale ? ctx->scale[1] : 1.f, sz = apply_scale ? ctx->scale[2] : 1.f;
    cudaMemcpyAsync(d_in, xyz, n * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    MCB_LAUNCH((eval_gradients_kernel), (unsigned)((n + 127) / 128), 128, 0, ctx->stream, ctx->eq[slot].point, d_in, d_out, (long long)n, sx, sy, sz);
    cudaMemcpyAsync(grad, d_out, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    e = cudaStreamSynchronize(ctx->stream);
    cudaError_t e2 = cudaGetLastError();
    cudaFree(d_in); cudaFree(d_out);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, MCB_E_CUDA, std::string("eval_gradients: ") + cudaGetErrorString(e != cudaSuccess ? e : e2));
    return MCB_OK;
}

int mcb_set_grid_step(mcb_ctx* ctx, float step) {
    if (!ctx) return MCB_E_ARG;
    int M = mcb_grid_axis(step, nullptr, 0);
    if (M < 0) return fail(ctx, MCB_E_ARG, "grid step out of range");
    ctx->axis = reference_axis(step);
    ctx->step = step;
    ctx->M = M;
    ctx->kb = 0;
    ctx->ke = M;
    ctx->grid_dirty = true;
    ctx->have_result = false;
    return M;
}

int mcb_set_slab(mcb_ctx* ctx, int k_begin, int k_end) {
    if (!ctx) return MCB_E_ARG;
    if (k_end <= 0) k_end = ctx->M;
    if (k_begin < 0 || k_begin >= k_end || k_end > ctx->M) return fail(ctx, MCB_E_ARG, "slab out of range");
    ctx->kb = k_begin;
    ctx->ke = k_end;
    ctx->grid_dirty = true;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_surface_constant(mcb_ctx* ctx, float iso) {
    if (!ctx) return MCB_E_ARG;
    ctx->iso = iso;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_scaling(mcb_ctx* ctx, float sx, float sy, float sz) {
    if (!ctx) return MCB_E_ARG;
    ctx->scale[0] = sx; ctx->scale[1] = sy; ctx->scale[2] = sz;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_constraint(mcb_ctx* ctx, int i, int op, float rhs, int in_use) {
    if (!ctx) return MCB_E_ARG;
    if (i < 0 || i > 2 || op < 0 || op > 3) return fail(ctx, MCB_E_ARG, "constraint index 0..2, op 0..3");
    if (in_use && !ctx->eq[i + 1].valid) return fail(ctx, MCB_E_STATE, "constraint has no left-hand side (mcb_set_equation slot i+1)");
    ctx->cons[i].op = op; ctx->cons[i].rhs = rhs; ctx->cons[i].in_use = in_use != 0;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_inspect_cube(mcb_ctx* ctx, float x0, float y0, float z0, mcb_step_data* out) {
    static_assert(sizeof(StepOut) == sizeof(mcb_step_data), "StepOut mirrors mcb_step_data");
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!out) return fail(ctx, MCB_E_ARG, "null output");
    if (!ctx->eq[0].valid) return fail(ctx, MCB_E_STATE, "no surface equation");
    mcb_program* d_progs = nullptr;
    StepOut* d_out = nullptr;
    MCB_CK(cudaMalloc((void**)&d_progs, 4 * sizeof(mcb_program)));
    if (cudaMalloc((void**)&d_out, sizeof(StepOut)) != cudaSuccess) { cudaFree(d_progs); return fail(ctx, MCB_E_NOMEM, "cudaMalloc"); }
    InspectCons cons{};
    int slots[3] = {0, 0, 0};
    for (int i = 0; i < 3; i++) {
        if (!(ctx->cons[i].in_use && ctx->eq[i + 1].valid)) continue;
        cons.op[cons.n] = ctx->cons[i].op; cons.rhs[cons.n] = ctx->cons[i].rhs; slots[cons.n] = i + 1; cons.n++;
    }
    for (int sl = 0; sl < 4; sl++)
        if (ctx->eq[sl].valid) cudaMemcpyAsync(d_progs + sl, &ctx->eq[sl].point, sizeof(mcb_program), cudaMemcpyHostToDevice, ctx->stream);
    MCB_LAUNCH((inspect_cube_kernel), 1, 1, 0, ctx->stream, d_progs, cons, slots[0], slots[1], slots[2], x0, y0, z0, ctx->step, ctx->scale[0],
                                                  ctx->scale[1], ctx->scale[2], ctx->iso, ctx->repeat_on ? 1 : 0, ctx->repeat_step, ctx->d_cls, d_out);
    cudaMemcpyAsync(out, d_out, sizeof(StepOut), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    cudaError_t e2 = cudaGetLastError();
    cudaFree(d_progs); cudaFree(d_out);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, MCB_E_CUDA, std::string("inspect_cube: ") + cudaGetErrorString(e != cudaSuccess ? e : e2));
    return MCB_OK;
}

int mcb_set_repeat(mcb_ctx* ctx, int enabled, float distance) {
    if (!ctx) return MCB_E_ARG;
    if (enabled && !(distance > 0.f)) return fail(ctx, MCB_E_ARG, "the distance between repeated surfaces must be positive"); /* marching.cpp:156-162 */
    ctx->repeat_on = enabled != 0;
    if (enabled) ctx->repeat_step = distance;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_seed(mcb_ctx* ctx, int enabled, float x, float y, float z) {
    if (!ctx) return MCB_E_ARG;
    if (enabled && !((x <= 1 && x >= -1) && (y >= -1 && y <= 1) && (z >= -1 && z <= 1))) /* marching.cpp:128-137 */
        return fail(ctx, MCB_E_ARG, "seed outside [-1,1]^3");
    ctx->seed_on = enabled != 0;
    if (enabled) { ctx->seed[0] = x; ctx->seed[1] = y; ctx->seed[2] = z; }
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_normals(mcb_ctx* ctx, int mode) {
    if (!ctx || mode < 0 || mode > 3) return MCB_E_ARG;
    ctx->normals = mode;
    ctx->have_result = false;
    return MCB_OK;
}

} /* extern "C" */

namespace {

/* One mcb_polygonise call, stage by stage.  Every stage only enqueues work on the context's stream; the host reads
 * the counters once at the end (seed mode and streamed output need them earlier and synchronise there). */
struct Run {
    mcb_ctx* ctx;
    Grid& g;
    EqSlot& eq;
    cudaStream_t s;
    bool any_constraint, want_soup, want_indexed;
    const uint32_t* dV; /* constraint validity planes or nullptr */
    ClsGeom cg;
    unsigned tiles, eblocks;
    uint32_t launches;

    int prepare_buffers();
    int encode_program(mcb_program& launch, bool& has_pow, bool& has_fn, bool& has_minmax, bool blocks);
    int ensure_block_buffers(FieldBlocks* fb, BlockDims* bd);
    int launch_block_eval(const FieldBlocks& fb, const uint32_t* list, const unsigned* count);
    int stage_eval_blocks();
    int stage_fill();
    int launch_eval_jit();
    int stage_tables();
    int stage_eval();
    int stage_classify();
    int stage_seed();
    int stage_soup();
    int stage_weld();
    int stage_normal_h();
    int stage_grad_normals(bool soup);
};

int Run::prepare_buffers() {
    int rc;
    const size_t ntab = (size_t)3 * eq.max_per_axis * g.P + 256; /* the last 128-column tile reads past the pitch */
    if ((rc = ensure(ctx, &ctx->d_tables, &ctx->cap_tables, ntab)) != MCB_OK) return rc;
    if (any_constraint) {
        const size_t nS = (size_t)g.NZ * g.NV * g.WP + 64;
        if ((rc = ensure(ctx, &ctx->d_V, &ctx->cap_V, nS)) != MCB_OK) return rc;
    }
    if (ctx->cap_active == 0) {
        unsigned long long guess = std::max<unsigned long long>(1ull << 16, 8ull * g.M * g.M);
        guess = std::min<unsigned long long>(guess, (unsigned long long)(g.ke - g.kb) * g.M * g.M);
        if ((rc = ensure_records(ctx, std::max<unsigned long long>(guess, 1024))) != MCB_OK) return rc;
    }
    if (want_soup && (ctx->cap_tris == 0 || (ctx->normals && !ctx->nrm_allocated))) {
        if ((rc = ensure_soup(ctx, std::max<unsigned long long>(2 * ctx->cap_active, 1024), ctx->normals != 0)) != MCB_OK) return rc;
    }
    if (want_indexed) {
        if ((rc = ensure_indexed(ctx, std::max<unsigned long long>(ctx->cap_verts, std::max<unsigned long long>(ctx->cap_active + ctx->cap_active / 4, 1024)),
                                 std::max<unsigned long long>(ctx->cap_itris, std::max<unsigned long long>(2 * ctx->cap_active, 1024)), ctx->normals != 0)) != MCB_OK) return rc;
    }
    return MCB_OK;
}

/* Device form of the fused grid program: dense handler numbers, table operands as absolute float offsets into
 * d_tables, and  LOAD/PUSH a ; op b  pairs folded into one two-word instruction (eval_pair). */
int Run::encode_program(mcb_program& launch, bool& has_pow, bool& has_fn, bool& has_minmax, bool blocks) {
    launch = eq.grid;
    has_pow = false;
    has_fn = false;
    has_minmax = false;
    {
        /* operand class of a source as the kernel's lane patch sees it; eval_blocks_kernel's patch is (y, z) per x
         * column, so there the x and z tables trade places */
        auto role = [blocks](uint32_t src) { return !blocks ? src : src == MCB_SRC_TX ? (uint32_t)MCB_SRC_TZ : src == MCB_SRC_TZ ? (uint32_t)MCB_SRC_TX : src; };
        auto leaf_class = [&](uint32_t src0) { const uint32_t src = role(src0); return src == MCB_SRC_K ? 0 : src == MCB_SRC_TX ? 1 : src == MCB_SRC_TY ? 2 : src == MCB_SRC_TZ ? 3 : -1; };
        auto resolve = [&](uint32_t src, uint32_t arg, uint32_t* out) {
            if (src >= MCB_SRC_TX && src <= MCB_SRC_TZ) {
                const size_t off = ((size_t)(src - MCB_SRC_TX) * eq.max_per_axis + arg) * g.P;
                if (off >= (1u << 24)) return false;
                arg = (uint32_t)off;
            }
            *out = arg;
            return true;
        };
        int n = 0;
        for (int pc = 0; pc < eq.grid.n; pc++) {
            const uint32_t wd = eq.grid.code[pc];
            uint32_t fop = MCB_FINSN_OP(wd), src = MCB_FINSN_SRC(wd);
            MCB_FINSN_DECODE(fop, src);
            const bool minmax = fop == MCB_F_MIN || fop == MCB_F_MAX;
            has_pow |= fop == MCB_F_POW || fop == MCB_F_RPOW;
            has_minmax |= minmax;
            if (fop == MCB_F_NEG) { launch.code[n++] = MCB_HANDLER_NEG; continue; }
            if (MCB_F_IS_FN(fop)) { launch.code[n++] = MCB_HANDLER_FN(fop); has_fn = true; continue; }
            if (src < MCB_SRC_K || src > MCB_SRC_POP) return fail(ctx, MCB_E_STATE, "internal: raw coordinate operand in a grid program");
            uint32_t arg;
            if (!resolve(src, MCB_FINSN_ARG(wd), &arg)) return fail(ctx, MCB_E_CAPACITY, "axis tables too large for the operand field");
            if ((fop == MCB_F_LOAD || fop == MCB_F_PUSH) && pc + 1 < eq.grid.n) {
                const uint32_t nx = eq.grid.code[pc + 1];
                uint32_t nop = MCB_FINSN_OP(nx), nsrc = MCB_FINSN_SRC(nx);
                MCB_FINSN_DECODE(nop, nsrc);
                const bool nminmax = nop == MCB_F_MIN || nop == MCB_F_MAX;
                if (((nop >= MCB_F_ADD && nop <= MCB_F_RPOW) || nminmax) && leaf_class(nsrc) >= 0) {
                    uint32_t arg_b;
                    if (!resolve(nsrc, MCB_FINSN_ARG(nx), &arg_b)) return fail(ctx, MCB_E_CAPACITY, "axis tables too large for the operand field");
                    has_pow |= nop == MCB_F_POW || nop == MCB_F_RPOW;
                    if (n + 2 + (fop == MCB_F_PUSH ? 1 : 0) > MCB_MAX_CODE) return fail(ctx, MCB_E_CAPACITY, "program too long");
                    if (fop == MCB_F_PUSH) launch.code[n++] = MCB_HANDLER_SPILL;
                    has_minmax |= nminmax;
                    launch.code[n++] = (uint32_t)(nminmax ? MCB_HANDLER_MINMAX_PAIR(nop, leaf_class(src), leaf_class(nsrc))
                                                          : MCB_HANDLER_PAIR(nop, leaf_class(src), leaf_class(nsrc))) | (arg << 8);
                    launch.code[n++] = arg_b;
                    pc++;
                    continue;
                }
            }
            if (n + 1 > MCB_MAX_CODE) return fail(ctx, MCB_E_CAPACITY, "program too long");
            const uint32_t cls = src == MCB_SRC_POP ? 4u : (uint32_t)leaf_class(src);
            launch.code[n++] = (uint32_t)(minmax ? MCB_HANDLER_MINMAX(fop, cls) : MCB_HANDLER(fop, role(src))) | (arg << 8); /* dense handler number | operand */
        }
        launch.n = n;
    }
    return MCB_OK;
}

/* K0b: per-axis tables of the hoisted single-variable subtrees */
int Run::stage_tables() {
    if (eq.n_axis > 0) {
        dim3 grid((g.P + 127) / 128, eq.n_axis);
        MCB_LAUNCH((axis_tables_kernel), grid, 128, 0, s, eq.d_slot_code, eq.d_slots, eq.n_const, eq.d_kpool, ctx->d_cs, g.NV, g.P,
                                                eq.max_per_axis, g.sx, g.sy, g.sz, ctx->d_tables);
        launches++;
    }
    return MCB_OK;
}

/* The module NVRTC compiled for this equation (mcb_jit.cpp), from the per-context cache or compiled now.
 * Returns MCB_OK with *out set, or a status with the reason in ctx->err. */
constexpr int kJitDeferred = 1; /* not an error: the compile runs in the background, this call interprets */

int jit_adopt(mcb_ctx* ctx, const std::string& src, const std::vector<char>& cubin, float ms, const mcb_ctx::JitKernel** out) {
    mcb_ctx::JitKernel jk;
    MCB_CK(cudaLibraryLoadData(&jk.lib, (void*)cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
    cudaError_t e = cudaLibraryGetKernel(&jk.kernel, jk.lib, "mcb_eval_jit");
    if (e == cudaSuccess) e = cudaLibraryGetKernel(&jk.fill, jk.lib, "mcb_fill_jit");
    if (e != cudaSuccess) {
        cudaLibraryUnload(jk.lib);
        return fail(ctx, MCB_E_CUDA, std::string("cudaLibraryGetKernel: ") + cudaGetErrorString(e));
    }
    if (ctx->jit_cache.size() >= 64) { /* a long GUI session types many equations: keep the cache bounded */
        for (auto& kv : ctx->jit_cache) if (kv.second.lib) cudaLibraryUnload(kv.second.lib);
        ctx->jit_cache.clear();
        ctx->jit_cur = nullptr;
    }
    *out = &ctx->jit_cache.emplace(src, jk).first->second;
    ctx->ms_compile += ms;
    return MCB_OK;
}

/* The module NVRTC compiled for this equation (mcb_jit.cpp): from the per-context cache, compiled now, or — MCB_JIT_AUTO,
 * `wait` false — being compiled by a background thread, in which case kJitDeferred is returned until it is there.
 * Returns MCB_OK with *out set, kJitDeferred, or a status with the reason in ctx->err. */
int jit_module(mcb_ctx* ctx, const EqSlot& eq, const mcb_ctx::JitKernel** out, bool wait = false) {
    std::string err;
    bool has_pow = false;
    const std::string src = mcbjit::generate(eq.grid.code, eq.grid.n, &has_pow, &err);
    if (src.empty()) return fail(ctx, MCB_E_STATE, "run-time specialisation: " + err);
    auto it = ctx->jit_cache.find(src);
    if (it != ctx->jit_cache.end()) { *out = &it->second; return MCB_OK; }
    auto bad = ctx->jit_failed.find(src);
    if (bad != ctx->jit_failed.end()) return fail(ctx, MCB_E_STATE, "run-time specialisation: " + bad->second);
    auto pend = ctx->jit_pending.find(src);
    const bool background = ctx->jit == MCB_JIT_AUTO && !ctx->jit_sync && !wait;
    if (pend == ctx->jit_pending.end() && background) {
        if (ctx->jit_pending.size() >= 8) return kJitDeferred; /* equations typed faster than they compile: interpret */
        const int grid_bytes = (int)sizeof(Grid);
        bool started = true;
        try {
            ctx->jit_pending.emplace(src, std::async(std::launch::async, [src, has_pow, grid_bytes]() {
                mcb_ctx::JitBuilt b;
                const auto t0 = std::chrono::steady_clock::now();
                b.err = mcbjit::compile(src, has_pow, grid_bytes, &b.cubin);
                b.ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
                return b;
            }));
        } catch (...) { started = false; } /* a host program that cannot start threads: compile here, below */
        if (started) return kJitDeferred;
    }
    if (pend != ctx->jit_pending.end()) {
        if (background && pend->second.wait_for(std::chrono::seconds(0)) != std::future_status::ready) return kJitDeferred;
        mcb_ctx::JitBuilt b = pend->second.get(); /* blocks when the caller wants the kernel now (MCB_JIT_ON, mcb_jit_wait) */
        ctx->jit_pending.erase(pend);
        if (!b.err.empty()) {
            if (ctx->jit_failed.size() < 64) ctx->jit_failed.emplace(src, b.err);
            return fail(ctx, MCB_E_STATE, "run-time specialisation: " + b.err);
        }
        const int rc = jit_adopt(ctx, src, b.cubin, b.ms, out);
        if (rc != MCB_OK && ctx->jit_failed.size() < 64) ctx->jit_failed.emplace(src, ctx->err); /* not compiled over and over */
        return rc;
    }
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<char> cubin;
    const std::string cerr = mcbjit::compile(src, has_pow, (int)sizeof(Grid), &cubin);
    if (!cerr.empty()) {
        if (ctx->jit_failed.size() < 64) ctx->jit_failed.emplace(src, cerr);
        return fail(ctx, MCB_E_STATE, "run-time specialisation: " + cerr);
    }
    const int rc = jit_adopt(ctx, src, cubin, std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count(), out);
    if (rc != MCB_OK && ctx->jit_failed.size() < 64) ctx->jit_failed.emplace(src, ctx->err);
    return rc;
}

/* auto: a program full of general `^` is bound by powf either way, and each inlined powf site costs compile time
 * (13 of them: seconds) — leave those to the interpreter */
bool jit_wanted(const mcb_ctx* ctx, const EqSlot& eq) {
    int n_pow = 0;
    for (int pc = 0; pc < eq.grid.n; pc++) {
        const uint32_t fop = MCB_FINSN_OP(eq.grid.code[pc]);
        n_pow += fop == MCB_F_POW || fop == MCB_F_RPOW;
    }
    return ctx->jit == MCB_JIT_ON || (ctx->jit == MCB_JIT_AUTO && n_pow <= 8);
}

/* The dense evaluation by the kernel compiled for this equation: same tile, same launch geometry as eval_field_kernel */
int Run::launch_eval_jit() {
    const mcb_ctx::JitKernel* jk = nullptr;
    int rc = jit_module(ctx, eq, &jk);
    if (rc != MCB_OK) return rc;
    const int rgpp = (g.NV + kEvalTileY - 1) / kEvalTileY;
    const dim3 blocks((unsigned)((g.P + kEvalTileX - 1) / kEvalTileX), (unsigned)((rgpp + kEvalThreads / 32 - 1) / (kEvalThreads / 32)),
                      (unsigned)g.NZ);
    struct { float k[MCB_MAX_K]; } consts;
    std::memcpy(consts.k, eq.grid.k, sizeof consts.k);
    Grid garg = g;
    const float* tables = ctx->d_tables;
    float* F = ctx->d_F;
    uint32_t* S = ctx->d_S;
    int rg = rgpp, spa = eq.max_per_axis;
    void* args[] = {&consts, &garg, &tables, &F, &S, &rg, &spa};
    MCB_CK(cudaLaunchKernel((const void*)jk->kernel, blocks, dim3(kEvalThreads), args, 0, s));
#ifdef __CUDACC__
    if (mcb_debug_sync_on()) mcb_debug_sync_check("mcb_eval_jit", s);
#endif
    ctx->jit_cur = jk;
    launches++;
    return MCB_OK;
}

/* K1b: constraint validity bit-planes */
int launch_constraints(Run& r) {
    mcb_ctx* ctx = r.ctx;
    if (!r.any_constraint) return MCB_OK;
    const long long words = (long long)r.g.NZ * r.g.NV * r.g.WP;
    int first = 1;
    for (int i = 0; i < 3; i++) {
        if (!(ctx->cons[i].in_use && ctx->eq[i + 1].valid)) continue;
        MCB_LAUNCH((eval_constraint_kernel), (unsigned)((words + 7) / 8), 256, 0, r.s, ctx->eq[i + 1].point, r.g, ctx->d_cs, ctx->cons[i].op,
                   ctx->cons[i].rhs, first, ctx->d_V, words);
        first = 0;
        r.launches++;
    }
    return MCB_OK;
}

/* K1, MCB_FIELD_DENSE: field + sign bit-planes at every grid vertex */
int Run::stage_eval() {
    const int rgpp = (g.NV + kEvalTileY - 1) / kEvalTileY; /* 4-row groups per plane */
    const dim3 blocks((unsigned)((g.P + kEvalTileX - 1) / kEvalTileX), (unsigned)((rgpp + kEvalThreads / 32 - 1) / (kEvalThreads / 32)),
                      (unsigned)g.NZ);
    ctx->jit_used = false;
    ctx->field_is_sparse = false;
    int rc;
    if (jit_wanted(ctx, eq)) {
        rc = launch_eval_jit();
        if (rc == MCB_OK) ctx->jit_used = true;
        else if (rc == kJitDeferred) ctx->jit_note = "compiling in the background";
        else if (ctx->jit == MCB_JIT_ON) return rc;      /* asked for explicitly: fail loudly */
        else ctx->jit_note = ctx->err;                   /* auto: the interpreter below does the same work */
    }
    if (!ctx->jit_used) {
        const size_t smem = (size_t)std::max(1, eq.c.grid_fused_depth) * kEvalRows * kEvalThreads * sizeof(float);
        mcb_program launch;
        bool has_pow, has_fn, has_minmax;
        if ((rc = encode_program(launch, has_pow, has_fn, has_minmax, false)) != MCB_OK) return rc;
        if (has_minmax && (has_pow || has_fn)) MCB_LAUNCH((eval_field_kernel<true, true, true, true>), blocks, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, rgpp);
        else if (has_minmax) MCB_LAUNCH((eval_field_kernel<false, true, false, true>), blocks, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, rgpp);
        else if (has_fn) MCB_LAUNCH((eval_field_kernel<true, true, true>), blocks, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, rgpp);
        else if (has_pow) MCB_LAUNCH((eval_field_kernel<true, true>), blocks, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, rgpp);
        else MCB_LAUNCH((eval_field_kernel<false, true>), blocks, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, rgpp);
        launches++;
    }
    return launch_constraints(*this);
}

/* the 32 x 4 x 4 vertex blocks of the slab and everything indexed by them */
int Run::ensure_block_buffers(FieldBlocks* fb, BlockDims* bd) {
    bd->nbx = g.P / kFieldBlockX;
    bd->nby = (g.NV + kFieldBlockY - 1) / kFieldBlockY;
    bd->nbz = (g.NZ + kFieldBlockZ - 1) / kFieldBlockZ;
    bd->nsy = (bd->nby + kSuper - 1) / kSuper;
    bd->nsz = (bd->nbz + kSuper - 1) / kSuper;
    bd->nb = std::max(bd->nbx, std::max(bd->nby, bd->nbz));
    bd->spa = eq.max_per_axis;
    bd->WC = (int)cg.WC;
    bd->cjb = (g.M + 3) / 4;
    bd->ckb = (g.ke - g.kb + 3) / 4;
    const size_t nb = (size_t)bd->nbx * bd->nby * bd->nbz;
    if (nb >= (1ull << 32)) return fail(ctx, MCB_E_CAPACITY, "too many field blocks: split the grid into more z-slabs");
    if (ctx->cap_fblocks < nb) {
        cudaFree(ctx->d_fflags); cudaFree(ctx->d_flist); cudaFree(ctx->d_bcls); cudaFree(ctx->d_elist);
        ctx->d_fflags = nullptr; ctx->d_flist = nullptr; ctx->d_bcls = nullptr; ctx->d_elist = nullptr; ctx->cap_fblocks = 0;
        if (cudaMalloc((void**)&ctx->d_fflags, nb + 16) != cudaSuccess || cudaMalloc((void**)&ctx->d_flist, (nb + 16) * sizeof(uint32_t)) != cudaSuccess ||
            cudaMalloc((void**)&ctx->d_bcls, nb + 16) != cudaSuccess || cudaMalloc((void**)&ctx->d_elist, (nb + 16) * sizeof(uint32_t)) != cudaSuccess)
            return fail(ctx, MCB_E_NOMEM, "cudaMalloc of the field-block lists failed");
        MCB_CK(cudaMemsetAsync(ctx->d_fflags, 0, nb + 16, s)); /* the padding field_list_kernel reads stays zero */
        MCB_CK(cudaMemsetAsync(ctx->d_bcls, 0, nb + 16, s));
        ctx->cap_fblocks = nb;
    }
    int rc;
    if ((rc = ensure(ctx, &ctx->d_bounds_iv, &ctx->cap_bounds_iv, (size_t)2 * 3 * bd->spa * bd->nb)) != MCB_OK) return rc;
    if ((rc = ensure(ctx, &ctx->d_cand, &ctx->cap_cand, (size_t)((bd->WC + 63) / 64) * bd->cjb * bd->ckb)) != MCB_OK) return rc;
    const size_t nsup = (size_t)bd->nbx * bd->nsy * bd->nsz;
    if (ctx->cap_scls < nsup) {
        cudaFree(ctx->d_scls); cudaFree(ctx->d_slist);
        ctx->d_scls = nullptr; ctx->d_slist = nullptr; ctx->cap_scls = 0;
        MCB_CK(cudaMalloc((void**)&ctx->d_scls, nsup));
        MCB_CK(cudaMalloc((void**)&ctx->d_slist, nsup * sizeof(uint32_t)));
        ctx->cap_scls = nsup;
    }
    *fb = FieldBlocks{bd->nbx, bd->nby, bd->nbz, ctx->d_fflags, ctx->d_flist};
    ctx->bd = *bd;
    return MCB_OK;
}

/* field values + sign words of the listed blocks: the kernel compiled for the equation, or the interpreter */
int Run::launch_block_eval(const FieldBlocks& fb, const uint32_t* list, const unsigned* count) {
    const unsigned fill_ctas = (unsigned)ctx->sm_count * 16;
    int rc;
    if (ctx->jit_used && ctx->jit_cur && ctx->jit_cur->fill) {
        struct { float k[MCB_MAX_K]; } consts;
        std::memcpy(consts.k, eq.grid.k, sizeof consts.k);
        Grid garg = g;
        const float* tables = ctx->d_tables;
        float* F = ctx->d_F;
        uint32_t* S = ctx->d_S;
        int spa = eq.max_per_axis;
        void* args[] = {&consts, &garg, &tables, &F, &S, &list, &count, &spa};
        MCB_CK(cudaLaunchKernel((const void*)ctx->jit_cur->fill, dim3(fill_ctas), dim3(kEvalThreads), args, 0, s));
#ifdef __CUDACC__
        if (mcb_debug_sync_on()) mcb_debug_sync_check("mcb_fill_jit", s);
#endif
    } else {
        mcb_program launch;
        bool has_pow, has_fn, has_minmax;
        if ((rc = encode_program(launch, has_pow, has_fn, has_minmax, true)) != MCB_OK) return rc;
        const size_t smem = (size_t)std::max(1, eq.c.grid_fused_depth) * kEvalRows * kEvalThreads * sizeof(float);
        if (has_minmax && (has_pow || has_fn)) MCB_LAUNCH((eval_blocks_kernel<true, true, true>), fill_ctas, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, list, count);
        else if (has_minmax) MCB_LAUNCH((eval_blocks_kernel<false, false, true>), fill_ctas, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, list, count);
        else if (has_fn) MCB_LAUNCH((eval_blocks_kernel<true, true>), fill_ctas, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, list, count);
        else if (has_pow) MCB_LAUNCH((eval_blocks_kernel<true>), fill_ctas, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, list, count);
        else MCB_LAUNCH((eval_blocks_kernel<false>), fill_ctas, kEvalThreads, smem, s, launch, g, ctx->d_tables, ctx->d_F, ctx->d_S, list, count);
    }
    launches++;
    return MCB_OK;
}

/* K1, block-field mode (MCB_FIELD_SPARSE / MCB_FIELD_AUTO): interval classes per 32 x 4 x 4 vertex block, field values
 * and signs only in the undecided blocks, the candidate map for classify (mcb_kernels.cuh, "decide, evaluate, skip") */
int Run::stage_eval_blocks() {
    FieldBlocks fb;
    BlockDims bd;
    int rc = ensure_block_buffers(&fb, &bd);
    if (rc != MCB_OK) return rc;
    if (ctx->poison_field) { /* tests: a read of a field value or a sign word nobody wrote must show */
        MCB_CK(cudaMemsetAsync(ctx->d_F, 0xff, (size_t)g.NZ * g.NV * g.P * sizeof(float), s));
        MCB_CK(cudaMemsetAsync(ctx->d_S, 0x5a, (size_t)g.NZ * g.NV * g.WP * sizeof(uint32_t), s));
    }
    ctx->field_is_sparse = true;
    ctx->jit_used = false;
    if (jit_wanted(ctx, eq)) {
        const mcb_ctx::JitKernel* jk = nullptr;
        rc = jit_module(ctx, eq, &jk);
        if (rc == MCB_OK) { ctx->jit_used = true; ctx->jit_cur = jk; }
        else if (rc == kJitDeferred) ctx->jit_note = "compiling in the background";
        else if (ctx->jit == MCB_JIT_ON) return rc;
        else ctx->jit_note = ctx->err;
    }
    const size_t nblocks = (size_t)bd.nbx * bd.nby * bd.nbz;
    const unsigned nsuper = (unsigned)bd.nbx * (unsigned)bd.nsy * (unsigned)bd.nsz;
    /* the three clears run on the side stream while the bounds and the super-block classes are computed; block_class, the
     * first kernel that writes into the cleared arrays, waits for them */
    cudaStream_t side = ctx->copy_stream;
    MCB_CK(cudaEventRecord(ctx->fork_ev[0], s));
    MCB_CK(cudaStreamWaitEvent(side, ctx->fork_ev[0], 0));
    MCB_CK(cudaMemsetAsync(ctx->d_cand, 0, (size_t)((bd.WC + 63) / 64) * bd.cjb * bd.ckb * 8, side));
    MCB_CK(cudaMemsetAsync(ctx->d_fflags, 0, nblocks, side));
    MCB_CK(cudaMemsetAsync(ctx->d_bcls, 0xFF, nblocks, side)); /* kClsInherit: the super-block's verdict holds unless the fine pass says otherwise */
    MCB_CK(cudaEventRecord(ctx->fork_ev[1], side));
    MCB_LAUNCH((axis_bounds_kernel), dim3((unsigned)((3 * bd.spa * bd.nb + 127) / 128), 2u), 128, 0, s, ctx->d_tables, g, bd, eq.c.n_axis_slots[0],
               eq.c.n_axis_slots[1], eq.c.n_axis_slots[2], ctx->d_bounds_iv);
    MCB_LAUNCH((super_class_kernel), (nsuper + 127) / 128, 128, 0, s, eq.grid, g, bd, ctx->d_bounds_iv, ctx->decide_blocks ? 1 : 0, ctx->d_scls,
               ctx->d_slist, ctx->d_ctr);
    MCB_CK(cudaStreamWaitEvent(s, ctx->fork_ev[1], 0));
    MCB_LAUNCH((block_class_kernel), (unsigned)ctx->sm_count * 8, 256, 0, s, eq.grid, g, bd, ctx->d_bounds_iv, ctx->d_slist, ctx->decide_blocks ? 1 : 0,
               ctx->d_bcls, ctx->d_fflags, ctx->d_elist, ctx->d_cand, ctx->d_ctr);
    /* Two latency-bound kernels that touch disjoint blocks — the sign words of the decided neighbours, the field of the
     * undecided blocks — run side by side: the first on the side stream, joined before anything reads the sign planes */
    MCB_CK(cudaEventRecord(ctx->fork_ev[0], s));
    MCB_CK(cudaStreamWaitEvent(side, ctx->fork_ev[0], 0));
    MCB_LAUNCH((decided_signs_kernel), (unsigned)ctx->sm_count * 8, 256, 0, side, g, bd, ctx->d_elist, ctx->d_ctr, ctx->d_bcls, ctx->d_scls, ctx->d_S);
    MCB_CK(cudaEventRecord(ctx->fork_ev[1], side));
    launches += 4;
    rc = launch_block_eval(fb, ctx->d_elist, &ctx->d_ctr->eval_blocks);
    MCB_CK(cudaStreamWaitEvent(s, ctx->fork_ev[1], 0)); /* joined on every path: the side stream never outlives the call */
    if (rc != MCB_OK) return rc;
    return launch_constraints(*this);
}

/* K2: classification (per tile, independent) -> face-centre tests of the ambiguous cubes -> scan of the tile totals ->
 * compaction */
int Run::stage_classify() {
    int rc;
    MCB_CK(cudaMemsetAsync(ctx->d_ctr, 0, kCountersClassifyBytes, s)); /* the evaluation stage's counters stay */
    uint32_t* tu = ctx->d_tile_u32;
    const size_t ct = ctx->cap_tiles;
    const bool skip = ctx->field_is_sparse; /* the candidate map of the block-field mode */
    const ClsScratch sc{ctx->d_ent, tu, tu + ct, tu + 2 * ct, tu + 3 * ct, tu + 4 * ct, ctx->d_amb, ctx->cap_amb, cg.tile_rows * cg.WC,
                        skip ? ctx->d_cand : nullptr, (uint32_t)((g.M + 3) / 4), (uint32_t)((cg.WC + 63) / 64)};
    const uint32_t* cw = nullptr;
    if (g.repeat) { /* per-cube iso levels: the corner signs come from the field, item by item */
        const unsigned long long items = (unsigned long long)cg.total_rows * cg.WC;
        if ((rc = ensure(ctx, &ctx->d_cw, &ctx->cap_cw, (size_t)items * 8)) != MCB_OK) return rc;
        MCB_LAUNCH((repeat_words_kernel), (unsigned)ctx->sm_count * 8, 256, 0, s, g, ctx->d_F, cg.WC, ctx->d_cw, items);
        launches++;
        cw = ctx->d_cw;
    }
    const bool need_items = want_indexed || ctx->seed_on; /* per-word record index for the weld / the seed walk */
    if (need_items && (rc = ensure_weld_scratch(ctx, g)) != MCB_OK) return rc;
    unsigned long long* items = need_items ? ctx->d_item : nullptr;
    const unsigned amb_ctas = (unsigned)ctx->sm_count * 2;
    const FieldBlocks apron = skip ? FieldBlocks{ctx->bd.nbx, ctx->bd.nby, ctx->bd.nbz, ctx->d_fflags, ctx->d_flist} : FieldBlocks{0, 0, 0, nullptr, nullptr};
#define MCB_CLASSIFY(HAS_V, REPEAT)                                                                                                   \
    do {                                                                                                                              \
        MCB_LAUNCH((classify_kernel<HAS_V, REPEAT>), tiles, kClsThreads, kClsSmemBytes, s, g, ctx->d_cls, ctx->d_S, dV, cg, sc, ctx->d_ctr, cw); \
        MCB_LAUNCH((ambiguity_kernel<REPEAT>), amb_ctas, 128, 0, s, eq.point, g, ctx->d_cs, ctx->d_cls, sc, ctx->d_ctr, ctx->d_F);          \
        MCB_LAUNCH((tile_scan_kernel), 1, 1024, 0, s, sc, tiles, ctx->d_ctr);                                                             \
        MCB_LAUNCH((compact_kernel<REPEAT>), tiles, kClsThreads, 0, s, g, ctx->d_cls, ctx->d_S, dV, cg, sc, ctx->d_rec, ctx->d_trioff,     \
                   ctx->cap_active, items, cw, apron);                                                                                 \
    } while (0)
    if (cw) { if (dV) MCB_CLASSIFY(true, true); else MCB_CLASSIFY(false, true); }
    else { if (dV) MCB_CLASSIFY(true, false); else MCB_CLASSIFY(false, false); }
#undef MCB_CLASSIFY
    launches += 4;
    return MCB_OK;
}

/* Block-field mode: the field values the mesh stages read — the corners of the active cubes and their +-1 neighbours
 * (gradient stencil, the weld's look at neighbouring grid edges) — reach into blocks the interval test decided and the
 * evaluation therefore skipped.  Those "apron" blocks are written now by the same evaluation kernel (their sign words
 * come out as the constants they already are). */
int Run::stage_fill() {
    FieldBlocks fb;
    BlockDims bd;
    int rc = ensure_block_buffers(&fb, &bd);
    if (rc != MCB_OK) return rc;
    const size_t nb = (size_t)fb.nbx * fb.nby * fb.nbz;
    MCB_LAUNCH((field_list_kernel), (unsigned)((nb / 16 + 256) / 256), 256, 0, s, fb, (unsigned)nb, ctx->d_ctr); /* the blocks compact_kernel marked */
    launches += 1;
    return launch_block_eval(fb, ctx->d_flist, &ctx->d_ctr->field_blocks);
}

/* K6: keep the component of the seed cube (marching.cpp:42-137, 310-331) */
int Run::stage_seed() {
    int rc;
    MCB_CK(cudaMemcpyAsync(ctx->h_ctr, ctx->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
    MCB_CK(cudaStreamSynchronize(s));
    if (ctx->h_ctr->active <= ctx->cap_active) { /* otherwise the records are truncated: the re-run comes first */
        if ((rc = ensure_seed_scratch(ctx)) != MCB_OK) return rc;
        const unsigned long long n = ctx->cap_seed;
        uint32_t *keep = ctx->d_seed_u32, *ktri = keep + n, *pa = ktri + n, *pt = pa + n, *sums = pt + n;
        const SeedBuffers SB{ctx->d_rec, ctx->d_item, cg.WC, ctx->d_mark, ctx->d_changed};
        const WeldView W{g, ctx->d_cs, ctx->d_F, dV, nullptr, cg.WC};
        const unsigned sblocks = (unsigned)ctx->sm_count * 8;
        int sc3[3];
        seed_cube(ctx, sc3);
        MCB_CK(cudaMemsetAsync(ctx->d_mark, 0, std::max<unsigned long long>(ctx->h_ctr->active, 1), s));
        MCB_CK(cudaMemsetAsync(ctx->d_changed, 0, 4, s));
        if (sc3[0] >= 0 && sc3[1] >= 0 && sc3[2] >= g.kb && sc3[0] < g.M && sc3[1] < g.M && sc3[2] < g.ke) {
            MCB_LAUNCH((seed_init_kernel), 1, 1, 0, s, SB, g, ctx->d_ctr, ctx->cap_active, sc3[0], sc3[1], sc3[2]);
            launches++;
        }
        for (int round = 0; round < 100000; round++) { /* monotone marking until nothing changes */
            uint32_t changed = 0;
            MCB_CK(cudaMemcpyAsync(&changed, ctx->d_changed, 4, cudaMemcpyDeviceToHost, s));
            MCB_CK(cudaStreamSynchronize(s));
            if (!changed) break;
            MCB_CK(cudaMemsetAsync(ctx->d_changed, 0, 4, s));
            for (int q = 0; q < 8; q++) {
                MCB_LAUNCH((seed_sweep_kernel), sblocks, 256, 0, s, SB, W, ctx->d_ctr, ctx->cap_active, 0.5 * (double)ctx->step);
                launches++;
            }
        }
        const unsigned long long* na = &ctx->d_ctr->active;
        MCB_LAUNCH((seed_flags_kernel), sblocks, 256, 0, s, SB, ctx->d_cls, ctx->d_ctr, ctx->cap_active, keep, ktri);
        MCB_LAUNCH((scan_block_sums_kernel), sblocks / 2, kScanBlock, 0, s, keep, na, sums);
        MCB_LAUNCH((scan_sums_kernel), 1, kScanBlock, 0, s, sums, na);
        MCB_LAUNCH((scan_apply_kernel), sblocks / 2, kScanBlock, 0, s, keep, sums, na, pa);
        MCB_LAUNCH((scan_block_sums_kernel), sblocks / 2, kScanBlock, 0, s, ktri, na, sums);
        MCB_LAUNCH((scan_sums_kernel), 1, kScanBlock, 0, s, sums, na);
        MCB_LAUNCH((scan_apply_kernel), sblocks / 2, kScanBlock, 0, s, ktri, sums, na, pt);
        MCB_LAUNCH((seed_scatter_kernel), sblocks, 256, 0, s, SB, keep, ktri, pa, pt, ctx->d_ctr, ctx->cap_active, ctx->d_rec2, ctx->d_trioff2);
        MCB_LAUNCH((seed_commit_kernel), 1, 1, 0, s, ctx->d_ctr);
        std::swap(ctx->d_rec, ctx->d_rec2);
        std::swap(ctx->d_trioff, ctx->d_trioff2);
        launches += 9;
        if (want_indexed) { /* the weld must only see the kept cubes: rebuild the per-word look-up from scratch */
            MCB_CK(cudaMemsetAsync(ctx->d_item, 0, (size_t)(g.ke - g.kb) * g.M * cg.WC * 8, s));
            MCB_LAUNCH((seed_items_kernel), sblocks, 256, 0, s, ctx->d_rec, g, cg.WC, ctx->d_ctr, ctx->d_item);
            launches++;
        }
    }
    return MCB_OK;
}

/* K3: interpolation + coalesced float4 emission of the triangle soup */
int Run::stage_soup() {
    const float* rinv = ctx->d_cs + ctx->rinv_ofs;
    const bool idx32 = (unsigned long long)g.NZ * g.NV * g.P < (1ull << 32) - 2ull * g.NV * g.P; /* offsets +- one plane stay below 2^32 */
    const unsigned grid = (unsigned)ctx->sm_count * (unsigned)kEmitBlocksPerSM; /* one resident wave: emit2 hands out chunks itself */
#define MCB_SOUP(NRM, I32)                                                                                                            \
    MCB_LAUNCH((emit2_kernel<NRM, I32>), grid, kEmitThreads, 0, s, g, ctx->d_cs, rinv, ctx->d_F, ctx->d_cls, ctx->d_rec, ctx->d_trioff, \
               ctx->d_ctr, ctx->cap_active, ctx->cap_tris, ctx->d_pos, NRM ? ctx->d_nrm : nullptr)
    if (ctx->normals == 1) { if (idx32) MCB_SOUP(true, true); else MCB_SOUP(true, false); }
    else { if (idx32) MCB_SOUP(false, true); else MCB_SOUP(false, false); }
#undef MCB_SOUP
    launches++;
    return MCB_OK;
}

/* K4: the reference's welded, indexed mesh (Poly_Data::vertex_list / tri_list) */
int Run::stage_weld() {
    int rc;
    if ((rc = ensure_weld_scratch(ctx, g)) != MCB_OK) return rc;
    const WeldView W{g, ctx->d_cs, ctx->d_F, any_constraint ? ctx->d_V : nullptr, ctx->seed_on ? ctx->d_item : nullptr, cg.WC};
    const WeldViewT<true> WR{W.g, W.cs, W.F, W.V, W.present, W.WC}; /* repeating-surface mode: same view, level checks compiled in */
    const WeldBuffers B{ctx->d_rec, ctx->d_trioff, ctx->d_item, ctx->d_vinfo, ctx->d_chunk_new, cg.WC};
    if (g.repeat) MCB_LAUNCH((weld_count_kernel), eblocks * 2, kWeldThreads, 0, s, WR, B, ctx->d_ctr, ctx->cap_active);
    else if (W.V != nullptr || W.present != nullptr) MCB_LAUNCH((weld_count_kernel), eblocks * 2, kWeldThreads, 0, s, W, B, ctx->d_ctr, ctx->cap_active);
    else MCB_LAUNCH((weld_count_fast_kernel), eblocks * 4, kWeldCubes, 0, s, W, B, ctx->d_cls, ctx->d_ctr, ctx->cap_active);
    MCB_LAUNCH((weld_scan_kernel), 1, 1024, 0, s, ctx->d_chunk_new, ctx->d_ctr, ctx->cap_active);
    MCB_LAUNCH((weld_base_kernel), eblocks * 2, kWeldCubes, 0, s, B, ctx->d_ctr, ctx->cap_active);
    /* streaming: with a registered host destination and everything fitting, weld_emit runs range by range and
     * each finished range of vertices / normals / triangles leaves over PCIe on the copy stream meanwhile */
    constexpr int K = 8;
    bool stream_out = ctx->h_out_v && ctx->h_out_t && ctx->normals <= 1 && (ctx->normals == 0 || ctx->h_out_n);
    ctx->streamed = false;
    if (stream_out) {
        MCB_LAUNCH((weld_bounds_kernel), 1, 32, 0, s, B, ctx->d_ctr, ctx->cap_active, K, ctx->d_bounds);
        MCB_CK(cudaMemcpyAsync(ctx->h_bounds, ctx->d_bounds, 3 * (K + 1) * 8, cudaMemcpyDeviceToHost, s));
        MCB_CK(cudaMemcpyAsync(ctx->h_ctr, ctx->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
        MCB_CK(cudaStreamSynchronize(s));
        launches++;
        const Counters& hc = *ctx->h_ctr;
        if (hc.active > ctx->cap_active || hc.vertices > ctx->cap_verts || hc.triangles > ctx->cap_itris ||
            hc.vertices > ctx->h_cap_v || hc.triangles > ctx->h_cap_t)
            stream_out = false; /* a device buffer has to grow first, or the host buffers are too small */
    }
    for (int j = 0; j < (stream_out ? K : 1); j++) {
        const unsigned long long cb = stream_out ? ctx->h_bounds[3 * j] : 0ull, ce = stream_out ? ctx->h_bounds[3 * j + 3] : ~0ull;
        if (stream_out && cb == ce) continue;
#define MCB_WELD_EMIT(NRM, VIEW)                                                                                              \
    MCB_LAUNCH((weld_emit_kernel<NRM>), eblocks * 2, kWeldThreads, 0, s, VIEW, B, ctx->d_ctr, ctx->cap_active, ctx->cap_verts, ctx->cap_itris, \
                                                               ctx->d_vlist, NRM ? ctx->d_vnrm : nullptr, ctx->d_tlist, cb, ce)
        if (ctx->normals == 1) { if (g.repeat) MCB_WELD_EMIT(true, WR); else MCB_WELD_EMIT(true, W); }
        else { if (g.repeat) MCB_WELD_EMIT(false, WR); else MCB_WELD_EMIT(false, W); }
#undef MCB_WELD_EMIT
        launches++;
        if (!stream_out) break;
        const unsigned long long v0 = ctx->h_bounds[3 * j + 1], v1 = ctx->h_bounds[3 * j + 4];
        const unsigned long long t0 = ctx->h_bounds[3 * j + 2], t1 = ctx->h_bounds[3 * j + 5];
        MCB_CK(cudaEventRecord(ctx->seg_ev[j], s));
        MCB_CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->seg_ev[j], 0));
        if (v1 > v0) {
            MCB_CK(cudaMemcpyAsync(ctx->h_out_v + 3 * v0, ctx->d_vlist + 3 * v0, (v1 - v0) * 12, cudaMemcpyDeviceToHost, ctx->copy_stream));
            if (ctx->normals == 1)
                MCB_CK(cudaMemcpyAsync(ctx->h_out_n + 3 * v0, ctx->d_vnrm + 3 * v0, (v1 - v0) * 12, cudaMemcpyDeviceToHost, ctx->copy_stream));
        }
        if (t1 > t0)
            MCB_CK(cudaMemcpyAsync(ctx->h_out_t + 3 * t0, ctx->d_tlist + 3 * t0, (t1 - t0) * 12, cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
    if (stream_out) {
        MCB_CK(cudaEventRecord(ctx->seg_ev[K], ctx->copy_stream));
        ctx->streamed = true;
    }
    launches += 3;
    return MCB_OK;
}

/* K5: CalculateNormal (normal.h:3-42) on the welded mesh, bit-exact */
int Run::stage_normal_h() {
    int rc;
    if ((rc = ensure_normal_h_scratch(ctx)) != MCB_OK) return rc;
    const unsigned long long* nv = &ctx->d_ctr->nh_vertices;
    MCB_LAUNCH((nh_gate_kernel), 1, 1, 0, s, ctx->d_ctr, ctx->cap_active, ctx->cap_verts, ctx->cap_itris);
    MCB_CK(cudaMemsetAsync(ctx->d_nh_count, 0, ctx->cap_verts * 4, s));
    MCB_CK(cudaMemsetAsync(ctx->d_nh_cursor, 0, ctx->cap_verts * 4, s));
    MCB_LAUNCH((nh_face_normals_kernel), eblocks * 2, 256, 0, s, ctx->d_vlist, ctx->d_tlist, ctx->d_ctr, ctx->cap_itris, ctx->d_fn, ctx->d_nh_count);
    MCB_LAUNCH((scan_block_sums_kernel), eblocks, kScanBlock, 0, s, ctx->d_nh_count, nv, ctx->d_nh_sums);
    MCB_LAUNCH((scan_sums_kernel), 1, kScanBlock, 0, s, ctx->d_nh_sums, nv);
    MCB_LAUNCH((scan_apply_kernel), eblocks, kScanBlock, 0, s, ctx->d_nh_count, ctx->d_nh_sums, nv, ctx->d_nh_start);
    MCB_LAUNCH((nh_fill_kernel), eblocks * 2, 256, 0, s, ctx->d_tlist, ctx->d_ctr, ctx->cap_itris, ctx->d_nh_start, ctx->d_nh_cursor, ctx->d_nh_adj);
    MCB_LAUNCH((nh_accumulate_kernel), eblocks * 4, 128, 0, s, ctx->d_fn, ctx->d_nh_start, ctx->d_nh_count, ctx->d_nh_adj, ctx->d_ctr, ctx->cap_verts, ctx->d_vnrm);
    launches += 7;
    return MCB_OK;
}

/* Analytic normals (mcb_set_normals 3): the surface's gradient at every soup or welded vertex, after the emitter / weld */
int Run::stage_grad_normals(bool soup) {
    const unsigned grid = (unsigned)ctx->sm_count * 8;
    if (soup)
        MCB_LAUNCH((grad_normals_kernel<true>), grid, 256, 0, s, eq.point, g.sx, g.sy, g.sz, ctx->d_ctr, ctx->cap_tris,
                   (const float*)ctx->d_pos, (float*)ctx->d_nrm);
    else
        MCB_LAUNCH((grad_normals_kernel<false>), grid, 256, 0, s, eq.point, g.sx, g.sy, g.sz, ctx->d_ctr, ctx->cap_verts,
                   ctx->d_vlist, ctx->d_vnrm);
    launches++;
    return MCB_OK;
}

} /* namespace */

extern "C" {

int mcb_polygonise(mcb_ctx* ctx, mcb_counts* out) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->eq[0].valid) return fail(ctx, MCB_E_STATE, "no surface equation");
    if ((rc = setup_grid(ctx)) != MCB_OK) return rc;
    Grid& g = ctx->g;
    g.sx = ctx->scale[0]; g.sy = ctx->scale[1]; g.sz = ctx->scale[2];
    g.iso = ctx->iso;
    g.repeat = ctx->repeat_on ? 1 : 0;
    g.rstep = ctx->repeat_step;
    if (ctx->repeat_on && ctx->seed_on) return fail(ctx, MCB_E_STATE, "repeating-surface mode and seed mode cannot be combined");
    if (ctx->seed_on && ctx->nccl_comm && ctx->comm_nranks > 1)
        return fail(ctx, MCB_E_STATE, "seed mode follows one component through the whole grid: it cannot be combined with z-slabs over several GPUs");
    if (ctx->normals == 2 && !(ctx->mesh_mode & MCB_MESH_INDEXED))
        return fail(ctx, MCB_E_STATE, "normal.h normals (mode 2) are defined on the welded mesh: request MCB_MESH_INDEXED");

    Run run{ctx, g, ctx->eq[0], ctx->stream, false, (ctx->mesh_mode & MCB_MESH_SOUP) != 0, (ctx->mesh_mode & MCB_MESH_INDEXED) != 0,
            nullptr, ClsGeom{}, 0u, (unsigned)ctx->sm_count * 4, 0u};
    for (int i = 0; i < 3; i++) run.any_constraint |= ctx->cons[i].in_use && ctx->eq[i + 1].valid;
    if ((rc = run.prepare_buffers()) != MCB_OK) return rc;
    run.dV = run.any_constraint ? ctx->d_V : nullptr;
    run.cg = classify_geometry(ctx, g, &run.tiles);
    cudaStream_t s = ctx->stream;
    uint32_t reruns = 0;

    /* Where the field lives.  Dense: every vertex (the mcb_get_field hook, per-cube iso levels).  Otherwise the
     * block-field mode: interval proof per 32 x 4 x 4 vertex block, evaluation of the undecided blocks only — decided
     * from this call's own data, so a first or changed configuration is as fast as a repeated one. */
    const bool blocks = ctx->field_mode != MCB_FIELD_DENSE && !g.repeat;
    const bool timing = ctx->stage_timing;
    MCB_CK(cudaMemsetAsync(ctx->d_ctr, 0, sizeof(Counters), s));
    if (timing) MCB_CK(cudaEventRecord(ctx->ev[0], s));
    if ((rc = run.stage_tables()) != MCB_OK) return rc;
    if (timing) MCB_CK(cudaEventRecord(ctx->ev[1], s));
    if ((rc = blocks ? run.stage_eval_blocks() : run.stage_eval()) != MCB_OK) return rc;
    if (timing) MCB_CK(cudaEventRecord(ctx->ev[2], s));
    MCB_CK(cudaGetLastError());

    bool need_classify = true;
    for (;;) { /* repeated only when an output buffer had to grow (mcb_counts::reruns) */
        if (need_classify) {
            if ((rc = run.stage_classify()) != MCB_OK) return rc;
            /* several GPUs: this slab's triangle count is final now (tile_scan_kernel) — its all-gather is enqueued here, on
             * the side stream, so that NCCL's launch cost hides behind the emission instead of following the call.  Once
             * per call: a repeated pass (buffer growth) must not add a collective the other ranks do not have */
            if (ctx->comm_auto && ctx->nccl_comm && reruns == 0 && (rc = comm_enqueue(ctx)) != MCB_OK) return rc;
            if (timing) MCB_CK(cudaEventRecord(ctx->ev[6], s));
            if (ctx->field_is_sparse && (rc = run.stage_fill()) != MCB_OK) return rc;
            if (timing) MCB_CK(cudaEventRecord(ctx->ev[7], s));
            if (ctx->seed_on && (rc = run.stage_seed()) != MCB_OK) return rc;
            if (timing) MCB_CK(cudaEventRecord(ctx->ev[3], s));
        }
        if (run.want_soup && (rc = run.stage_soup()) != MCB_OK) return rc;
        if (run.want_soup && ctx->normals == 3 && (rc = run.stage_grad_normals(true)) != MCB_OK) return rc;
        if (timing) MCB_CK(cudaEventRecord(ctx->ev[4], s));
        if (run.want_indexed) {
            if ((rc = run.stage_weld()) != MCB_OK) return rc;
            if (ctx->normals == 2 && (rc = run.stage_normal_h()) != MCB_OK) return rc;
            if (ctx->normals == 3 && (rc = run.stage_grad_normals(false)) != MCB_OK) return rc;
        }
        if (timing) MCB_CK(cudaEventRecord(ctx->ev[5], s));
        if (run.want_indexed && ctx->streamed) MCB_CK(cudaStreamWaitEvent(s, ctx->seg_ev[8], 0)); /* return when the mesh is on the host */
        MCB_CK(cudaMemcpyAsync(ctx->h_ctr, ctx->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
        MCB_CK(cudaStreamSynchronize(s));
        MCB_CK(cudaGetLastError());
        if (ctx->h_ctr->error == 2 || ctx->h_ctr->triangles >= (1ull << 31))
            return fail(ctx, MCB_E_CAPACITY, "2^31 or more triangles in one slab: split the grid into more z-slabs");
        const unsigned long long needA = ctx->h_ctr->active, needT = ctx->h_ctr->triangles, needV = ctx->h_ctr->vertices;
        bool again = false;
        need_classify = false;
        if (needA > ctx->cap_active) {
            if ((rc = ensure_records(ctx, needA + needA / 8 + 1024)) != MCB_OK) return rc;
            need_classify = true;
            again = true;
        }
        if (ctx->h_ctr->amb_n > ctx->cap_amb) { /* more ambiguous cubes than the face-test list holds: counts are provisional */
            const uint32_t want = ctx->h_ctr->amb_n + ctx->h_ctr->amb_n / 8 + 1024;
            cudaFree(ctx->d_amb);
            ctx->d_amb = nullptr; ctx->cap_amb = 0;
            MCB_CK(cudaMalloc((void**)&ctx->d_amb, (size_t)want * 16));
            ctx->cap_amb = want;
            need_classify = true;
            again = true;
        }
        if (run.want_soup && needT > ctx->cap_tris) {
            if ((rc = ensure_soup(ctx, needT + needT / 8 + 1024, ctx->normals != 0)) != MCB_OK) return rc;
            again = true;
        }
        if (run.want_indexed && (needT > ctx->cap_itris || needV > ctx->cap_verts || need_classify)) {
            /* with truncated records the vertex count is a lower bound: size generously, the re-run settles it */
            const unsigned long long v = std::max(needV + needV / 8 + 1024, need_classify ? needA + needA / 4 : 0ull);
            if ((rc = ensure_indexed(ctx, v, needT + needT / 8 + 1024, ctx->normals != 0)) != MCB_OK) return rc;
            again = true;
        }
        if (!again) break;
        reruns++;
        if (reruns > 6) return fail(ctx, MCB_E_CAPACITY, "output buffers did not settle");
    }

    mcb_counts& c = ctx->last;
    std::memset(&c, 0, sizeof c);
    c.cubes = (uint64_t)(g.ke - g.kb) * g.M * g.M;
    c.active = ctx->h_ctr->active;
    c.triangles = ctx->h_ctr->triangles;
    c.ambiguous = ctx->h_ctr->ambiguous;
    c.redirected = ctx->h_ctr->redirected;
    c.M = g.M; c.k_begin = g.kb; c.k_end = g.ke;
    if (timing) {
        cudaEventElapsedTime(&c.ms_tables, ctx->ev[0], ctx->ev[1]);
        cudaEventElapsedTime(&c.ms_eval, ctx->ev[1], ctx->ev[2]);
        cudaEventElapsedTime(&c.ms_classify, ctx->ev[2], ctx->ev[3]);
        cudaEventElapsedTime(&c.ms_fill, ctx->ev[6], ctx->ev[7]);
        c.ms_classify -= c.ms_fill;
        cudaEventElapsedTime(&c.ms_emit, ctx->ev[3], ctx->ev[4]);
        cudaEventElapsedTime(&c.ms_weld, ctx->ev[4], ctx->ev[5]);
        cudaEventElapsedTime(&c.ms_total, ctx->ev[0], ctx->ev[5]);
    }
    c.field_mode = ctx->field_is_sparse ? MCB_FIELD_SPARSE : MCB_FIELD_DENSE;
    c.field_blocks = ctx->field_is_sparse ? (uint64_t)ctx->h_ctr->field_blocks + ctx->h_ctr->eval_blocks : 0;
    c.jit = ctx->jit_used ? 1u : 0u;
    c.ms_compile = ctx->jit_used ? ctx->ms_compile : 0.f; /* compile time of the module this call adopted (or mcb_jit_wait before it) */
    if (ctx->jit_used) ctx->ms_compile = 0.f;
    if (run.want_indexed) ctx->index_base_applied = 0; /* weld_emit has just rewritten tri_list from zero */
    c.vertices = run.want_indexed ? ctx->h_ctr->vertices : 0;
    c.mesh_mode = (uint32_t)ctx->mesh_mode;
    c.launches = run.launches;
    c.reruns = reruns;
    ctx->have_result = true;
    if (out) *out = c;
    return MCB_OK;
}

int mcb_get_mesh(mcb_ctx* ctx, float* pos4, float* nrm4, uint64_t cap_triangles) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    if (!(ctx->last.mesh_mode & MCB_MESH_SOUP)) return fail(ctx, MCB_E_STATE, "the triangle soup was not requested (mcb_set_mesh_mode)");
    const uint64_t T = ctx->last.triangles;
    if (T > cap_triangles) return fail(ctx, MCB_E_CAPACITY, "mesh buffer too small");
    if (nrm4 && ctx->normals != 1 && ctx->normals != 3) return fail(ctx, MCB_E_STATE, "soup normals need mcb_set_normals(ctx, 1) or 3");
    if (T == 0) return MCB_OK;
    if (pos4) MCB_CK(cudaMemcpyAsync(pos4, ctx->d_pos, T * 3 * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    if (nrm4) MCB_CK(cudaMemcpyAsync(nrm4, ctx->d_nrm, T * 3 * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    return MCB_OK;
}

int mcb_set_stage_timing(mcb_ctx* ctx, int enabled) {
    if (!ctx) return MCB_E_ARG;
    ctx->stage_timing = enabled != 0;
    return MCB_OK;
}

int mcb_set_field_mode(mcb_ctx* ctx, int mode) {
    if (!ctx || mode < MCB_FIELD_DENSE || mode > MCB_FIELD_AUTO) return MCB_E_ARG;
    ctx->field_mode = mode;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_jit(mcb_ctx* ctx, int enabled) {
    if (!ctx || enabled < MCB_JIT_OFF || enabled > MCB_JIT_AUTO) return MCB_E_ARG;
    ctx->jit = enabled;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_jit_wait(mcb_ctx* ctx) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->eq[0].valid) return fail(ctx, MCB_E_STATE, "no surface equation");
    if (!jit_wanted(ctx, ctx->eq[0])) return 0;
    const mcb_ctx::JitKernel* jk = nullptr;
    rc = jit_module(ctx, ctx->eq[0], &jk, true);
    if (rc == MCB_OK) return 1;
    if (ctx->jit == MCB_JIT_ON) return rc;
    ctx->jit_note = ctx->err;
    return 0;
}

int mcb_jit_check(const char* equation, char* log, size_t cap) { return mcb_jit_check_grammar(equation, MCB_GRAMMAR_REFERENCE, log, cap); }

int mcb_jit_check_grammar(const char* equation, int grammar, char* log, size_t cap) {
    if (grammar != MCB_GRAMMAR_REFERENCE && grammar != MCB_GRAMMAR_FUNCTIONS) return MCB_E_ARG;
    mcb::Compiled c;
    int rc = mcb::compile(equation ? equation : "", c, nullptr, grammar);
    if (rc != MCB_OK) return rc;
    std::string err;
    bool has_pow = false;
    const std::string src = mcbjit::generate(c.grid_fused.data(), (int)c.grid_fused.size(), &has_pow, &err);
    if (src.empty()) { copy_text(err, log, cap); return MCB_E_STATE; }
    std::vector<char> cubin;
    err = mcbjit::compile(src, has_pow, (int)sizeof(Grid), &cubin);
    if (!err.empty()) { copy_text(err, log, cap); return MCB_E_STATE; }
    copy_text(src, log, cap); /* best effort: a short buffer just truncates the listing */
    return (int)cubin.size();
}

int mcb_set_mesh_mode(mcb_ctx* ctx, int mode) {
    if (!ctx || mode < 1 || mode > 3) return MCB_E_ARG;
    ctx->mesh_mode = mode;
    ctx->have_result = false;
    return MCB_OK;
}

int mcb_set_host_output(mcb_ctx* ctx, float* vertex_list, uint32_t* tri_list, float* normals, uint64_t cap_vertices, uint64_t cap_triangles) {
    if (!ctx) return MCB_E_ARG;
    ctx->h_out_v = vertex_list; ctx->h_out_t = tri_list; ctx->h_out_n = normals;
    ctx->h_cap_v = vertex_list ? cap_vertices : 0; ctx->h_cap_t = tri_list ? cap_triangles : 0;
    ctx->streamed = false;
    return MCB_OK;
}

int mcb_host_output_filled(const mcb_ctx* ctx) { return ctx && ctx->streamed ? 1 : 0; }

int mcb_get_indexed_mesh(mcb_ctx* ctx, float* vertex_list, uint32_t* tri_list, float* normals, uint64_t cap_vertices,
                         uint64_t cap_triangles) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    if (!(ctx->last.mesh_mode & MCB_MESH_INDEXED)) return fail(ctx, MCB_E_STATE, "the indexed mesh was not requested (mcb_set_mesh_mode)");
    const uint64_t Vn = ctx->last.vertices, T = ctx->last.triangles;
    if ((vertex_list || normals) && Vn > cap_vertices) return fail(ctx, MCB_E_CAPACITY, "vertex buffer too small");
    if (tri_list && T > cap_triangles) return fail(ctx, MCB_E_CAPACITY, "triangle buffer too small");
    if (normals && !ctx->normals) return fail(ctx, MCB_E_STATE, "normals are switched off");
    if (vertex_list && Vn) MCB_CK(cudaMemcpyAsync(vertex_list, ctx->d_vlist, Vn * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (normals && Vn) MCB_CK(cudaMemcpyAsync(normals, ctx->d_vnrm, Vn * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (tri_list && T) {
        if (ctx->index_base != ctx->index_base_applied) { /* the slab's indices moved to their place in the assembled mesh, on the device */
            MCB_LAUNCH((add_index_base_kernel), (unsigned)ctx->sm_count * 8, 256, 0, ctx->stream, ctx->d_tlist, (unsigned long long)T * 3ull,
                       ctx->index_base - ctx->index_base_applied);
            ctx->index_base_applied = ctx->index_base;
        }
        MCB_CK(cudaMemcpyAsync(tri_list, ctx->d_tlist, T * 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    return MCB_OK;
}

int mcb_set_index_base(mcb_ctx* ctx, uint32_t base) {
    if (!ctx) return MCB_E_ARG;
    ctx->index_base = base;
    return MCB_OK;
}

int mcb_get_indexed_mesh_device(mcb_ctx* ctx, const float** vertex_list, const uint32_t** tri_list, const float** normals) {
    if (!ctx) return MCB_E_ARG;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    if (!(ctx->last.mesh_mode & MCB_MESH_INDEXED)) return fail(ctx, MCB_E_STATE, "the indexed mesh was not requested (mcb_set_mesh_mode)");
    if (vertex_list) *vertex_list = ctx->d_vlist;
    if (tri_list) *tri_list = ctx->d_tlist;
    if (normals) *normals = ctx->normals ? ctx->d_vnrm : nullptr;
    return MCB_OK;
}

int mcb_counts_device(mcb_ctx* ctx, const uint64_t** counts) {
    if (!ctx || !counts) return MCB_E_ARG;
    *counts = reinterpret_cast<const uint64_t*>(ctx->d_ctr);
    return MCB_OK;
}

int mcb_get_mesh_device(mcb_ctx* ctx, const float** pos4, const float** nrm4) {
    if (!ctx) return MCB_E_ARG;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    if (pos4) *pos4 = (const float*)ctx->d_pos;
    if (nrm4) *nrm4 = ctx->normals == 1 || ctx->normals == 3 ? (const float*)ctx->d_nrm : nullptr;
    return MCB_OK;
}

int mcb_get_cases(mcb_ctx* ctx, uint8_t* cube_code, uint8_t* table_idx) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    const Grid& g = ctx->g;
    const long long n = (long long)ctx->last.cubes;
    bool any_constraint = false;
    for (int i = 0; i < 3; i++) any_constraint |= ctx->cons[i].in_use && ctx->eq[i + 1].valid;
    if (ctx->field_is_sparse) { /* block-field mode: only the decided blocks next to the surface carry their sign words so far */
        const unsigned nblocks = (unsigned)ctx->bd.nbx * (unsigned)ctx->bd.nby * (unsigned)ctx->bd.nbz;
        MCB_LAUNCH((decided_signs_all_kernel), (nblocks + 255) / 256, 256, 0, ctx->stream, g, ctx->bd, ctx->d_bcls, ctx->d_scls, ctx->d_S);
    }
    uint8_t *d_code = nullptr, *d_tidx = nullptr;
    MCB_CK(cudaMalloc((void**)&d_code, (size_t)n));
    if (cudaMalloc((void**)&d_tidx, (size_t)n) != cudaSuccess) { cudaFree(d_code); return fail(ctx, MCB_E_NOMEM, "cudaMalloc"); }
    MCB_LAUNCH((dense_codes_kernel), (unsigned)((n + 255) / 256), 256, 0, ctx->stream, g, ctx->d_S, any_constraint ? ctx->d_V : nullptr, d_code, d_tidx, n,
                                                                             g.repeat ? ctx->d_cw : nullptr, (uint32_t)((g.M + 31) / 32));
    if (ctx->last.active)
        MCB_LAUNCH((scatter_tidx_kernel), (unsigned)((ctx->last.active + 255) / 256), 256, 0, ctx->stream, g, ctx->d_rec, ctx->last.active, d_tidx);
    if (cube_code) cudaMemcpyAsync(cube_code, d_code, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    if (table_idx) cudaMemcpyAsync(table_idx, d_tidx, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    cudaError_t e2 = cudaGetLastError();
    cudaFree(d_code); cudaFree(d_tidx);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, MCB_E_CUDA, std::string("get_cases: ") + cudaGetErrorString(e != cudaSuccess ? e : e2));
    return MCB_OK;
}

int mcb_get_field(mcb_ctx* ctx, float* out) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    if (!out) return fail(ctx, MCB_E_ARG, "null buffer");
    if (ctx->field_is_sparse) return fail(ctx, MCB_E_STATE, "the field is not materialised in sparse-field mode (mcb_set_field_mode)");
    const Grid& g = ctx->g;
    const size_t n1 = (size_t)g.M + 1;
    cudaMemcpy3DParms p = {};
    p.srcPtr = make_cudaPitchedPtr(ctx->d_F, (size_t)g.P * sizeof(float), (size_t)g.P, (size_t)g.NV);
    p.srcPos = make_cudaPos(sizeof(float), 1, 1);
    p.dstPtr = make_cudaPitchedPtr(out, n1 * sizeof(float), n1, n1);
    p.dstPos = make_cudaPos(0, 0, 0);
    p.extent = make_cudaExtent(n1 * sizeof(float), n1, (size_t)(g.ke - g.kb) + 1);
    p.kind = cudaMemcpyDeviceToHost;
    MCB_CK(cudaMemcpy3DAsync(&p, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    return MCB_OK;
}

int mcb_get_active(mcb_ctx* ctx, uint64_t* records, uint32_t* tri_offsets, uint64_t cap) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    const uint64_t A = ctx->last.active;
    if (A > cap) return fail(ctx, MCB_E_CAPACITY, "record buffer too small");
    if (A == 0) return MCB_OK;
    if (records) MCB_CK(cudaMemcpyAsync(records, ctx->d_rec, A * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (tri_offsets) MCB_CK(cudaMemcpyAsync(tri_offsets, ctx->d_trioff, A * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    return MCB_OK;
}

} /* extern "C" */

/* ---- z-slabs over several GPUs --------------------------------------------------------------------------------- */
namespace {

/* libnccl.so.2, loaded on first use (in a torchrun process this is the copy torch already mapped) */
struct NcclId { char internal[128]; };
struct Nccl {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string error;
};
constexpr int kNcclUint32 = 3, kNcclUint64 = 5, kNcclSum = 0; /* ncclDataType_t / ncclRedOp_t values (nccl.h) */

Nccl& nccl() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            n.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (n.lib) break;
        }
        if (!n.lib) { n.error = "libnccl.so.2 not found: the multi-GPU exchange is unavailable"; return; }
#define MCB_SYM(field, sym)                                                \
    n.field = reinterpret_cast<decltype(n.field)>(dlsym(n.lib, sym));      \
    if (!n.field) n.error = std::string("libnccl lacks ") + sym;
        MCB_SYM(GetUniqueId, "ncclGetUniqueId")
        MCB_SYM(CommInitRank, "ncclCommInitRank")
        MCB_SYM(CommDestroy, "ncclCommDestroy")
        MCB_SYM(AllGather, "ncclAllGather")
        MCB_SYM(AllReduce, "ncclAllReduce")
        MCB_SYM(GetErrorString, "ncclGetErrorString")
#undef MCB_SYM
    });
    return n;
}

#define MCB_NCCL(call)                                                                                                  \
    do {                                                                                                                \
        const int r_ = (call);                                                                                          \
        if (r_ != 0) return fail(ctx, MCB_E_CUDA, std::string(#call) + ": " + nccl().GetErrorString(r_));                \
    } while (0)

/* slabs of (nearly) equal cost: cuts[r] = first layer of rank r, at least one layer each */
void cut_by_cost(int M, int nranks, const double* cost, int* cuts) {
    double total = 0;
    for (int k = 0; k < M; k++) total += cost[k];
    cuts[0] = 0;
    double run = 0;
    int k = 0;
    for (int r = 1; r < nranks; r++) {
        const double want = total * (double)r / (double)nranks;
        /* take layers while that brings the prefix closer to the target */
        while (k < M && run + 0.5 * cost[k] <= want) { run += cost[k]; k++; }
        int c = std::max(k, cuts[r - 1] + 1);            /* at least one layer per slab ... */
        c = std::min(c, M - (nranks - r));               /* ... for the ranks still to come as well */
        while (k < c) { run += cost[k]; k++; }
        cuts[r] = c;
    }
    cuts[nranks] = M;
}

/* all-gather of this slab's triangle count, straight from the device counters, on the side stream */
int comm_enqueue(mcb_ctx* ctx) {
    /* the next polygonisation resets the live counters: the count is first copied aside, in stream order */
    unsigned long long* stg = ctx->d_comm + ctx->comm_flip;
    ctx->comm_flip ^= 1;
    MCB_CK(cudaMemcpyAsync(stg, &ctx->d_ctr->triangles, 8, cudaMemcpyDeviceToDevice, ctx->stream));
    MCB_CK(cudaEventRecord(ctx->comm_ready, ctx->stream));
    MCB_CK(cudaStreamWaitEvent(ctx->comm_stream, ctx->comm_ready, 0));
    MCB_NCCL(nccl().AllGather(stg, ctx->d_comm + 2, 1, kNcclUint64, ctx->nccl_comm, ctx->comm_stream));
    MCB_CK(cudaMemcpyAsync(ctx->h_comm, ctx->d_comm + 2, (size_t)ctx->comm_nranks * 8, cudaMemcpyDeviceToHost, ctx->comm_stream));
    MCB_CK(cudaEventRecord(ctx->comm_done, ctx->comm_stream));
    ctx->comm_pending = true;
    return MCB_OK;
}

} /* namespace */

extern "C" {

int mcb_balance_slabs(int M, int nranks, const uint32_t* tri, double fixed, int* cuts) {
    if (M <= 0 || nranks <= 0 || nranks > M || !tri || !cuts) return MCB_E_ARG;
    if (fixed < 0) fixed = 0.0015 * (double)M * (double)M;
    std::vector<double> cost((size_t)M);
    for (int k = 0; k < M; k++) cost[(size_t)k] = (double)tri[k] + fixed;
    cut_by_cost(M, nranks, cost.data(), cuts);
    return MCB_OK;
}

int mcb_rebalance_slabs(int M, int nranks, double* cost, int* cuts, const double* ms) {
    if (M <= 0 || nranks <= 0 || nranks > M || !cost || !cuts || !ms || cuts[0] != 0 || cuts[nranks] != M) return MCB_E_ARG;
    for (int r = 0; r < nranks; r++)
        if (!(ms[r] > 0.0) || cuts[r] >= cuts[r + 1]) return MCB_E_ARG;
    /* the time a slab took is spread over its layers in proportion to their modelled cost; then the same cut as before.
     * Equal times are the fixed point; what does not move with the layers (launch latencies) makes each pass undershoot a
     * little instead of overshooting */
    for (int r = 0; r < nranks; r++) {
        double sum = 0;
        for (int k = cuts[r]; k < cuts[r + 1]; k++) sum += cost[k];
        const double scale = sum > 0 ? ms[r] / sum : 1.0;
        for (int k = cuts[r]; k < cuts[r + 1]; k++) cost[k] = sum > 0 ? cost[k] * scale : ms[r] / (double)(cuts[r + 1] - cuts[r]);
    }
    cut_by_cost(M, nranks, cost, cuts);
    return MCB_OK;
}

int mcb_layer_triangles(mcb_ctx* ctx, uint32_t* per_layer) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change");
    if (!per_layer) return fail(ctx, MCB_E_ARG, "null buffer");
    const size_t M = (size_t)ctx->g.M;
    if ((rc = ensure(ctx, &ctx->d_layer_hist, &ctx->cap_layer_hist, M)) != MCB_OK) return rc;
    MCB_CK(cudaMemsetAsync(ctx->d_layer_hist, 0, M * 4, ctx->stream));
    MCB_LAUNCH((layer_hist_kernel), (unsigned)ctx->sm_count * 4, 256, 0, ctx->stream, ctx->d_rec, ctx->d_trioff, ctx->d_ctr, ctx->cap_active, ctx->d_layer_hist);
    MCB_CK(cudaMemcpyAsync(per_layer, ctx->d_layer_hist + ctx->g.kb, (size_t)(ctx->g.ke - ctx->g.kb) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    MCB_CK(cudaGetLastError());
    return MCB_OK;
}

int mcb_comm_unique_id(void* id128) {
    if (!id128) return MCB_E_ARG;
    Nccl& N = nccl();
    if (!N.error.empty()) return MCB_E_STATE;
    NcclId id;
    if (N.GetUniqueId(&id) != 0) return MCB_E_CUDA;
    std::memcpy(id128, &id, sizeof id);
    return MCB_OK;
}

int mcb_comm_finalize(mcb_ctx* ctx) {
    if (!ctx) return MCB_E_ARG;
    if (ctx->nccl_comm) {
        cudaSetDevice(ctx->device);
        if (ctx->comm_stream) cudaStreamSynchronize(ctx->comm_stream);
        nccl().CommDestroy(ctx->nccl_comm);
        ctx->nccl_comm = nullptr;
    }
    if (ctx->comm_stream) { cudaStreamDestroy(ctx->comm_stream); ctx->comm_stream = nullptr; }
    if (ctx->comm_ready) { cudaEventDestroy(ctx->comm_ready); ctx->comm_ready = nullptr; }
    if (ctx->comm_done) { cudaEventDestroy(ctx->comm_done); ctx->comm_done = nullptr; }
    cudaFree(ctx->d_comm); ctx->d_comm = nullptr;
    if (ctx->h_comm) { cudaFreeHost(ctx->h_comm); ctx->h_comm = nullptr; }
    ctx->comm_nranks = 1; ctx->comm_rank = 0; ctx->comm_pending = false;
    return MCB_OK;
}

int mcb_comm_init(mcb_ctx* ctx, const void* id128, int rank, int nranks) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, MCB_E_ARG, "rank / nranks out of range");
    Nccl& N = nccl();
    if (!N.error.empty()) return fail(ctx, MCB_E_STATE, N.error);
    mcb_comm_finalize(ctx);
    NcclId id;
    std::memcpy(&id, id128, sizeof id);
    MCB_NCCL(N.CommInitRank(&ctx->nccl_comm, nranks, id, rank));
    ctx->comm_rank = rank; ctx->comm_nranks = nranks;
    MCB_CK(cudaStreamCreateWithFlags(&ctx->comm_stream, cudaStreamNonBlocking));
    MCB_CK(cudaEventCreateWithFlags(&ctx->comm_ready, cudaEventDisableTiming));
    MCB_CK(cudaEventCreateWithFlags(&ctx->comm_done, cudaEventDisableTiming));
    MCB_CK(cudaMalloc((void**)&ctx->d_comm, (size_t)(2 + nranks) * 8));
    MCB_CK(cudaMallocHost((void**)&ctx->h_comm, (size_t)nranks * 8));
    int k0, k1;
    if ((rc = mcb_slab_range(ctx->M, rank, nranks, &k0, &k1)) != MCB_OK) return fail(ctx, rc, "fewer cube layers than ranks");
    return mcb_set_slab(ctx, k0, k1);
}

int mcb_comm_exchange(mcb_ctx* ctx) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->nccl_comm) return fail(ctx, MCB_E_STATE, "mcb_comm_init has not been called");
    if (ctx->comm_auto) return MCB_OK; /* mcb_polygonise has enqueued it already */
    return comm_enqueue(ctx);
}

int mcb_comm_set_auto(mcb_ctx* ctx, int enabled) {
    if (!ctx) return MCB_E_ARG;
    ctx->comm_auto = enabled != 0;
    return MCB_OK;
}

int mcb_comm_offsets(mcb_ctx* ctx, uint64_t* offset, uint64_t* total, uint64_t* per_rank) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->nccl_comm || !ctx->comm_pending) return fail(ctx, MCB_E_STATE, "no exchange to wait for");
    MCB_CK(cudaEventSynchronize(ctx->comm_done));
    uint64_t off = 0, tot = 0;
    for (int r = 0; r < ctx->comm_nranks; r++) {
        if (r < ctx->comm_rank) off += ctx->h_comm[r];
        tot += ctx->h_comm[r];
        if (per_rank) per_rank[r] = ctx->h_comm[r];
    }
    if (offset) *offset = off;
    if (total) *total = tot;
    return MCB_OK;
}

int mcb_comm_balance(mcb_ctx* ctx, double fixed_cost_per_layer, int* k_begin, int* k_end) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->nccl_comm) return fail(ctx, MCB_E_STATE, "mcb_comm_init has not been called");
    if (!ctx->have_result) return fail(ctx, MCB_E_STATE, "mcb_polygonise has not run since the last change: nothing to balance by");
    const size_t M = (size_t)ctx->g.M;
    if ((rc = ensure(ctx, &ctx->d_layer_hist, &ctx->cap_layer_hist, M)) != MCB_OK) return rc;
    MCB_CK(cudaMemsetAsync(ctx->d_layer_hist, 0, M * 4, ctx->stream));
    MCB_LAUNCH((layer_hist_kernel), (unsigned)ctx->sm_count * 4, 256, 0, ctx->stream, ctx->d_rec, ctx->d_trioff, ctx->d_ctr, ctx->cap_active, ctx->d_layer_hist);
    /* one collective at a time per communicator: an all-gather still in flight on the side stream goes first */
    if (ctx->comm_pending) MCB_CK(cudaStreamWaitEvent(ctx->stream, ctx->comm_done, 0));
    /* every rank's layers are disjoint: the sum over ranks is the whole grid's histogram */
    MCB_NCCL(nccl().AllReduce(ctx->d_layer_hist, ctx->d_layer_hist, M, kNcclUint32, kNcclSum, ctx->nccl_comm, ctx->stream));
    std::vector<uint32_t> hist(M);
    MCB_CK(cudaMemcpyAsync(hist.data(), ctx->d_layer_hist, M * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->comm_nranks > (int)M) return fail(ctx, MCB_E_ARG, "fewer cube layers than ranks");
    /* what a layer costs besides its triangles: the dense field writes every vertex of it, the block-field mode only looks
     * at its block classes and candidate words (fitted on 2048^3 slabs: ~1.5e-4 M^2 triangle-equivalents) */
    if (fixed_cost_per_layer < 0) fixed_cost_per_layer = (ctx->field_is_sparse ? 0.00015 : 0.0015) * (double)M * (double)M;
    ctx->layer_cost.resize(M);
    for (size_t k = 0; k < M; k++) ctx->layer_cost[k] = (double)hist[k] + fixed_cost_per_layer;
    std::vector<int>& cuts = ctx->comm_cuts;
    cuts.assign((size_t)ctx->comm_nranks + 1, 0);
    cut_by_cost((int)M, ctx->comm_nranks, ctx->layer_cost.data(), cuts.data());
    const int k0 = cuts[(size_t)ctx->comm_rank], k1 = cuts[(size_t)ctx->comm_rank + 1];
    if (k_begin) *k_begin = k0;
    if (k_end) *k_end = k1;
    return mcb_set_slab(ctx, k0, k1);
}

int mcb_comm_rebalance(mcb_ctx* ctx, double ms_measured, int* k_begin, int* k_end) {
    int rc = enter(ctx);
    if (rc != MCB_OK) return rc;
    if (!ctx->nccl_comm) return fail(ctx, MCB_E_STATE, "mcb_comm_init has not been called");
    const size_t M = (size_t)ctx->M;
    const int n = ctx->comm_nranks;
    if (ctx->layer_cost.size() != M || (int)ctx->comm_cuts.size() != n + 1 || ctx->comm_cuts[(size_t)ctx->comm_rank] != ctx->kb ||
        ctx->comm_cuts[(size_t)ctx->comm_rank + 1] != ctx->ke)
        return fail(ctx, MCB_E_STATE, "mcb_comm_balance has not cut the current slabs");
    if (!(ms_measured > 0.0)) return fail(ctx, MCB_E_ARG, "the measured time must be positive");
    /* every rank's time, as the bits of a double, through the count exchange's buffers */
    unsigned long long bits;
    std::memcpy(&bits, &ms_measured, 8);
    if (ctx->comm_pending) MCB_CK(cudaStreamWaitEvent(ctx->stream, ctx->comm_done, 0));
    MCB_CK(cudaMemcpyAsync(ctx->d_comm, &bits, 8, cudaMemcpyHostToDevice, ctx->stream));
    MCB_NCCL(nccl().AllGather(ctx->d_comm, ctx->d_comm + 2, 1, kNcclUint64, ctx->nccl_comm, ctx->stream));
    std::vector<unsigned long long> all((size_t)n);
    MCB_CK(cudaMemcpyAsync(all.data(), ctx->d_comm + 2, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MCB_CK(cudaStreamSynchronize(ctx->stream));
    std::vector<double> ms((size_t)n);
    std::memcpy(ms.data(), all.data(), (size_t)n * 8);
    if ((rc = mcb_rebalance_slabs((int)M, n, ctx->layer_cost.data(), ctx->comm_cuts.data(), ms.data())) != MCB_OK) return fail(ctx, rc, "a rank reported no time");
    const int k0 = ctx->comm_cuts[(size_t)ctx->comm_rank], k1 = ctx->comm_cuts[(size_t)ctx->comm_rank + 1];
    if (k_begin) *k_begin = k0;
    if (k_end) *k_end = k1;
    return mcb_set_slab(ctx, k0, k1);
}

int mcb_host_register(void* ptr, size_t bytes) {
    if (!ptr || !bytes) return MCB_E_ARG;
    return cudaHostRegister(ptr, bytes, cudaHostRegisterPortable) == cudaSuccess ? MCB_OK : MCB_E_CUDA;
}

int mcb_host_unregister(void* ptr) {
    if (!ptr) return MCB_E_ARG;
    return cudaHostUnregister(ptr) == cudaSuccess ? MCB_OK : MCB_E_CUDA;
}

} /* extern "C" */

