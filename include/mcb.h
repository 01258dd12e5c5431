/* mcb.h — C ABI of the B200-native marching-cubes polygoniser (libmcb200.so).
 *
 * This is the drop-in boundary for the one hot path of raineyeh/Marching-Cube-for-Implicit-Surfaces:
 *     equation -> field on the grid -> cube classification (+ambiguity) -> scan/compaction -> triangles (+normals)
 * The reference has no plugin/FFI interface; its boundary is two C++ headers (Source/evaluator.h, Source/marching.h)
 * consumed by main.cpp:11-20 and drawer.cpp:785-942.  include/evaluator.h and include/marching.h in this repository
 * keep those class names and public signatures and forward to the functions below; any other host language binds
 * the same symbols (INTEGRATION.md shows the stubs).  Plain pointers and sizes only: no C++ or torch types cross
 * this boundary, no exception does either.  Every function returns MCB_OK (0) or a negative mcb_status.
 *
 * There is no CPU implementation behind this ABI: every function that computes field values, cases or triangles
 * runs CUDA kernels on the context's device and fails with MCB_E_NODEVICE / MCB_E_CUDA when it cannot.
 * The only host-side work is what the reference also does once per equation (tokenising) plus the lowering of the
 * token list to bytecode.
 *
 * Threading: a context may be used from any one thread at a time (the reference calls recalculate() from the GLUT
 * thread and from its "movie" std::thread, drawer.cpp:135); each call makes the context's device current.
 */
#ifndef MCB_H
#define MCB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCB_ABI_VERSION 4

typedef enum {
    MCB_OK = 0,
    MCB_E_PARSE = -1,    /* equation rejected (Evaluator::set_equation returning false, evaluator.cpp:15-17) */
    MCB_E_ARG = -2,      /* argument out of range (the reference's `return false` paths, e.g. marching.cpp:226-238) */
    MCB_E_CUDA = -3,     /* a CUDA call or kernel failed; mcb_last_error() has the text */
    MCB_E_NOMEM = -4,    /* device or host allocation failed */
    MCB_E_STATE = -5,    /* call order: e.g. mcb_get_mesh before mcb_polygonise */
    MCB_E_CAPACITY = -6, /* equation too large for the bytecode limits, or caller buffer too small */
    MCB_E_NODEVICE = -7  /* no usable CUDA device: there is no CPU fallback */
} mcb_status;

typedef struct mcb_ctx mcb_ctx;

/* Result of one polygonisation (one Marching::recalculate(), marching.cpp:308-433 full-grid branch). */
typedef struct {
    uint64_t cubes;       /* cubes visited = (k_end-k_begin) * M * M  ("voxels") */
    uint64_t active;      /* cubes with cube_code not in {0,255} that passed the constraints */
    uint64_t triangles;   /* triangles emitted */
    uint64_t ambiguous;   /* active cubes whose code has a redirect entry (marching_lookup.h:329-587) */
    uint64_t redirected;  /* ... of which the face-centre test chose row 255-code (marching.cpp:545-547) */
    int32_t M;            /* cubes per axis visited by the reference loop (marching.cpp:375-377) */
    int32_t k_begin, k_end; /* cube layers of this context's z-slab */
    float ms_tables;      /* device time of the stages, CUDA events on the context's stream */
    float ms_eval;
    float ms_classify;
    float ms_emit;
    float ms_total;
    uint32_t launches;    /* kernels launched by this call */
    uint32_t reruns;      /* passes repeated because an output buffer had to grow (0 in steady state) */
    float ms_weld;        /* device time of the indexed-mesh stage (0 unless MCB_MESH_INDEXED) */
    uint32_t mesh_mode;   /* MCB_MESH_* bits this result was produced with */
    uint64_t vertices;    /* welded vertices of the indexed mesh (0 unless MCB_MESH_INDEXED) */
    float ms_fill;        /* sparse-field mode: device time of the block refill (flag, list, evaluate); else 0 */
    uint32_t field_mode;  /* MCB_FIELD_* this result was produced with */
    uint64_t field_blocks; /* sparse-field mode: 32 x 4 x 4 vertex blocks the field was written in */
    uint32_t jit;         /* 1: the field was evaluated by the kernel compiled for this equation (mcb_set_jit) */
    float ms_compile;     /* host milliseconds this call spent in NVRTC (0 when the equation's kernel was cached) */
} mcb_counts;

/* Where the scalar field lives (mcb_set_field_mode; default MCB_FIELD_DENSE). */
#define MCB_FIELD_DENSE 0   /* every grid vertex is evaluated and its value written to device memory (4 B per vertex) */
#define MCB_FIELD_SPARSE 1  /* block-field mode: an interval evaluation of the equation per 32 x 4 x 4 vertex block (an exact
                               proof, csrc/mcb_interval.h) decides which blocks can hold a sign change; only those, and the
                               blocks the mesh stages read next to them, are evaluated, and classification visits nothing
                               else.  Decided inside the call from its own data: a first or changed configuration costs
                               the same as a repeated one.  Meshes, normals and counts are bit-identical to
                               MCB_FIELD_DENSE; mcb_get_field is unavailable; mcb_counts::field_blocks = blocks evaluated */
#define MCB_FIELD_AUTO 2    /* MCB_FIELD_SPARSE wherever it applies (everything except the repeating-surface mode, whose
                               per-cube iso levels read the field everywhere); mcb_counts::field_mode says which ran */

/* What mcb_polygonise leaves in device memory (mcb_set_mesh_mode; default MCB_MESH_SOUP). */
#define MCB_MESH_SOUP 1     /* triangle soup: 3 float4 positions (+ 3 float4 normals) per triangle, emission order */
#define MCB_MESH_INDEXED 2  /* Poly_Data layout: welded vertex_list (xyz floats) + tri_list (3 indices per triangle) */

/* ---- library / host-only helpers (no GPU needed) ---------------------------------------------------------- */

int mcb_abi_version(void);
/* sha256 (hex) over the sources the loaded library was built from (csrc/, include/mcb.h): lets a test or a deployment
 * check that the binary in use is the build of the sources next to it */
const char* mcb_build_stamp(void);
/* sizeof of the structs that cross the boundary, so a binding can check its mirror: 0 = mcb_counts, 1 = mcb_step_data */
int mcb_struct_size(int which);
const char* mcb_status_string(int status);

/* Equation grammars (mcb_set_grammar, mcb_grammar_text).
 *   MCB_GRAMMAR_REFERENCE (default)  the reference's language: numbers, x y z (either case), + - * / ^, brackets.
 *   MCB_GRAMMAR_FUNCTIONS            the same plus four functions, lowercase, each written with its bracket: sin( cos(
 *                                    sqrt( abs( (blanks are stripped first, so `sin (x)` is `sin(x)`; `sinx`, `SIN(x)`,
 *                                    `sin()` are parse errors).  A function bracket is a '(' for every rule of the
 *                                    reference's tokenizer and evaluator: implicit multiplication before it (`2sin(x)`
 *                                    is 2*sin(x)), unary minus after it (`sin(-x)`), and `f(E)` is the bracketed operand
 *                                    (E) with f applied at its ')' — so `-sin(x)^2` is (-sin(x))^2, as `-(x)^2` is (-x)^2.
 *                                    Every equation of the reference grammar parses to the same tokens, operation order
 *                                    and bytecode.  sin / cos are glibc's sinf / cosf restated bit for bit on the device
 *                                    (csrc/mcb_trig.h), sqrt is correctly rounded, abs clears the sign bit; all else is
 *                                    unchanged fp32 without FMA contraction.
 *                                    Also two functions of two arguments, min( max(, for unions (min), intersections
 *                                    (max) and differences (max(a,-b)) of signed-distance shapes.  Exactly one ',' goes
 *                                    directly inside their bracket and nowhere else (`(x,y)`, `sin(x,y)`, `min(x)`,
 *                                    `min(x,y,z)` are parse errors).  Each argument is a bracketed operand closed at its
 *                                    ',' or ')', so `max(x-y+z,0)` is max(x-(y+z),0); after the ',' a unary minus is
 *                                    allowed as after '('.  `max(` is matched as a name, so its x is no variable
 *                                    (`xmax(y,z)` is x*max(y,z), `maxx(y,z)` an error).  min / max are IEEE 754-2019
 *                                    minimumNumber / maximumNumber: a NaN operand is ignored, -0 < +0. */
#define MCB_GRAMMAR_REFERENCE 0
#define MCB_GRAMMAR_FUNCTIONS 1

/* Evaluator::tokenize accept/reject (evaluator.cpp:139-237) + the operand-stack check: MCB_OK or MCB_E_PARSE. */
int mcb_parse(const char* equation);
/* Token list as text, blank separated, unary minus printed as NEG (evaluator.cpp:165).  Returns MCB_OK,
 * MCB_E_PARSE, or MCB_E_CAPACITY if `cap` is too small. */
int mcb_tokens(const char* equation, char* out, size_t cap);
/* The operation order the reference's two-stack evaluator (evaluator.cpp:22-107) executes, as postfix text:
 * "x-y+z" -> "x y z + -". */
int mcb_postfix(const char* equation, char* out, size_t cap);
/* Bytecode listing; which: 0 = point program, 1 = grid program (postfix), 2 = hoisted slot programs,
 * 3 = grid program in the fused accumulator form the grid kernel executes. */
int mcb_disassemble(const char* equation, int which, char* out, size_t cap);
/* The four helpers above under a chosen grammar (MCB_GRAMMAR_*; MCB_E_ARG for another value).  what: -1 = accept/reject
 * only (out unused; as mcb_parse), 0 = tokens (as mcb_tokens; a function prints as `sin(`), 1 = postfix (as mcb_postfix;
 * a function follows its operand: `x sin`), 2 + w = bytecode listing w of mcb_disassemble. */
int mcb_grammar_text(const char* equation, int grammar, int what, char* out, size_t cap);
/* The reference's grid loop on one axis (marching.cpp:372-377): returns M = number of cubes per axis for `step`
 * and, when coords != NULL and cap >= M+1, the cube origins c[0..M-1] and the far corner c[M] = c[M-1]+step. */
int mcb_grid_axis(float step, float* coords, int cap);
/* Row `table_idx` of the packed triangle table: sixteen 4-bit edge indices, 0xF terminated (marching_lookup.h:64-320). */
uint64_t mcb_tri_row(int table_idx);
/* Balanced split of M cube layers into nranks contiguous z-slabs (SURVEY.md §8e): layers [*k_begin,*k_end). */
int mcb_slab_range(int M, int rank, int nranks, int* k_begin, int* k_end);

/* ---- context --------------------------------------------------------------------------------------------- */

/* One context = one Marching object (marching.h:72-157) on one CUDA device.  Defaults follow Marching::Marching
 * (marching.cpp:23-37): step 0.25, iso 0, scale 1, no constraints, equation "x+y" (evaluator.cpp:6-8). */
int mcb_create(int device, mcb_ctx** out);
void mcb_destroy(mcb_ctx* ctx);
const char* mcb_last_error(const mcb_ctx* ctx);
/* Use the caller's cudaStream_t (e.g. torch's current stream) instead of the context's own. NULL restores it. */
int mcb_set_stream(mcb_ctx* ctx, void* cuda_stream);

/* ---- evaluator.h ----------------------------------------------------------------------------------------- */

/* Evaluator::set_equation (evaluator.cpp:15-17).  slot 0 = the surface equation (Marching::set_evaluator,
 * marching.cpp:140-147); slots 1..3 = left-hand sides of constraints 0..2 (marching.cpp:173-200).
 * On MCB_E_PARSE the previous equation of that slot stays in force. */
int mcb_set_equation(mcb_ctx* ctx, int slot, const char* equation);
/* MCB_GRAMMAR_REFERENCE (default) or MCB_GRAMMAR_FUNCTIONS for the mcb_set_equation calls that follow, in every slot
 * (surface and constraint left-hand sides).  Equations already set keep their programs. */
int mcb_set_grammar(mcb_ctx* ctx, int grammar);
/* Evaluator::evaluate (evaluator.cpp:53-107) for n points on the GPU.  xyz = 3n floats, out = n floats, host
 * memory.  apply_scale != 0 multiplies by the per-axis scale first, i.e. Marching::evaluate (marching.cpp:209-224). */
int mcb_eval_points(mcb_ctx* ctx, int slot, const float* xyz, float* out, size_t n, int apply_scale);
/* The gradient of the same point program at n points on the GPU: grad = 3n floats (df/dx, df/dy, df/dz), unnormalised,
 * host memory; the forward-mode rules of mcb_set_normals mode 3.  With apply_scale != 0 the program runs at (sx*x, sy*y,
 * sz*z) and the gradient is taken with respect to the unscaled (x, y, z).  Same slots and errors as mcb_eval_points. */
int mcb_eval_gradients(mcb_ctx* ctx, int slot, const float* xyz, float* grad, size_t n, int apply_scale);

/* ---- marching.h ------------------------------------------------------------------------------------------ */

/* Marching::set_grid_step_size (marching.cpp:226-238) without its [0.001,0.5] clamp (the C++ class applies it;
 * 2048^3 needs 2/2048 < 0.001, SURVEY.md D4).  Any finite step in (0, 1] with M <= 4094 is accepted. */
int mcb_set_grid_step(mcb_ctx* ctx, float step);
/* Restrict this context to cube layers [k_begin,k_end) of [0,M) — its z-slab; the one-vertex halo planes are
 * recomputed locally.  k_end <= 0 means M.  Reset to the full grid by mcb_set_grid_step. */
int mcb_set_slab(mcb_ctx* ctx, int k_begin, int k_end);
int mcb_set_surface_constant(mcb_ctx* ctx, float iso);          /* marching.cpp:149-154 */
int mcb_set_scaling(mcb_ctx* ctx, float sx, float sy, float sz); /* marching.cpp:240-251 */
/* Constraint i (0..2): lhs(sx*x,sy*y,sz*z) op rhs with op 0 '>', 1 '<', 2 '>=', 3 '<=' (Comp_Op, marching.h:58);
 * in_use as Marching::use_constraint (marching.cpp:202-207).  The lhs is slot i+1 of mcb_set_equation.  A cube is
 * skipped unless all 8 corners satisfy every constraint in use (marching.cpp:255-280, 475-477). */
int mcb_set_constraint(mcb_ctx* ctx, int i, int op, float rhs, int in_use);
/* Seed mode (Marching::seed_mode + set_seed, marching.cpp:42-137, 310-331): polygonise only the cubes connected to
 * the cube containing (x,y,z) — a point of [-1,1]^3, else MCB_E_ARG — through cube faces that carry a crossing edge.
 * The set of cubes and triangles of the reference's BFS on dyadic grid steps, emitted in the full-grid loop order instead
 * of BFS order.  Deviation: the reference's walk derives its cube origins from the seed (-1 + floor(d) * h, then +-h per
 * move: marching.cpp:76-79, 104-113), not from the accumulated loop coordinates; for non-dyadic steps such as the GUI's
 * 0.2 its positions therefore differ from the full-grid ones by ~2e-6 and tests/test_gpu_seed.py compares with a
 * tolerance there.  The walk stays inside the context's slab: seed mode is a single-context feature — with z-slabs a rank
 * without the seed emits nothing and a component that leaves and re-enters a slab is cut (mcb_comm_init refuses seed mode).
 * enabled = 0 switches back to the full grid. */
int mcb_set_seed(mcb_ctx* ctx, int enabled, float x, float y, float z);
/* 0 = positions only; 1 = also normals from central-difference field gradients (per soup vertex and per welded
 * vertex; DESIGN.md, normals); 2 = CalculateNormal of the reference (normal.h:3-42: area-weighted face normals summed
 * per welded vertex in triangle order, glm::normalize), bit-exact, per welded vertex — needs MCB_MESH_INDEXED;
 * 3 = analytic normals (DESIGN.md §12): the equation's own gradient at every soup and welded vertex, by forward-mode
 * differentiation of the point program in fp32, bit-identical on host and GPU.  Positions, indices and counts are those of
 * mode 0.  With a the left and b the right operand of each operation of the equation:
 *     x, y, z -> (sx,0,0), (0,sy,0), (0,0,sz)     constant -> 0           a+-b -> ga+-gb       a*b -> ga*b + a*gb
 *     a/b -> (ga - q*gb)/b, q = a/b               -a -> -ga               sin a -> cos(a)*ga   cos a -> (-sin(a))*ga
 *     sqrt a -> ga/(s+s), s = sqrt(a)             abs a -> sign bit of a set ? -ga : ga
 *     a^b -> gb exactly 0: (b * a^(b-1)) * ga, else a^b * (ln(a)*gb + (b/a)*ga)  (ln from the fp64 log2 of `^`; NaN for a <= 0)
 *     min / max -> the gradient of the operand whose bits equal the result, (ga+gb)*0.5f when both (or neither) do
 * Normalisation: m = max |g_i|; (0,0,0) when m is 0, infinite or NaN or a component is NaN; otherwise u = g/m,
 * d = ux*ux + uy*uy + uz*uz, n = u * (1/sqrt(d)) (correctly rounded square root).  The normal points towards increasing f,
 * as mode 1's does.  Like mode 2, mode 3 is not streamed through mcb_set_host_output. */
int mcb_set_normals(mcb_ctx* ctx, int mode);

/* The hot path: Marching::recalculate() (marching.cpp:368-384) for this context's slab, entirely on the GPU.
 * On return the triangle soup is resident in device memory in the reference's emission order (cube loop order
 * x fastest, then y, then z; tri_table order inside a cube) and *out holds the counts. */
int mcb_polygonise(mcb_ctx* ctx, mcb_counts* out);

/* The per-stage device times in the counts struct, ms_tables .. ms_total, come from CUDA events recorded between the stages:
 * enabled by default; 0 drops the events (the fields read 0), which shortens the gaps between the short kernels. */
int mcb_set_stage_timing(mcb_ctx* ctx, int enabled);

/* Copy the soup to host memory: pos4 / nrm4 = 3*triangles float4 (x,y,z,1) / (nx,ny,nz,0); either may be NULL.
 * cap_triangles = capacity of the buffers in triangles. */
int mcb_get_mesh(mcb_ctx* ctx, float* pos4, float* nrm4, uint64_t cap_triangles);
/* Device pointers to the same buffers (valid until the next mcb_polygonise / mcb_destroy). */
int mcb_get_mesh_device(mcb_ctx* ctx, const float** pos4, const float** nrm4);

/* Device address of the live counters of the last mcb_polygonise, five uint64: active cubes, triangles, ambiguous,
 * redirected, welded vertices (stable for the lifetime of the context).  For multi-GPU placement the per-slab
 * triangle count can be all-gathered straight from here (NCCL) without a host round trip. */
int mcb_counts_device(mcb_ctx* ctx, const uint64_t** counts);

/* Repeating-surface mode (Marching::repeating_surface_mode / set_surface_repeat_step_distance, marching.cpp:156-170,
 * 481-494; no GUI control in the reference): every cube is polygonised with the highest level
 * surface_constant + n * distance that does not exceed its largest corner value, so one call draws the whole family of
 * level sets.  distance must be > 0.  Forces MCB_FIELD_DENSE; not available together with seed mode. */
int mcb_set_repeat(mcb_ctx* ctx, int enabled, float distance);

/* Run-time specialisation of the evaluator (SURVEY §8f N4).  After an equation change that equation's fused grid program is
 * compiled into straight-line sm_100a kernels with NVRTC (libnvrtc.so.12, loaded on demand; some tens of milliseconds,
 * reported in mcb_counts::ms_compile of the call that adopts them) and later calls reuse them.  The kernel executes the interpreter's fp32
 * operations in the interpreter's order on the interpreter's tile, so every result is bit-identical; it just has no
 * dispatch (torus 2.3 -> 1.5 ms, polynomial gyroid 1.3 -> 0.7 ms at 1024^3).  Constants, grid size and scaling are
 * kernel arguments: only a new equation compiles again.
 *   MCB_JIT_AUTO (default)  use it when NVRTC is there, the compile succeeds and the program has at most 8 `^` left after
 *                           hoisting (more: powf dominates either way and compile time grows; sin and cos of the function
 *                           grammar do not count: the kernel calls one out-of-line copy of each), else the bytecode
 *                           interpreter — both are the same CUDA path with the same results; mcb_counts::jit says which ran.
 *                           The compile runs on a background thread: the first mesh of a new equation does not wait for
 *                           NVRTC, the calls made meanwhile interpret, the first call after the compile has finished
 *                           switches over (mcb_jit_wait blocks until then; $MCB_JIT_SYNC=1 compiles inside the call)
 *   MCB_JIT_ON              require it: mcb_polygonise returns MCB_E_STATE with the log in mcb_last_error otherwise
 *   MCB_JIT_OFF             always interpret
 * One module per equation holds the kernel of the dense mode and the block kernel of the block-field mode. */
#define MCB_JIT_OFF 0
#define MCB_JIT_ON 1
#define MCB_JIT_AUTO 2
int mcb_set_jit(mcb_ctx* ctx, int mode);
/* Block until the compile of the current surface equation's kernels has finished.  1: the next mcb_polygonise runs them;
 * 0: it interprets (MCB_JIT_OFF, no NVRTC, too many powers, or the compile failed — mcb_last_error); < 0: MCB_JIT_ON and the
 * compile failed. */
int mcb_jit_wait(mcb_ctx* ctx);
/* Host-only: generate and compile the specialised kernel for `equation` (no GPU needed).  Returns the cubin size in
 * bytes (> 0) and the generated CUDA source in `log`, or a negative status with the error / compile log in `log`. */
int mcb_jit_check(const char* equation, char* log, size_t cap);
/* The same under a chosen grammar (MCB_GRAMMAR_*). */
int mcb_jit_check_grammar(const char* equation, int grammar, char* log, size_t cap);

/* MCB_FIELD_DENSE (default), MCB_FIELD_SPARSE or MCB_FIELD_AUTO: whether mcb_polygonise evaluates and writes the whole
 * scalar field or only the blocks of it around the surface (SURVEY §8f N4).  Results are bit-identical.  The C++ drop-in
 * class, which never reads the field back, uses MCB_FIELD_AUTO. */
int mcb_set_field_mode(mcb_ctx* ctx, int mode);

/* MCB_MESH_SOUP, MCB_MESH_INDEXED or both (3).  The indexed mesh is what Marching::recalculate() leaves in
 * Poly_Data (marching.h:26-30): vertices welded and numbered as add_step_to_poly_data / add_point do it
 * (marching.cpp:599-654, tolerance comparator marching.h:38-54), triangles in emission order. */
int mcb_set_mesh_mode(mcb_ctx* ctx, int mode);
/* Copy the indexed mesh to host memory: vertex_list = 3*vertices floats (x,y,z), tri_list = 3*triangles indices,
 * normals = 3*vertices floats (normals per welded vertex; needs mcb_set_normals 1, 2 or 3).  Any may be NULL. */
int mcb_get_indexed_mesh(mcb_ctx* ctx, float* vertex_list, uint32_t* tri_list, float* normals, uint64_t cap_vertices,
                         uint64_t cap_triangles);
/* A mesh assembled from several slabs (one context each) numbers the vertices of slab r from the sum of the earlier slabs'
 * vertex counts: `base` is added, on the device, to every index mcb_get_indexed_mesh delivers from then on (default 0;
 * the streamed host output of mcb_set_host_output and mcb_get_indexed_mesh_device are not shifted). */
int mcb_set_index_base(mcb_ctx* ctx, uint32_t base);
int mcb_get_indexed_mesh_device(mcb_ctx* ctx, const float** vertex_list, const uint32_t** tri_list, const float** normals);
/* Register host buffers (pinned memory for real overlap) as the destination of the indexed mesh.  While they are
 * registered, mcb_polygonise in MCB_MESH_INDEXED mode streams vertex_list / normals / tri_list out range by range
 * while the later ranges are still being produced, and returns when the mesh is on the host — one call, like
 * Marching::recalculate() filling Poly_Data.  normals may be NULL when normals are off.  When a device buffer has to
 * grow first, the mesh does not fit the registered capacities, or normals mode 2 or 3 is on, nothing is
 * streamed: mcb_host_output_filled() returns 0 and mcb_get_indexed_mesh delivers the mesh.  NULL pointers unregister. */
int mcb_set_host_output(mcb_ctx* ctx, float* vertex_list, uint32_t* tri_list, float* normals, uint64_t cap_vertices,
                        uint64_t cap_triangles);
int mcb_host_output_filled(const mcb_ctx* ctx);

/* ---- z-slabs over several GPUs (SURVEY.md §8e; BASELINE.json configs[4]) ---------------------------------------
 * One context per GPU, each with its slab of cube layers (mcb_set_slab); the field is analytic, so every slab recomputes
 * its halo planes and the only exchange of the path is one integer per rank: the slab's triangle count, all-gathered
 * over NCCL (NVLink / NVSwitch) so that every rank knows its offset in the global triangle list (the reference emits z
 * slowest, marching.cpp:375-383: concatenating the slabs in rank order reproduces its order).  libnccl.so.2 is loaded
 * on first use, like NVRTC; without it these calls return MCB_E_STATE and the single-GPU path is unaffected.
 * The ranks may be processes (one GPU each, the id travelling by any out-of-band means) or threads of one process
 * (include/marching.h: Marching::set_devices). */
/* Triangles per cube layer of this context's slab in the last polygonisation, k_end - k_begin values. */
int mcb_layer_triangles(mcb_ctx* ctx, uint32_t* per_layer);
/* Host only: cut M cube layers into nranks contiguous slabs of (nearly) equal cost, cost(layer) = triangles_per_layer[k]
 * + fixed_cost_per_layer (< 0: the default, 0.0015 * M * M — what a layer costs before it emits anything, in
 * triangles).  cuts[0..nranks]: rank r takes layers [cuts[r], cuts[r+1]).  Every slab gets at least one layer. */
int mcb_balance_slabs(int M, int nranks, const uint32_t* triangles_per_layer, double fixed_cost_per_layer, int* cuts);
/* Host only: one refinement of such a cut by measured time.  cost[M] (in/out): the cost of every layer as the cut saw it
 * (triangles + fixed cost); cuts[nranks+1] (in/out); ms[nranks]: what each slab was measured to take.  Each slab's time is
 * spread over its layers in proportion to their cost, then the layers are cut again. */
int mcb_rebalance_slabs(int M, int nranks, double* cost, int* cuts, const double* ms);
/* ncclGetUniqueId into 128 bytes: call on one rank, hand the bytes to the others. */
int mcb_comm_unique_id(void* id128);
/* Join the communicator (ncclCommInitRank on the context's device) and take the balanced-by-layer-count slab of `rank`
 * (mcb_slab_range).  Collective over the nranks contexts. */
int mcb_comm_init(mcb_ctx* ctx, const void* id128, int rank, int nranks);
/* Enqueue the all-gather of this slab's triangle count, straight from the device counters of the last mcb_polygonise,
 * on a side stream: the next polygonisation does not wait for the slowest rank.  Collective. */
int mcb_comm_exchange(mcb_ctx* ctx);
/* enabled != 0: mcb_polygonise enqueues that all-gather itself, right after classification, when the slab's triangle count
 * is final — NCCL's launch cost then hides behind the emission instead of following the call; mcb_comm_exchange becomes
 * a no-op.  Every rank must use the same setting.  (The count is the one of the call's first pass; a pass repeated
 * because the ambiguity list overflowed — 2^18 ambiguous cubes in one slab — can change it, the next call corrects it.) */
int mcb_comm_set_auto(mcb_ctx* ctx, int enabled);
/* Result of the last exchange (waits for it): offset of this slab in the global triangle list, the global total, and the
 * per-rank counts (nranks values; may be NULL). */
int mcb_comm_offsets(mcb_ctx* ctx, uint64_t* offset, uint64_t* total, uint64_t* per_rank);
/* Re-cut the slabs so that every rank carries the same cost: all-reduce (NCCL) of the per-layer triangle counts of the
 * last polygonisation, mcb_balance_slabs on every rank, mcb_set_slab with this rank's share.  Collective; the new slab
 * is returned in *k_begin / *k_end (either may be NULL).  A configuration is profiled once with the uniform slabs and
 * polygonised with the balanced ones from then on. */
int mcb_comm_balance(mcb_ctx* ctx, double fixed_cost_per_layer, int* k_begin, int* k_end);
/* Refine the cut of mcb_comm_balance with MEASURED time: ms_measured is what this rank's balanced slab took (e.g. the mean
 * mcb_counts::ms_total of a few calls).  The times are all-gathered, each slab's time is spread over its layers in
 * proportion to their modelled cost, and the layers are cut again; equal times are the fixed point, one or two passes
 * settle it.  (fixed_cost_per_layer < 0 in mcb_comm_balance: 0.00015 M^2 in the block-field mode, 0.0015 M^2 with the
 * dense field.)  Collective; needs mcb_comm_balance to have cut the current slabs. */
int mcb_comm_rebalance(mcb_ctx* ctx, double ms_measured, int* k_begin, int* k_end);
/* Leave the communicator (also done by mcb_destroy). */
int mcb_comm_finalize(mcb_ctx* ctx);

/* Page-lock host memory the caller owns (cudaHostRegister / cudaHostUnregister), so that mcb_set_host_output can stream
 * into it at full PCIe speed: what the C++ drop-in does with the storage of its Poly_Data vectors. */
int mcb_host_register(void* ptr, size_t bytes);
int mcb_host_unregister(void* ptr);

/* Marching::calculate_step(x_0, y_0, z_0) (marching.cpp:456-595) for ONE cube with origin (x0,y0,z0) and the context's
 * step, scale, iso, equation and constraints: the Step_Data (marching.h:15-23) the GUI's step-by-step / movie mode
 * displays.  skipped = 1 when a constraint rejects a corner (the reference returns before filling anything else). */
typedef struct {
    float corner_coords[24];
    float corner_values[8];
    float intersect_coord[36]; /* 3 per crossing edge, ascending edge order */
    int32_t edge_list[12];
    int32_t tri_vlist[15];     /* indices into intersect_coord / 3, three per triangle */
    int32_t n_edges, n_tri_idx, cube_code, table_idx, skipped;
    float surf_constant;       /* the iso value this cube was polygonised with (Step_Data::surf_constant in repeating-surface mode) */
} mcb_step_data;
int mcb_inspect_cube(mcb_ctx* ctx, float x0, float y0, float z0, mcb_step_data* out);

/* Parity hooks.  Dense per-cube arrays of the slab in loop order, host memory, `cubes` bytes each (NULL = skip):
 * cube_code = raw 8-bit sign code (marching.cpp:497-505); table_idx = tri_table row actually used (code or
 * 255-code); a cube skipped by a constraint reports 0 in both. */
int mcb_get_cases(mcb_ctx* ctx, uint8_t* cube_code, uint8_t* table_idx);
/* Field values at the slab's grid vertices, (k_end-k_begin+1) * (M+1) * (M+1) floats, x fastest. */
int mcb_get_field(mcb_ctx* ctx, float* out);
/* Compacted active-cube list: record = i | j<<12 | k<<24 | code<<36 | table_idx<<44; tri_offset = index of the
 * cube's first triangle.  cap = capacity in records. */
int mcb_get_active(mcb_ctx* ctx, uint64_t* records, uint32_t* tri_offsets, uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* MCB_H */
