/* TEST INFRASTRUCTURE ONLY — CPU restatement (plain C) of the reference's hot path.  See mc_oracle.c. */
#ifndef MC_ORACLE_H
#define MC_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mco mco;

mco* mco_create(void);
void mco_destroy(mco*);

/* pow_mode: 0 = libm powf (what the reference calls), 1 = the product's mcb_powf restatement */
void mco_set_pow_mode(mco*, int mode);
int mco_parse_ok(const char* eq);                                  /* evaluator.cpp:139-237 */
int mco_tokenize_ok(const char* eq);                               /* Evaluator::tokenize alone: no operand-underflow check */
int mco_set_equation(mco*, int slot, const char* eq);              /* slot 0 surface, 1..3 constraint lhs */
float mco_evaluate(mco*, int slot, float x, float y, float z);     /* evaluator.cpp:53-107 */
void mco_eval_points(mco*, int slot, const float* xyz, float* out, long n, int apply_scale);
int mco_set_step(mco*, float step);                                /* returns M */
void mco_set_scale(mco*, float sx, float sy, float sz);
void mco_set_iso(mco*, float iso);
int mco_set_constraint(mco*, int i, int op, float rhs, int in_use);
int mco_grid(mco*, float* coords, int cap);                        /* M; coords[0..M] */

/* Sweep cube layers [k0,k1) in loop order (marching.cpp:375-383) with nthreads workers (per-cube outputs are
 * independent; welding, if requested, is done serially afterwards in loop order).
 * Outputs (any may be NULL): per-cube code/table_idx/ntri; soup = 9 floats per triangle; gradient normals soup
 * (product definition) = 9 floats per triangle.  Returns triangles; counts through the pointers. */
long mco_sweep(mco*, int k0, int k1, int nthreads, uint8_t* code, uint8_t* tidx, uint8_t* ntri, float* soup,
               float* grad_normals, long cap_tris, long* n_active, long* n_ambiguous, long* n_redirected);

/* Weld a soup exactly like add_step_to_poly_data/add_point (marching.cpp:599-643, marching.h:38-54).
 * ntri_per_cube/ncubes describe how the soup splits into cubes (vertices are added per cube in ascending-edge
 * order, which the soup does not record) — pass the per-cube edge lists instead: see mco_weld_cubes. */
long mco_recalculate(mco*, int nthreads);                          /* full grid + weld; returns triangles */
long mco_num_vertices(mco*);
long mco_num_triangles(mco*);
void mco_copy_mesh(mco*, float* verts, unsigned* tris);
void mco_normals(mco*, float* out);                                /* normal.h:3-42 on the welded mesh */

/* timing helper for bench.py's cpu_baseline "port" leg: sweep rows [row0,row0+nrows) with nthreads; seconds */
double mco_timed_rows(mco*, long row0, long nrows, int nthreads, long* cubes, long* tris);

#ifdef __cplusplus
}
#endif
#endif
