/* TEST INFRASTRUCTURE ONLY — the host build of the refined vertices (csrc/mcb_refine.h: mcb_refine_vertex) on the product's
 * own lowering, through oracle/host_interp_fn.cpp (included unchanged).
 *   int mcrh_refine(eq, c, M, iso, sx, sy, sz, xyz, n, out, evals, bracket)
 *       for each of the n points xyz (unscaled x, y, z): out = the refined point (3 floats), evals = mcb_refine_vertex's
 *       return value (evaluations, 0 off an edge's interior, -1 same sign at both ends), bracket = the final bracket
 *       (2 floats); c[0..M] = the grid's coordinate table (mcb_grid_axis)
 *   int mcrh_eval(eq, xyz, n, sx, sy, sz, out)   mcb_interp_scalar of the point program at (sx*x, sy*y, sz*z)
 *   float mcrh_interp(xs, xe, t)                  mcb_interp_ref (Marching::interp)
 * Built by tests/refine_common.py with -ffp-contract=off, as the product's host code is. */
#include "../../oracle/host_interp_fn.cpp"
#include "../../marching-cube-for-implicit-surfaces_b200/csrc/mcb_refine.h"

extern "C" int mcrh_refine(const char* eq, const float* c, int M, float iso, float sx, float sy, float sz, const float* xyz, long n,
                           float* out, int* evals, float* bracket) {
    mcb::Compiled cc;
    int rc = mcb::compile(eq, cc, nullptr, g_grammar);
    if (rc != MCB_OK) return rc;
    fold(cc);
    const uint32_t* code = cc.point_code.data();
    const int nc = (int)cc.point_code.size();
    for (long i = 0; i < n; i++) {
        float p[3] = {xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]}, br[2] = {0.f, 0.f};
        evals[i] = mcb_refine_vertex(code, nc, cc.kpool.data(), c, M, iso, sx, sy, sz, p, br);
        out[3 * i] = p[0]; out[3 * i + 1] = p[1]; out[3 * i + 2] = p[2];
        bracket[2 * i] = br[0]; bracket[2 * i + 1] = br[1];
    }
    return MCB_OK;
}

extern "C" int mcrh_eval(const char* eq, const float* xyz, long n, float sx, float sy, float sz, float* out) {
    mcb::Compiled cc;
    int rc = mcb::compile(eq, cc, nullptr, g_grammar);
    if (rc != MCB_OK) return rc;
    fold(cc);
    for (long i = 0; i < n; i++)
        out[i] = mcb_interp_scalar(cc.point_code.data(), (int)cc.point_code.size(), cc.kpool.data(), sx * xyz[3 * i], sy * xyz[3 * i + 1],
                                   sz * xyz[3 * i + 2], nullptr, nullptr, nullptr);
    return MCB_OK;
}

extern "C" float mcrh_interp(float xs, float xe, float t) { return mcb_interp_ref(xs, xe, t); }
