/* Dual contouring (mcb_set_mesh_mode MCB_MESH_DC, include/mcb.h, DESIGN.md §14): one vertex per active cube, placed by
 * the Hermite data of the cube's crossing grid edges (each edge's refined crossing point and the analytic normal there),
 * and one quad per crossing grid edge whose four cubes are active.  One source for g++ (the host build the tests compare
 * with) and nvcc (dc_edges_kernel, dc_vertex_kernel, dc_emit_kernel); all arithmetic is fp32 without FMA contraction and
 * the square root is correctly rounded, so both give the same bits.
 *
 * The vertex minimises sum_k (n_k . (x - p_k))^2 (Ju, Losasso, Schaefer, Warren, SIGGRAPH 2002), solved around the mass
 * point with the small eigenvalues of A = sum n n^T truncated, then clamped to the cube. */
#ifndef MCB_QEF_H
#define MCB_QEF_H

#include "mcb_bytecode.h"
#include "mcb_refine.h"

#define MCB_QEF_SWEEPS 6 /* cyclic Jacobi sweeps: off-diagonal entries below 1e-6 of the largest eigenvalue on every cell of tests/test_dc_host.py */
#define MCB_QEF_CUT 0.01f /* eigenvalues below MCB_QEF_CUT * the largest are dropped: singular values below 0.1 of the largest */

/* Hermite data of one crossing grid edge.  lo[3] = the edge's lower end point, axis = its direction, (c[ia], c[ia + 1]) its
 * extent on that axis, flo / fhi the field values at its ends.  out: the refined coordinate along the axis, then the unit
 * normal there (mode 3's normal; (0,0,0) where the gradient has none). */
MCB_BC_FN void mcb_dc_edge(const uint32_t* code, int n, const float* k, const float* c, int M, float iso, float sx, float sy, float sz,
                           const float lo[3], int axis, int ia, float flo, float fhi, float out[4]) {
    float p[3] = {lo[0], lo[1], lo[2]};
    p[axis] = mcb_interp_ref(c[ia], c[ia + 1], (iso - flo) / (fhi - flo)); /* the emitter's linear point, lower -> upper */
    mcb_refine_vertex(code, n, k, c, M, iso, sx, sy, sz, p, 0);
    float g[3];
    mcb_interp_grad_scalar(code, n, k, sx * p[0], sy * p[1], sz * p[2], sx, sy, sz, g);
    out[0] = p[axis];
    mcb_grad_normalise(g, out + 1);
}

/* One rotation of cyclic Jacobi on the symmetric 3 x 3 matrix a (row-major, both triangles kept), accumulated into the
 * eigenvector columns of v: the classic stable form (t the smaller root of t^2 + 2 theta t - 1 = 0). */
MCB_BC_FN void mcb_qef_rotate(float a[9], float v[9], int p, int q) {
    const float apq = a[3 * p + q];
    if (apq == 0.f) return;
    const float theta = (a[3 * q + q] - a[3 * p + p]) / (apq + apq);
    const float at = mcb_abs(theta);
    float t = 1.f / (at + mcb_sqrt(theta * theta + 1.f));
    if (theta < 0.f) t = -t;
    const float cs = 1.f / mcb_sqrt(t * t + 1.f), sn = t * cs;
    a[3 * p + p] = a[3 * p + p] - t * apq;
    a[3 * q + q] = a[3 * q + q] + t * apq;
    a[3 * p + q] = 0.f;
    a[3 * q + p] = 0.f;
    const int r = 3 - p - q; /* the third index */
    const float arp = a[3 * r + p], arq = a[3 * r + q];
    a[3 * r + p] = cs * arp - sn * arq;
    a[3 * p + r] = a[3 * r + p];
    a[3 * r + q] = sn * arp + cs * arq;
    a[3 * q + r] = a[3 * r + q];
    for (int i = 0; i < 3; i++) {
        const float vp = v[3 * i + p], vq = v[3 * i + q];
        v[3 * i + p] = cs * vp - sn * vq;
        v[3 * i + q] = sn * vp + cs * vq;
    }
}

/* Eigen-decomposition of the symmetric a (overwritten: its diagonal becomes the eigenvalues) with the eigenvectors as the
 * columns of v.  `sweeps` full sweeps in the pair order (0,1), (0,2), (1,2). */
MCB_BC_FN void mcb_qef_jacobi(float a[9], float v[9], int sweeps) {
    for (int i = 0; i < 9; i++) v[i] = (i % 4 == 0) ? 1.f : 0.f;
    for (int s = 0; s < sweeps; s++) {
        mcb_qef_rotate(a, v, 0, 1);
        mcb_qef_rotate(a, v, 0, 2);
        mcb_qef_rotate(a, v, 1, 2);
    }
}

/* The vertex of one active cube.  pts[m][3] / nrm[m][3]: the Hermite data of its crossing edges in edge order 0..11;
 * lo[3] / hi[3]: the cube's corners.  Returns the number of eigenvalues kept (the rank used, 0..3); x[3] = the vertex.
 * When `sweeps_out` is not null the matrix after the Jacobi sweeps is left there (diagonal = eigenvalues) and the
 * eigenvectors in sweeps_out + 9, for the tests. */
MCB_BC_FN int mcb_qef_vertex(const float (*pts)[3], const float (*nrm)[3], int m, const float lo[3], const float hi[3], float x[3],
                             float* sweeps_out) {
    float c[3] = {0.f, 0.f, 0.f};
    for (int q = 0; q < m; q++)
        for (int d = 0; d < 3; d++) c[d] = c[d] + pts[q][d];
    const float fm = (float)m;
    for (int d = 0; d < 3; d++) c[d] = c[d] / fm;
    float a[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, r[3] = {0.f, 0.f, 0.f};
    for (int q = 0; q < m; q++) {
        const float nx = nrm[q][0], ny = nrm[q][1], nz = nrm[q][2];
        if (nx == 0.f && ny == 0.f && nz == 0.f) continue; /* no plane: the point only counts for the mass point */
        a[0] = a[0] + nx * nx; a[1] = a[1] + nx * ny; a[2] = a[2] + nx * nz;
        a[4] = a[4] + ny * ny; a[5] = a[5] + ny * nz; a[8] = a[8] + nz * nz;
        const float dot = (nx * (pts[q][0] - c[0]) + ny * (pts[q][1] - c[1])) + nz * (pts[q][2] - c[2]);
        r[0] = r[0] + nx * dot; r[1] = r[1] + ny * dot; r[2] = r[2] + nz * dot;
    }
    a[3] = a[1]; a[6] = a[2]; a[7] = a[5];
    float v[9];
    mcb_qef_jacobi(a, v, MCB_QEF_SWEEPS);
    if (sweeps_out) for (int i = 0; i < 9; i++) { sweeps_out[i] = a[i]; sweeps_out[9 + i] = v[i]; }
    float lmax = a[0];
    if (a[4] > lmax) lmax = a[4];
    if (a[8] > lmax) lmax = a[8];
    float off[3] = {0.f, 0.f, 0.f};
    int rank = 0;
    if (lmax > 0.f) {
        const float cut = MCB_QEF_CUT * lmax;
        for (int i = 0; i < 3; i++) {
            const float li = a[4 * i];
            if (!(li >= cut)) continue;
            const float w = ((v[i] * r[0] + v[3 + i] * r[1]) + v[6 + i] * r[2]) / li;
            for (int d = 0; d < 3; d++) off[d] = off[d] + w * v[3 * d + i];
            rank++;
        }
    }
    for (int d = 0; d < 3; d++) {
        const float xd = c[d] + off[d];
        x[d] = !(xd >= lo[d]) ? lo[d] : xd > hi[d] ? hi[d] : xd; /* never outside the cube (a NaN lands on the lower face) */
    }
    return rank;
}

/* A quad's split: its vertices w0..w3 in winding order; true = along w0-w2 (triangles w0 w1 w2, w0 w2 w3), false = along
 * w1-w3 (w0 w1 w3, w1 w2 w3).  The shorter diagonal, squared lengths summed x, y, z; w0-w2 on a tie. */
MCB_BC_FN bool mcb_dc_split02(const float* w0, const float* w1, const float* w2, const float* w3) {
    const float ax = w2[0] - w0[0], ay = w2[1] - w0[1], az = w2[2] - w0[2];
    const float bx = w3[0] - w1[0], by = w3[1] - w1[1], bz = w3[2] - w1[2];
    const float d02 = (ax * ax + ay * ay) + az * az, d13 = (bx * bx + by * by) + bz * bz;
    return !(d13 < d02);
}

/* The four cubes around the quad edge of axis `axis` owned by cube (i,j,k) — the edge through the cube's corner
 * (i+1, j+1, k+1) — in cycle order (0,0), (1,0), (1,1), (0,1) over the edge's two other axes taken cyclically (y,z for x,
 * z,x for y, x,y for z); reversed (0,0), (0,1), (1,1), (1,0) when the edge's lower end lies above the level.  out[4][3]. */
MCB_BC_FN void mcb_dc_quad_cubes(int i, int j, int k, int axis, bool reverse, int out[4][3]) {
    const int ua[4] = {0, 1, 1, 0}, ub[4] = {0, 0, 1, 1};
    for (int s = 0; s < 4; s++) {
        const int t = reverse ? (4 - s) & 3 : s;
        const int a = ua[t], b = ub[t];
        if (axis == 0) { out[s][0] = i; out[s][1] = j + a; out[s][2] = k + b; }
        else if (axis == 1) { out[s][0] = i + b; out[s][1] = j; out[s][2] = k + a; }
        else { out[s][0] = i + a; out[s][1] = j + b; out[s][2] = k; }
    }
}

/* Local edge of a cube through its corner (i+1, j+1, k+1) along each axis (mcb_tables.h numbering): 6 (x), 5 (y), 10 (z). */
MCB_BC_FN int mcb_dc_quad_edge(int axis) { return axis == 0 ? 6 : axis == 1 ? 5 : 10; }

#endif /* MCB_QEF_H */
