/* TEST INFRASTRUCTURE ONLY — the host build of dual contouring (csrc/mcb_qef.h) on the product's own lowering, through
 * oracle/host_interp_fn.cpp (included unchanged).
 *   long mcdh_mesh(eq, c, M, iso, sx, sy, sz, F, valid, vlist, cap_v, tlist, cap_t, ntri, cell_p, cell_n, cell_m, rank)
 *       the DC mesh of the field F[(M+1)^3] (x fastest; the grid program at the scaled grid coordinates) on the coordinate
 *       table c[0..M]; valid[(M+1)^3] (or null) = every constraint holds at the vertex.  Returns the vertex count (= the
 *       active cubes) and *ntri.  Cubes are visited in loop order, every crossing edge's Hermite data is computed afresh by
 *       each cube that uses it (the same function of the edge's own data as the device's once-per-edge pass), quads as the
 *       device emits them.  cell_p / cell_n [cap_v][12][3], cell_m [cap_v], rank [cap_v]: the Hermite data each vertex
 *       was solved from and the rank its solve kept (any may be null).
 *   int mcdh_qef(pts, nrm, m, lo, hi, x, mat)   mcb_qef_vertex; mat = the matrix after the sweeps (9) + eigenvectors (9)
 * Built by tests/dc_common.py with -ffp-contract=off, as the product's host code is. */
#include <vector>

#include "../../oracle/host_interp_fn.cpp"
#include "../../marching-cube-for-implicit-surfaces_b200/csrc/mcb_qef.h"
#include "../../marching-cube-for-implicit-surfaces_b200/csrc/mcb_tables.h"

namespace {

struct Field {
    const float* F;
    const uint8_t* valid;
    int M;
    float at(int i, int j, int k) const { return F[((size_t)k * (M + 1) + j) * (M + 1) + i]; }
    bool ok(int i, int j, int k) const { return !valid || valid[((size_t)k * (M + 1) + j) * (M + 1) + i]; }
};

void corners(const Field& f, int i, int j, int k, float v[8]) {
    for (int q = 0; q < 8; q++) {
        const int o = mcb_corner_ofs(q);
        v[q] = f.at(i + (o & 1), j + ((o >> 1) & 1), k + (o >> 2));
    }
}

}  // namespace

extern "C" long mcdh_mesh(const char* eq, const float* c, int M, float iso, float sx, float sy, float sz, const float* F, const uint8_t* valid,
                          float* vlist, long cap_v, uint32_t* tlist, long cap_t, long* ntri, float* cell_p, float* cell_n, int* cell_m, int* rank) {
    mcb::Compiled cc;
    if (mcb::compile(eq, cc, nullptr, g_grammar) != MCB_OK) return -1;
    fold(cc);
    const uint32_t* code = cc.point_code.data();
    const int nc = (int)cc.point_code.size();
    const float* kp = cc.kpool.data();
    const Field fd{F, valid, M};
    std::vector<long> index((size_t)M * M * M, -1);
    auto cube_ok = [&](int i, int j, int k) {
        if (i < 0 || j < 0 || k < 0 || i >= M || j >= M || k >= M) return false;
        for (int q = 0; q < 8; q++)
            if (!fd.ok(i + (q & 1), j + ((q >> 1) & 1), k + (q >> 2))) return false;
        return true;
    };
    long A = 0;
    std::vector<int> cubes;
    for (int k = 0; k < M; k++)
        for (int j = 0; j < M; j++)
            for (int i = 0; i < M; i++) {
                float v[8];
                corners(fd, i, j, k, v);
                int code8 = 0;
                for (int q = 0; q < 8; q++) code8 |= (v[q] > iso ? 1 : 0) << q;
                if (code8 == 0 || code8 == 255 || !cube_ok(i, j, k)) continue;
                index[((size_t)k * M + j) * M + i] = A++;
                cubes.push_back(i); cubes.push_back(j); cubes.push_back(k);
            }
    for (long q = 0; q < A; q++) {
        const int i = cubes[3 * q], j = cubes[3 * q + 1], k = cubes[3 * q + 2];
        float v[8];
        corners(fd, i, j, k, v);
        float pts[12][3], nrm[12][3];
        int m = 0;
        for (int e = 0; e < 12; e++) {
            const int a = mcb_edge_a(e), b = mcb_edge_b(e);
            if ((v[a] > iso) == (v[b] > iso)) continue;
            const int oa = mcb_corner_ofs(a), ob = mcb_corner_ofs(b), lo = oa & ob, d = oa ^ ob;
            const int axis = d == 1 ? 0 : d == 2 ? 1 : 2;
            const int g[3] = {i + (lo & 1), j + ((lo >> 1) & 1), k + (lo >> 2)};
            const float plo[3] = {c[g[0]], c[g[1]], c[g[2]]};
            const float flo = oa < ob ? v[a] : v[b], fhi = oa < ob ? v[b] : v[a];
            float h[4];
            mcb_dc_edge(code, nc, kp, c, M, iso, sx, sy, sz, plo, axis, g[axis], flo, fhi, h);
            pts[m][0] = plo[0]; pts[m][1] = plo[1]; pts[m][2] = plo[2];
            pts[m][axis] = h[0];
            nrm[m][0] = h[1]; nrm[m][1] = h[2]; nrm[m][2] = h[3];
            m++;
        }
        const float clo[3] = {c[i], c[j], c[k]}, chi[3] = {c[i + 1], c[j + 1], c[k + 1]};
        float x[3];
        const int rk = mcb_qef_vertex(pts, nrm, m, clo, chi, x, nullptr);
        if (q < cap_v) {
            vlist[3 * q] = x[0]; vlist[3 * q + 1] = x[1]; vlist[3 * q + 2] = x[2];
            if (rank) rank[q] = rk;
            if (cell_m) cell_m[q] = m;
            for (int s = 0; s < 12 * 3; s++) {
                if (cell_p) cell_p[36 * q + s] = s / 3 < m ? pts[s / 3][s % 3] : 0.f;
                if (cell_n) cell_n[36 * q + s] = s / 3 < m ? nrm[s / 3][s % 3] : 0.f;
            }
        }
    }
    long T = 0;
    for (long q = 0; q < A; q++) {
        const int i = cubes[3 * q], j = cubes[3 * q + 1], k = cubes[3 * q + 2];
        float v[8];
        corners(fd, i, j, k, v);
        for (int axis = 0; axis < 3; axis++) {
            const int e = mcb_dc_quad_edge(axis), a = mcb_edge_a(e), b = mcb_edge_b(e);
            if ((v[a] > iso) == (v[b] > iso)) continue;
            const float flo = mcb_corner_ofs(a) < mcb_corner_ofs(b) ? v[a] : v[b];
            int cb[4][3];
            mcb_dc_quad_cubes(i, j, k, axis, flo > iso, cb);
            long w[4];
            bool ok = true;
            for (int s = 0; s < 4; s++) {
                ok = ok && cube_ok(cb[s][0], cb[s][1], cb[s][2]);
                w[s] = ok ? index[((size_t)cb[s][2] * M + cb[s][1]) * M + cb[s][0]] : -1;
            }
            if (!ok) continue;
            const bool d02 = mcb_dc_split02(vlist + 3 * w[0], vlist + 3 * w[1], vlist + 3 * w[2], vlist + 3 * w[3]);
            const long tri[6] = {w[0], w[1], d02 ? w[2] : w[3], d02 ? w[0] : w[1], w[2], w[3]};
            for (int h = 0; h < 2; h++, T++)
                if (T < cap_t)
                    for (int s = 0; s < 3; s++) tlist[3 * T + s] = (uint32_t)tri[3 * h + s];
        }
    }
    *ntri = T;
    return A;
}

extern "C" int mcdh_qef(const float* pts, const float* nrm, int m, const float* lo, const float* hi, float* x, float* mat) {
    return mcb_qef_vertex(reinterpret_cast<const float(*)[3]>(pts), reinterpret_cast<const float(*)[3]>(nrm), m, lo, hi, x, mat);
}
