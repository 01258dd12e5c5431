"""Shared material of the dual-contouring tests (test_dc_host.py, test_gpu_dc.py): the host build of the rule
(tests/cpp/dc_host.cpp on csrc/mcb_qef.h), the field it runs on, an independent integer statement of the quads, mesh
checks, and the pipeline in MCB_MESH_DC mode."""
import ctypes as C
import os

import numpy as np

from .functions_common import CSRC, GRAMMAR_FUNCTIONS, ORACLE, ROOT, _build, _headers, host_fn_lib

F = GRAMMAR_FUNCTIONS
QEF_SWEEPS = 6  # MCB_QEF_SWEEPS, csrc/mcb_qef.h
QEF_CUT = 0.01  # MCB_QEF_CUT
MESH_DC = 4
BOX = "max(max(abs(x)-0.5,abs(y)-0.4),abs(z)-0.3)"
SPHERE = "x^2+y^2+z^2-0.49"
OPS = {">": np.greater, "<": np.less, ">=": np.greater_equal, "<=": np.less_equal}

_host = None


def host_lib():
    global _host
    if _host is None:
        so = _build("libmcb_dc_host.so", [os.path.join(ROOT, "tests", "cpp", "dc_host.cpp"), os.path.join(CSRC, "mcb_lower.cpp")],
                    _headers() + [os.path.join(CSRC, "mcb_qef.h"), os.path.join(CSRC, "mcb_refine.h"), os.path.join(ORACLE, "host_interp.cpp"),
                                  os.path.join(ORACLE, "host_interp_fn.cpp")],
                    ["g++", "-std=c++17", "-O2", "-ffp-contract=off"], shared=True)
        L = C.CDLL(so)
        vp, f = C.c_void_p, C.c_float
        L.mcoh_set_grammar.argtypes = [C.c_int]
        L.mcdh_mesh.argtypes = [C.c_char_p, vp, C.c_int, f, f, f, f, vp, vp, vp, C.c_long, vp, C.c_long, vp, vp, vp, vp, vp]
        L.mcdh_mesh.restype = C.c_long
        L.mcdh_qef.argtypes = [vp, vp, C.c_int, vp, vp, vp, vp]
        _host = L
    return _host


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def grid_axis(step):
    """c[0..M] of the reference loop (mcb_grid_axis), without a device"""
    c, v, upper = [], np.float32(-1.0), np.float32(1.0 + 0.5 * float(np.float32(step)))
    while v <= upper:
        c.append(v)
        v = np.float32(v + np.float32(step))
    c.append(np.float32(c[-1] + np.float32(step)))
    return np.array(c, np.float32)


def host_field(eq, c, scale=(1.0, 1.0, 1.0), grammar=F):
    """the grid program at the scaled grid coordinates, [k][j][i] over c[0..M]^3: the field the device writes"""
    H = host_fn_lib()
    H.mcoh_set_grammar(grammar)
    ax = [np.ascontiguousarray(np.float32(s) * c, np.float32) for s in scale]
    n = len(c)
    out = np.empty(n ** 3, np.float32)
    assert H.mcoh_eval_grid(eq.encode(), _p(ax[0]), n, _p(ax[1]), n, _p(ax[2]), n, _p(out)) == 0, eq
    return out.reshape(n, n, n)


def host_dc(eq, step, iso=0.0, scale=(1.0, 1.0, 1.0), grammar=F, cons=()):
    """The host build's DC mesh: dict with c, M, field, valid (per vertex), vl[V,3], tl[T,3], and per vertex the Hermite
    data it was solved from (cell_p / cell_n [V,12,3], cell_m) and the rank its solve kept."""
    c = grid_axis(step)
    M = len(c) - 1
    fld = host_field(eq, c, scale, grammar)
    valid = None
    if cons:
        valid = np.ones(fld.shape, bool)
        for lhs, op, rhs in cons:
            valid &= OPS[op](host_field(lhs, c, scale, grammar), np.float32(rhs))
        valid = valid.astype(np.uint8)
    L = host_lib()
    L.mcoh_set_grammar(grammar)
    cap_v = int(np.count_nonzero(active_cubes(dict(field=fld, valid=valid, iso=iso, M=M)))) + 1
    vl = np.empty((cap_v, 3), np.float32)
    cap_t = 6 * cap_v
    tl = np.empty((cap_t, 3), np.uint32)
    cp, cn = np.zeros((cap_v, 12, 3), np.float32), np.zeros((cap_v, 12, 3), np.float32)
    cm, rk = np.zeros(cap_v, np.int32), np.zeros(cap_v, np.int32)
    nt = C.c_long(0)
    V = L.mcdh_mesh(eq.encode(), _p(c), M, C.c_float(iso), *[C.c_float(x) for x in scale], _p(np.ascontiguousarray(fld)), _p(valid),
                    _p(vl), cap_v, _p(tl), cap_t, C.byref(nt), _p(cp), _p(cn), _p(cm), _p(rk))
    assert 0 <= V <= cap_v and nt.value <= cap_t, (eq, V, nt.value)
    return dict(c=c, M=M, field=fld, valid=valid, vl=vl[:V].copy(), tl=tl[:nt.value].copy(), cell_p=cp[:V], cell_n=cn[:V], cell_m=cm[:V],
                rank=rk[:V], iso=iso)


def qef(pts, nrm, lo, hi):
    """mcb_qef_vertex of the host build: (x[3], rank, matrix after the sweeps [3,3], eigenvectors [3,3])"""
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 3)
    nrm = np.ascontiguousarray(nrm, np.float32).reshape(-1, 3)
    x, mat = np.empty(3, np.float32), np.empty(18, np.float32)
    rk = host_lib().mcdh_qef(_p(pts), _p(nrm), len(pts), _p(np.asarray(lo, np.float32)), _p(np.asarray(hi, np.float32)), _p(x), _p(mat))
    return x, rk, mat[:9].reshape(3, 3), mat[9:].reshape(3, 3)


def active_cubes(d):
    """flat loop-order indices of the active cubes of a host_dc result (sign change and, with constraints, all 8 corners valid)"""
    s = d["field"] > np.float32(d["iso"])
    M = d["M"]
    corners = [s[dz:dz + M, dy:dy + M, dx:dx + M] for dz in (0, 1) for dy in (0, 1) for dx in (0, 1)]
    anyp = np.logical_or.reduce(corners)
    allp = np.logical_and.reduce(corners)
    act = anyp & ~allp
    if d["valid"] is not None:
        v = d["valid"].astype(bool)
        act &= np.logical_and.reduce([v[dz:dz + M, dy:dy + M, dx:dx + M] for dz in (0, 1) for dy in (0, 1) for dx in (0, 1)])
    return act


def python_quads(d):
    """The quads as integer logic from the active cubes and the signs, independent of the C++: triangle list [T,3] uint32
    (the split reads the host build's vertex positions)."""
    M = d["M"]
    s = d["field"] > np.float32(d["iso"])
    act = active_cubes(d)
    index = -np.ones(M ** 3, np.int64)
    index[np.flatnonzero(act.ravel())] = np.arange(np.count_nonzero(act))
    index = index.reshape(M, M, M)
    recs = []  # (owner index, axis, four vertex indices in winding order)
    cyc, rev = [(0, 0), (1, 0), (1, 1), (0, 1)], [(0, 0), (0, 1), (1, 1), (1, 0)]
    for k in range(M):
        for j in range(M):
            for i in range(M):
                if index[k, j, i] < 0:
                    continue
                # the three edges through the corner (i+1, j+1, k+1): x from (i, j+1, k+1), y from (i+1, j, k+1), z from (i+1, j+1, k)
                for axis, lo, hi in ((0, (k + 1, j + 1, i), (k + 1, j + 1, i + 1)), (1, (k + 1, j, i + 1), (k + 1, j + 1, i + 1)),
                                     (2, (k, j + 1, i + 1), (k + 1, j + 1, i + 1))):
                    if s[lo] == s[hi]:
                        continue
                    w = []
                    for a, b in (rev if s[lo] else cyc):
                        ci, cj, ck = ((i, j + a, k + b), (i + b, j, k + a), (i + a, j + b, k))[axis]
                        w.append(index[ck, cj, ci] if max(ci, cj, ck) < M else -1)
                    if min(w) >= 0:
                        recs.append(w)
    vl = d["vl"]
    out = []
    for w in recs:
        p = vl[w]
        a, b = p[2] - p[0], p[3] - p[1]
        d02 = (a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]
        d13 = (b[0] * b[0] + b[1] * b[1]) + b[2] * b[2]
        if not d13 < d02:
            out += [(w[0], w[1], w[2]), (w[0], w[2], w[3])]
        else:
            out += [(w[0], w[1], w[3]), (w[1], w[2], w[3])]
    return np.array(out, np.uint32).reshape(-1, 3)


def edge_use(tl):
    """{undirected edge: number of triangles using it}"""
    e = np.sort(np.concatenate([tl[:, [0, 1]], tl[:, [1, 2]], tl[:, [2, 0]]]).astype(np.int64), axis=1)
    u, n = np.unique(e[:, 0] * (1 << 32) + e[:, 1], return_counts=True)
    return u, n


def euler(tl):
    u, _ = edge_use(tl)
    return len(np.unique(tl)) - len(u) + len(tl)


def nonmanifold_edges(tl):
    _, n = edge_use(tl)
    return int(np.count_nonzero(n != 2))


def signed_volume(vl, tl):
    v = vl.astype(np.float64)
    a, b, c = v[tl[:, 0]], v[tl[:, 1]], v[tl[:, 2]]
    return float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0)


def run_dc(mcb, eq, step, scale=(1.0, 1.0, 1.0), normals=0, field_mode=None, jit=None, grammar=F, cons=(), iso=0.0, timing=None):
    """One polygonisation in MCB_MESH_DC mode: dict with counts, vl[V,3], tl[T,3], vn[V,3] (normals != 0)."""
    ctx = mcb.Context(0)
    try:
        ctx.set_mesh_mode(MESH_DC)
        ctx.set_grammar(grammar)
        assert ctx.set_equation(eq) == 0
        ctx.set_grid_step(step)
        ctx.set_scaling(*scale)
        ctx.set_surface_constant(iso)
        for i, (lhs, op, rhs) in enumerate(cons):
            assert ctx.set_equation(lhs, slot=i + 1) == 0
            assert ctx.set_constraint(i, op, rhs, True) == 0
        if field_mode is not None:
            ctx.set_field_mode(field_mode)
        if jit is not None:
            ctx.set_jit(jit)
            if jit == mcb.JIT_ON:
                ctx.jit_wait()
        if timing is not None:
            ctx.set_stage_timing(timing)
        ctx.set_normals(normals)
        cnt = ctx.polygonise()
        r = ctx.get_indexed_mesh(normals=normals != 0)
        out = {"counts": cnt, "vl": r[0], "tl": r[1], "vn": r[2] if normals else None}
    finally:
        ctx.close()
    return out
