"""Shared material of the refined-vertex tests (test_refine_host.py, test_gpu_refine.py): the host build of the product's
refinement (tests/cpp/refine_host.cpp), crossing edges of an equation on the grid with their linear points, an independent
float64 root along an edge (scipy.optimize.brentq on a float64 evaluator of the reference's postfix text), and the
pipeline with refinement on or off."""
import ctypes as C
import os

import numpy as np

from .functions_common import CSRC, GRAMMAR_FUNCTIONS, ORACLE, ROOT, _build, _headers
from .normals_common import grad64

REFINE_EVALS = 40  # MCB_REFINE_EVALS, csrc/mcb_refine.h
SAME_SIGN = -1     # MCB_REFINE_SAME_SIGN

_host = None


def host_lib():
    """tests/cpp/refine_host.cpp: mcb_refine_vertex compiled by g++ on the product's lowering"""
    global _host
    if _host is None:
        so = _build("libmcb_refine_host.so", [os.path.join(ROOT, "tests", "cpp", "refine_host.cpp"), os.path.join(CSRC, "mcb_lower.cpp")],
                    _headers() + [os.path.join(CSRC, "mcb_refine.h"), os.path.join(ORACLE, "host_interp.cpp"),
                                  os.path.join(ORACLE, "host_interp_fn.cpp")],
                    ["g++", "-std=c++17", "-O2", "-ffp-contract=off"], shared=True)
        L = C.CDLL(so)
        vp, f = C.c_void_p, C.c_float
        L.mcoh_set_grammar.argtypes = [C.c_int]
        L.mcrh_refine.argtypes = [C.c_char_p, vp, C.c_int, f, f, f, f, vp, C.c_long, vp, vp, vp]
        L.mcrh_eval.argtypes = [C.c_char_p, vp, C.c_long, f, f, f, vp]
        L.mcrh_interp.argtypes = [f, f, f]
        L.mcrh_interp.restype = f
        _host = L
    return _host


def host_refine(eq, c, xyz, iso=0.0, scale=(1.0, 1.0, 1.0), grammar=GRAMMAR_FUNCTIONS):
    """(refined[n,3], evals[n], bracket[n,2]) of the host build for the points xyz[n,3] on the coordinate table c[0..M]"""
    L = host_lib()
    c = np.ascontiguousarray(c, np.float32)
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    n = len(xyz)
    out, ev, br = np.empty((n, 3), np.float32), np.empty(n, np.int32), np.empty((n, 2), np.float32)
    L.mcoh_set_grammar(grammar)
    rc = L.mcrh_refine(eq.encode(), c.ctypes.data, len(c) - 1, C.c_float(iso), *[C.c_float(s) for s in scale], xyz.ctypes.data, n,
                       out.ctypes.data, ev.ctypes.data, br.ctypes.data)
    assert rc == 0, (eq, rc)
    return out, ev, br


def host_f(eq, xyz, scale=(1.0, 1.0, 1.0), grammar=GRAMMAR_FUNCTIONS):
    """the point program at (sx*x, sy*y, sz*z), fp32, as mcb_eval_points(apply_scale=1) computes it"""
    L = host_lib()
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    out = np.empty(len(xyz), np.float32)
    L.mcoh_set_grammar(grammar)
    assert L.mcrh_eval(eq.encode(), xyz.ctypes.data, len(xyz), *[C.c_float(s) for s in scale], out.ctypes.data) == 0, eq
    return out


def interp_ref(xs, xe, t):
    return np.float32(host_lib().mcrh_interp(C.c_float(xs), C.c_float(xe), C.c_float(t)))


def crossing_edges(eq, c, n, rng, iso=0.0, scale=(1.0, 1.0, 1.0), grammar=GRAMMAR_FUNCTIONS):
    """Up to n random grid edges of the table c that the surface crosses (s(f) differs at the two ends, s(v) = v > iso).
    Returns (lower end[k,3], axis[k], index i of the lower coordinate[k], f at the lower and upper end)."""
    M = len(c) - 1
    ijk = rng.integers(0, M + 1, (8 * n + 64, 3))
    ax = rng.integers(0, 3, len(ijk))
    ok = ijk[np.arange(len(ijk)), ax] < M
    ijk, ax = ijk[ok], ax[ok]
    lo = c[ijk].astype(np.float32)
    hi = lo.copy()
    hi[np.arange(len(hi)), ax] = c[ijk[np.arange(len(hi)), ax] + 1]
    flo, fhi = host_f(eq, lo, scale, grammar), host_f(eq, hi, scale, grammar)
    x = (flo > np.float32(iso)) != (fhi > np.float32(iso))
    k = np.flatnonzero(x)[:n]
    return lo[k], ax[k], ijk[k, ax[k]], flo[k], fhi[k]


def linear_points(lo, ax, ilo, flo, fhi, c, iso=0.0):
    """The edge's crossing point as the emitter computes it, from the lower end (the canonical linear point) and from the
    upper end (what a cube whose edge runs the other way interpolates)"""
    fwd, bwd = lo.copy(), lo.copy()
    iso = np.float32(iso)
    with np.errstate(all="ignore"):
        for r in range(len(lo)):
            a, b = c[ilo[r]], c[ilo[r] + 1]
            fwd[r, ax[r]] = interp_ref(a, b, (iso - flo[r]) / (fhi[r] - flo[r]))
            bwd[r, ax[r]] = interp_ref(b, a, (iso - fhi[r]) / (flo[r] - fhi[r]))
    return fwd, bwd


# ---- independent float64 reference -----------------------------------------------------------------------------------
def value64(prog, X):
    """the postfix program (normals_common.postfix_program) in float64 at the scaled points X[n,3] (float64)"""
    X = np.asarray(X, np.float64).reshape(-1, 3)
    st = []
    with np.errstate(all="ignore"):
        for t in prog:
            if isinstance(t, float):
                st.append(np.full(len(X), t))
            elif t in ("x", "y", "z"):
                st.append(X[:, "xyz".index(t)].copy())
            elif t in ("NEG", "sin", "cos", "sqrt", "abs"):
                a = st.pop()
                st.append({"NEG": np.negative, "sin": np.sin, "cos": np.cos, "sqrt": np.sqrt, "abs": np.abs}[t](a))
            else:
                b, a = st.pop(), st.pop()
                st.append({"+": np.add, "-": np.subtract, "*": np.multiply, "/": np.divide, "^": np.power,
                           "min": np.fmin, "max": np.fmax}[t](a, b))
    assert len(st) == 1
    return st[0]


def root64(prog, p, ax, a, b, iso=0.0, scale=(1.0, 1.0, 1.0)):
    """The float64 root of f - iso along the edge [a, b] of axis ax through p (scipy brentq), or None when f64 does not
    change sign there"""
    from scipy.optimize import brentq
    s = np.asarray(scale, np.float32).astype(np.float64)
    P = np.asarray(p, np.float64).copy()

    def g(t):
        P[ax] = t
        return float(value64(prog, (P * s)[None])[0]) - iso
    ga, gb = g(float(a)), g(float(b))
    if not (np.isfinite(ga) and np.isfinite(gb)) or ga * gb > 0:
        return None
    if ga == 0 or gb == 0:
        return float(a) if ga == 0 else float(b)
    return brentq(g, float(a), float(b), xtol=1e-15, rtol=1e-15, maxiter=200)


def well_conditioned_root(prog, r, p, ax, scale=(1.0, 1.0, 1.0), seed=0):
    """The stated rule for comparing a refined coordinate with the float64 root r: at the fp32 point nearest r, the fp32
    evaluation error of f (estimated as the largest change of the float64 value when every intermediate result is
    perturbed by a relative 2^-22, two random draws) divided by |df/d(axis)| there must be at most 1e-6, and that
    derivative finite and non-zero.  Returns (kept, that bound)."""
    q = np.asarray(p, np.float32).copy()
    q[ax] = np.float32(r)
    v, g = grad64(prog, q[None], scale)
    d = abs(float(g[0, ax]))
    rng = np.random.default_rng(seed)
    noise = 0.0
    for _ in range(2):
        vp, _ = grad64(prog, q[None], scale, perturb=rng)
        noise = max(noise, abs(float(vp[0]) - float(v[0])))
    if not (np.isfinite(d) and d > 0 and np.isfinite(noise)):
        return False, np.inf
    bound = noise / d
    return bound <= 1e-6, bound


# ---- the pipeline with refinement on or off ------------------------------------------------------------------------------
def run_refined(mcb, eq, step, scale=(1.0, 1.0, 1.0), refine=True, normals=0, field_mode=None, jit=None, grammar=GRAMMAR_FUNCTIONS,
                slab=None, seed=None, cons=(), iso=0.0):
    """One polygonisation in soup + indexed mode: dict with counts, pos[T,3,4], nrm, vl[V,3], tl[T,3], vn."""
    ctx = mcb.Context(0)
    try:
        ctx.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
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
        if slab is not None:
            ctx.set_slab(*slab)
        if seed is not None:
            assert ctx.set_seed(True, *seed) == 0
        ctx.set_normals(normals)
        ctx.set_refine_vertices(refine)
        cnt = ctx.polygonise()
        pos, nrm = ctx.get_mesh(normals=normals in (1, 3))
        r = ctx.get_indexed_mesh(normals=normals != 0)
        out = {"counts": cnt, "pos": pos, "nrm": nrm, "vl": r[0], "tl": r[1], "vn": r[2] if normals else None,
               "jit": int(cnt.jit), "field_mode": int(cnt.field_mode)}
    finally:
        ctx.close()
    return out


def counts_tuple(c):
    return (int(c.cubes), int(c.active), int(c.triangles), int(c.vertices), int(c.ambiguous), int(c.redirected))
