"""Shared material of the analytic-normal tests (test_normals_host.py, test_gpu_normals.py): the host build of the product's
rules (tests/cpp/normals_host.cpp), the normalisation restated in numpy float32, and an independent float64 forward-mode
evaluator over the reference's postfix text (mcb.postfix), with a stated rule for points where the gradient is
ill-conditioned."""
import ctypes as C
import os
import re

import numpy as np

from .functions_common import CSRC, GRAMMAR_FUNCTIONS, ORACLE, ROOT, _build, _headers

NORMALS_ANALYTIC = 3
SPECIAL = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.0, -1.0, 0.5, -2.5, 3.4e38, -3.4e38, np.inf, -np.inf, np.nan,
                    0.37, -7.25], np.float32)

_host = None


def host_lib():
    """tests/cpp/normals_host.cpp: mcb_interp_grad_scalar / mcb_grad_normalise compiled by g++ on the product's lowering"""
    global _host
    if _host is None:
        so = _build("libmcb_normals_host.so", [os.path.join(ROOT, "tests", "cpp", "normals_host.cpp"), os.path.join(CSRC, "mcb_lower.cpp")],
                    _headers() + [os.path.join(ORACLE, "host_interp.cpp"), os.path.join(ORACLE, "host_interp_fn.cpp")],
                    ["g++", "-std=c++17", "-O2", "-ffp-contract=off"], shared=True)
        L = C.CDLL(so)
        vp, f = C.c_void_p, C.c_float
        L.mcoh_set_grammar.argtypes = [C.c_int]
        L.mcnh_eval.argtypes = [C.c_char_p, vp, C.c_long, f, f, f, vp, vp, vp, vp]
        L.mcnh_normalise.argtypes = [vp, vp, C.c_long]
        _host = L
    return _host


def host_eval(eq, xyz, scale=(1.0, 1.0, 1.0), grammar=GRAMMAR_FUNCTIONS):
    """(value, plain, grad[n,3], normal[n,3]) of the host build at the unscaled points xyz[n,3]"""
    L = host_lib()
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    n = len(xyz)
    value, plain = np.empty(n, np.float32), np.empty(n, np.float32)
    grad, nrm = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32)
    L.mcoh_set_grammar(grammar)
    rc = L.mcnh_eval(eq.encode(), xyz.ctypes.data, n, *[C.c_float(s) for s in scale], value.ctypes.data, plain.ctypes.data,
                     grad.ctypes.data, nrm.ctypes.data)
    assert rc == 0, (eq, rc)
    return value, plain, grad, nrm


def host_normalise(g):
    L = host_lib()
    g = np.ascontiguousarray(g, np.float32).reshape(-1, 3)
    out = np.empty_like(g)
    L.mcnh_normalise(g.ctypes.data, out.ctypes.data, len(g))
    return out


def normalise32(g):
    """The normalisation of include/mcb.h restated in numpy float32: m = max |g_i|; 0 when m is 0, inf or NaN or a component
    is NaN; u = g/m, d = ux*ux + uy*uy + uz*uz, n = u * (1/sqrt(d))."""
    g = np.asarray(g, np.float32).reshape(-1, 3)
    with np.errstate(all="ignore"):
        m = np.max(np.abs(g), axis=1)
        bad = np.isnan(g).any(axis=1) | ~(m > 0) | np.isinf(m)
        u = g / np.where(bad, np.float32(1), m)[:, None]
        d = u[:, 0] * u[:, 0] + u[:, 1] * u[:, 1]
        d = d + u[:, 2] * u[:, 2]
        r = np.float32(1) / np.sqrt(d)
        n = u * r[:, None]
    n[bad] = 0
    return n.astype(np.float32)


# ---- independent float64 reference -----------------------------------------------------------------------------------
_NUM = re.compile(r"\d+\.?\d*|\.\d+")
_BIN = {"+", "-", "*", "/", "^", "min", "max"}
_UN = {"NEG", "sin", "cos", "sqrt", "abs"}


def postfix_program(mcb, eq, grammar=GRAMMAR_FUNCTIONS):
    """The reference's postfix of eq as tokens, its numbers replaced by the fp32 values of the equation's literals (the
    text prints them with 6 digits; operands keep their left-to-right order, which is checked)."""
    toks = mcb.postfix(eq, grammar=grammar).split()
    lits = [np.float32(t) for t in _NUM.findall(eq.lower())]
    out, j = [], 0
    for t in toks:
        if t in _BIN or t in _UN or t in ("x", "y", "z"):
            out.append(t)
            continue
        v = float(t)
        assert j < len(lits) and abs(float(lits[j]) - v) <= 1e-5 * max(1.0, abs(v)), (eq, t, lits)
        out.append(float(lits[j]))
        j += 1
    assert j == len(lits), (eq, lits)
    return out


def grad64(prog, xyz, scale=(1.0, 1.0, 1.0), perturb=None):
    """(value, gradient[n,3]) in float64 by forward-mode dual numbers, with respect to the unscaled coordinates, at the
    scaled coordinates the product evaluates (fp32 sx*x).  Same conventions as the product: a is the left operand; min /
    max take the gradient of the operand they return, the mean on a tie, the other operand's when one is NaN; abs takes
    the sign bit.  perturb = rng: every intermediate result (value and partials) is multiplied by 1 +- 2^-22."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    n = len(xyz)
    s32 = np.asarray(scale, np.float32)
    X = (xyz * s32).astype(np.float64)
    st = []

    def jig(v, g):
        if perturb is not None:
            v = v * (1 + 2.0 ** -22 * perturb.choice([-1.0, 1.0], size=v.shape))
            g = g * (1 + 2.0 ** -22 * perturb.choice([-1.0, 1.0], size=g.shape))
        return v, g

    with np.errstate(all="ignore"):
        for t in prog:
            if isinstance(t, float):
                st.append((np.full(n, t), np.zeros((n, 3))))
                continue
            if t in ("x", "y", "z"):
                k = "xyz".index(t)
                g = np.zeros((n, 3))
                g[:, k] = float(s32[k])
                st.append((X[:, k].copy(), g))
                continue
            if t in _UN:
                a, ga = st.pop()
                if t == "NEG":
                    v, g = -a, -ga
                elif t == "sin":
                    v, g = np.sin(a), np.cos(a)[:, None] * ga
                elif t == "cos":
                    v, g = np.cos(a), -np.sin(a)[:, None] * ga
                elif t == "sqrt":
                    v = np.sqrt(a)
                    g = ga / (2 * v)[:, None]
                else:
                    v = np.abs(a)
                    g = np.where(np.signbit(a)[:, None], -ga, ga)
                st.append(jig(v, g))
                continue
            b, gb = st.pop()
            a, ga = st.pop()
            if t == "+":
                v, g = a + b, ga + gb
            elif t == "-":
                v, g = a - b, ga - gb
            elif t == "*":
                v, g = a * b, ga * b[:, None] + a[:, None] * gb
            elif t == "/":
                v = a / b
                g = (ga - v[:, None] * gb) / b[:, None]
            elif t == "^":
                v = np.power(a, b)
                const_b = np.all(gb == 0, axis=1)
                g_c = (b * np.power(a, b - 1))[:, None] * ga
                g_v = v[:, None] * (np.log(a)[:, None] * gb + (b / a)[:, None] * ga)
                g = np.where(const_b[:, None], g_c, g_v)
            else:
                v = np.fmin(a, b) if t == "min" else np.fmax(a, b)
                pick_a = (a == v) & (b != v) | np.isnan(b)
                pick_b = (b == v) & (a != v) | np.isnan(a)
                g = np.where(pick_a[:, None], ga, np.where(pick_b[:, None], gb, (ga + gb) * 0.5))
            st.append(jig(v, g))
    assert len(st) == 1
    return st[0]


def unit64(g):
    with np.errstate(all="ignore"):
        return g / np.linalg.norm(g, axis=1)[:, None]


def well_conditioned(prog, xyz, scale=(1.0, 1.0, 1.0), seed=0):
    """The stated rule for comparing fp32 with float64: a point is kept when its float64 gradient is finite and non-zero and
    its unit normal moves by at most 1e-6 (per component) when every intermediate result is perturbed by a relative 2^-22
    (a few fp32 ulps), in each of two random draws.  Kinks (min / max / abs near a switch), cancellations and powers of
    negative bases fail it."""
    v, g = grad64(prog, xyz, scale)
    u = unit64(g)
    ok = np.isfinite(v) & np.isfinite(g).all(axis=1) & (np.abs(g).max(axis=1) > 0)
    rng = np.random.default_rng(seed)
    for _ in range(2):
        _, gp = grad64(prog, xyz, scale, perturb=rng)
        with np.errstate(invalid="ignore"):
            ok &= np.isfinite(gp).all(axis=1) & (np.abs(unit64(gp) - u).max(axis=1) <= 1e-6)
    return ok, u


# ---- the pipeline in each normals mode ----------------------------------------------------------------------------------
def run_mesh(mcb, eq, step, scale=(1.0, 1.0, 1.0), normals=NORMALS_ANALYTIC, field_mode=None, jit=None, grammar=GRAMMAR_FUNCTIONS,
             slab=None, seed=None, levels=None, iso=0.0):
    """One polygonisation in soup + indexed mode: dict with counts, pos[T,3,4], nrm[T,3,4], vl[V,3], tl[T,3], vn[V,3]."""
    ctx = mcb.Context(0)
    try:
        ctx.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        ctx.set_grammar(grammar)
        assert ctx.set_equation(eq) == 0
        ctx.set_grid_step(step)
        ctx.set_scaling(*scale)
        ctx.set_surface_constant(iso)
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
        if levels is not None:
            assert ctx.set_repeat(True, levels) == 0
        ctx.set_normals(normals)
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


def soup_matches_welded(m):
    """(soup normals, welded normals) at the soup vertices whose position bits equal their welded vertex's"""
    p = m["pos"][:, :, :3].reshape(-1, 3)
    idx = m["tl"].reshape(-1).astype(np.int64)
    w = m["vl"][idx]
    same = (p.view(np.uint32) == w.view(np.uint32)).all(axis=1)
    return m["nrm"][:, :, :3].reshape(-1, 3)[same], m["vn"][idx][same], int(same.sum())
