"""CPU tier of min( max( in the function grammar (unions, intersections and differences of implicit shapes): the grammar
rules, the listings of every older equation unchanged, the arithmetic against its definition and the oracle's own
restatement (oracle/mc_oracle_csg.c), identities, the lowering against the oracle, hoisting, the interval rules against brute
force, the run-time compiled kernels executed on the host and the emulated device pipeline against the oracle's meshes."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from .csg_common import (CSG_BOX_SDF, CSG_EQUATIONS, CSG_LENS, CSG_SPHERE_MINUS_CYLINDER, CSG_UNION2, CSG_UNION8, CsgOracle,
                         csg_oracle_minmax, csg_parse_ok, random_csg_equations)
from .functions_common import FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, host_fn_lib
from .helpers import same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = GRAMMAR_FUNCTIONS

# (equation, tokens, postfix)
CSG_GRAMMAR_TABLE = [
    ("min(x,y)", "min( x , y )", "x y min"),
    ("max(x-y+z,0)", "max( x - y + z , 0 )", "x y z + - 0 max"),
    ("-min(x,y)^2", "NEG min( x , y ) ^ 2", "x y min NEG 2 ^"),
    ("2max(x,y)", "2 * max( x , y )", "2 x y max *"),
    ("xmax(y,z)", "x * max( y , z )", "x y z max *"),
    ("min(x,-y)", "min( x , NEG y )", "x y NEG min"),
    ("min(min(x,y),z)", "min( min( x , y ) , z )", "x y min z min"),
    ("min(x,y)(z)", "min( x , y ) * ( z )", "x y min z *"),
    ("max(abs(x)-0.5,0)^2", "max( abs( x ) - 0.5 , 0 ) ^ 2", "x abs 0.5 - 0 max 2 ^"),
    ("min (x , y)", "min( x , y )", "x y min"),
    ("xmin(y,z)", "x * min( y , z )", "x y z min *"),
    ("min(x,y)max(y,z)", "min( x , y ) * max( y , z )", "x y min y z max *"),
    ("sin(min(x,2y))", "sin( min( x , 2 * y ) )", "x 2 y * min sin"),
    ("min(-x,(y))", "min( NEG x , ( y ) )", "x NEG y min"),
]
CSG_REJECTED = ["min(x)", "min(x,y,z)", "min(,x)", "min(x,)", "min(x,+y)", "min(,)", "min()", "min(x,y", "(x,y)", "x,y",
                "min(x,y),z", "sin(x,y)", "MIN(x,y)", "Min(x,y)", "maxx(y,z)", "mn(x,y)", "ma(x,y)", "MAX(x,y)", "min(x,y)),",
                "min((x,y))", "min(x,-)", "min(x,y-)", "min(-,y)", "max(x;y)", "min[x,y]", "min(x,,y)"]


@pytest.mark.parametrize("eq,toks,pf", CSG_GRAMMAR_TABLE)
def test_csg_grammar_table(mcb, eq, toks, pf):
    assert mcb.parse_ok(eq, grammar=F) and csg_parse_ok(eq), eq
    assert mcb.tokens(eq, grammar=F) == toks
    assert mcb.postfix(eq, grammar=F) == pf
    assert not mcb.parse_ok(eq) and not mcb.parse_ok(eq, grammar=0)  # the reference grammar has no names and no ','


@pytest.mark.parametrize("eq", CSG_REJECTED)
def test_csg_rejections(mcb, eq):
    assert not mcb.parse_ok(eq, grammar=F), eq
    assert not csg_parse_ok(eq), eq  # the oracle's own restatement of the grammar
    assert not mcb.parse_ok(eq), eq
    assert mcb.lib.mcb_parse(eq.encode()) == mcb.MCB_E_PARSE


def test_grammar_two_is_still_an_argument_error(mcb):
    buf = C.create_string_buffer(64)
    assert mcb.lib.mcb_grammar_text(b"min(x,y)", 2, 0, buf, 64) == mcb.MCB_E_ARG


def test_listings_of_older_equations_are_unchanged():
    """Tokens, postfix, the four mcb_disassemble listings and the run-time compiled source (the compile cache key) of every
    golden equation (both grammars) and every named function equation: their hashes before min( max( existed
    (tests/golden/listing_hashes.json) equal the ones now."""
    import hashlib
    import importlib
    from .helpers import load_meta
    mcb = importlib.import_module("marching-cube-for-implicit-surfaces_b200")
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "listing_hashes.json")))
    meta = load_meta(np.load(os.path.join(ROOT, "tests", "golden", "cases.npz")))
    ref = sorted(set([c["eq"] for c in meta.values()] + [l for c in meta.values() for (l, _, _) in c.get("cons", [])]))
    assert sorted(want["0"]) == ref and sorted(want["1"]) == sorted(set(ref + FUNCTION_EQUATIONS))
    for grammar, eqs in want.items():
        grammar = int(grammar)
        for eq, digest in eqs.items():
            h = hashlib.sha256()
            h.update(mcb.tokens(eq, grammar=grammar).encode() + b"\n" + mcb.postfix(eq, grammar=grammar).encode() + b"\n")
            for which in (0, 1, 2, 3):
                h.update(mcb.disassemble(eq, which, grammar=grammar).encode() + b"\n")
            h.update(mcb.jit_check(eq, cap=1 << 20, grammar=grammar)[1].encode())
            assert h.hexdigest() == digest, (grammar, eq)


# ---- arithmetic ----------------------------------------------------------------------------------------------------
def special_pairs():
    """every pair drawn from {+-0, +-smallest denormal, +-1, +-FLT_MAX, +-inf, NaN, a few random values}"""
    f32 = np.float32
    vals = [f32(0.0), f32(-0.0), np.uint32(1).view(f32), np.uint32(0x80000001).view(f32), f32(1), f32(-1),
            np.finfo(f32).max, -np.finfo(f32).max, f32(np.inf), f32(-np.inf), f32(np.nan),
            np.uint32(0x7fc0abcd).view(f32), f32(0.37), f32(-2.5e-3), f32(12345.678)]
    v = np.array(vals, np.float32)
    a, b = np.meshgrid(v, v, indexing="ij")
    return a.ravel().copy(), b.ravel().copy()


def definition(a, b, is_max):
    """minimumNumber / maximumNumber in numpy: a NaN operand ignored, -0 < +0, otherwise the smaller / larger operand"""
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    pick_a = (a > b) if is_max else (a < b)
    r = np.where(pick_a, a, b)
    eq = a == b
    zero_sign = np.where(np.signbit(a) != is_max, a, b)  # among +0 / -0: min takes the negative one, max the positive
    r = np.where(eq, zero_sign, r)
    r = np.where(np.isnan(a), b, r)
    r = np.where(np.isnan(b) & ~np.isnan(a), a, r)
    return r.astype(np.float32)


@pytest.fixture(scope="module")
def host():
    """oracle/host_interp.cpp's runners of the product's bytecode, lowering under the function grammar"""
    return host_fn_lib()


def _product_eval(host, eq, a, b):
    pts = np.stack([a, b, np.zeros_like(a)], 1).astype(np.float32)
    out = np.empty(len(a), np.float32)
    assert host.mcoh_eval_points(eq.encode(), pts.ctypes.data, out.ctypes.data, len(a)) == 0, eq
    return out


def test_min_max_on_special_pairs_equal_the_definition_and_the_oracle(host):
    """mcb_min / mcb_max (the host build of csrc/mcb_bytecode.h, through the point interpreter: `min(x,y)` is
    PUSH_X PUSH_Y MIN) against the numpy statement of the definition, the oracle's plain-C restatement called directly and
    the oracle's walk; sign of zero included, NaN as a class."""
    a, b = special_pairs()
    omin, omax = csg_oracle_minmax()
    for name, is_max, ofn in (("min", False, omin), ("max", True, omax)):
        got = _product_eval(host, "%s(x,y)" % name, a, b)
        assert same_bits(got, definition(a, b, is_max)), name
        assert same_bits(got, np.array([ofn(float(x), float(y)) for x, y in zip(a, b)], np.float32)), name
        pts = np.stack([a, b, np.zeros_like(a)], 1).astype(np.float32)
        assert same_bits(got, CsgOracle("%s(x,y)" % name).eval_points(pts)), name
    # the cases the definition singles out, spelt out
    z, nz = np.float32(0.0), np.float32(-0.0)
    assert np.signbit(_product_eval(host, "min(x,y)", np.array([z, nz]), np.array([nz, z]))).all()
    assert not np.signbit(_product_eval(host, "max(x,y)", np.array([z, nz]), np.array([nz, z]))).any()
    nan = np.float32(np.nan)
    assert np.isnan(_product_eval(host, "min(x,y)", np.array([nan]), np.array([nan]))).all()


def test_min_max_on_1e7_random_bit_pairs(host):
    rng = np.random.default_rng(2024)
    n = 10 ** 7
    a = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32).view(np.float32)
    b = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32).view(np.float32)
    b[: n // 10] = a[: n // 10]  # equal operands
    b[n // 10: n // 5] = -a[n // 10: n // 5]
    for name, is_max in (("min", False), ("max", True)):
        got = _product_eval(host, "%s(x,y)" % name, a, b)
        assert same_bits(got, definition(a, b, is_max)), name
        assert same_bits(got, _product_eval(host, "%s(y,x)" % name, a, b)), name  # commutative


def test_identities_bit_for_bit(mcb, host):
    """min(A,B) = min(B,A), max(A,B) = -min(-A,-B), abs(E) = max(E,-E), min(A,A) = A, at random points, NaN as a class"""
    rng = np.random.default_rng(17)
    pts = (rng.random((400, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    pts[:8] = 0
    pts[8:16] = -1
    exprs = CSG_EQUATIONS + FUNCTION_EQUATIONS + random_csg_equations(mcb, 3, 60, max_len=70)

    def ev(eq):
        assert mcb.parse_ok(eq, grammar=F), eq
        out = np.empty(len(pts), np.float32)
        assert host.mcoh_eval_points(eq.encode(), pts.ctypes.data, out.ctypes.data, len(pts)) == 0, eq
        return out

    for i in range(0, len(exprs) - 1):
        A, B = exprs[i], exprs[i + 1]
        assert same_bits(ev("min(%s,%s)" % (A, B)), ev("min(%s,%s)" % (B, A))), (A, B)
        assert same_bits(ev("max(%s,%s)" % (A, B)), ev("-min(-(%s),-(%s))" % (A, B))), (A, B)
        assert same_bits(ev("abs(%s)" % A), ev("max(%s,-(%s))" % (A, A))), A
        assert same_bits(ev("min(%s,%s)" % (A, A)), ev(A)), A


# ---- lowering --------------------------------------------------------------------------------------------------------
def test_csg_lowering_bit_exact_against_the_oracle(mcb, host):
    """About 500 random CSG equations and the named shapes: the product's bytecode run by the host build of its
    interpreters (folded constants, hoisted axis tables, fused grid form) against the oracle's own tokenizer and walk, at
    random points and on a tensor grid; each equation also as a constraint left-hand side of the oracle."""
    rng = np.random.default_rng(321)
    pts = (rng.random((300, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    pts[:8] = 0
    pts[8:16] = -1
    pts[16:24] = np.float32(0.5)
    cx = np.linspace(-1.1, 1.2, 9, dtype=np.float32)
    cy = np.linspace(-0.9, 1.3, 6, dtype=np.float32)
    cz = np.linspace(-1, 1, 4, dtype=np.float32)
    Z, Y, X = np.meshgrid(cz, cy, cx, indexing="ij")
    gp = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    eqs = CSG_EQUATIONS + ["min(2,3)+x", "max(sqrt(-1),x)", "min(sqrt(x),0.5)", "max(x,y)^2", "min(x,max(y,min(z,0.1)))",
                           "-min(x,y)^2", "max(x-y+z,0)"] + random_csg_equations(mcb, 99, 490)
    for eq in eqs:
        o = CsgOracle(eq)
        assert o.set_equation(1, eq)
        out = np.empty(len(pts), np.float32)
        assert host.mcoh_eval_points(eq.encode(), pts.ctypes.data, out.ctypes.data, len(pts)) == 0, eq
        assert same_bits(out, o.eval_points(pts)), eq
        assert same_bits(out, o.eval_points(pts, slot=1)), eq
        g = np.empty(len(gp), np.float32)
        assert host.mcoh_eval_grid(eq.encode(), cx.ctypes.data, len(cx), cy.ctypes.data, len(cy), cz.ctypes.data, len(cz),
                                   g.ctypes.data) == 0, eq
        assert same_bits(g, o.eval_points(gp)), eq


def test_min_max_subtrees_are_folded_and_hoisted(mcb):
    """Each max(abs(.)-c,0)^2 of the box SDF is one axis table, so its grid program has no MIN / MAX word; a constant
    min folds into the constant pool; the union of spheres keeps its min words between table sums and needs no powf."""
    fused = mcb.disassemble(CSG_BOX_SDF, 3, grammar=F)
    assert "MIN" not in fused and "MAX" not in fused and "POW" not in fused, fused
    slots = mcb.disassemble(CSG_BOX_SDF, 2, grammar=F)
    assert slots.count("MAX") == 3 and slots.count("TX") == 1 and slots.count("TY") == 1 and slots.count("TZ") == 1, slots
    assert mcb.disassemble("min(2,3)+x", 3, grammar=F) == "LOAD TX0"
    assert mcb.disassemble("min(2,3)+x", 2, grammar=F).startswith("K2: K0 K1 MIN")
    assert mcb.disassemble("min(2,3)", 1, grammar=F) == "K2"
    u8 = mcb.disassemble(CSG_UNION8, 3, grammar=F)
    assert u8.count("MIN") == 7 and "POW" not in u8 and "SQRT" not in u8, u8
    assert mcb.disassemble(CSG_LENS, 3, grammar=F).endswith("MAX POP")


# ---- interval proof ----------------------------------------------------------------------------------------------------
INTERVAL_EQUATIONS = CSG_EQUATIONS + ["min(sqrt(x),0.5)", "max(sqrt(x+y)-0.3,z)", "min(x,y)-max(z,0.2)", "max(abs(x),abs(y))-0.5+z",
                                      "min(sin(20(x+y+z)),0.5z)", "max(x*y,-(z^2))", "min(1/x,y)", "max(x^3,y)+min(z,0)"]


@pytest.mark.parametrize("eq", INTERVAL_EQUATIONS)
def test_csg_interval_rules_never_prove_wrongly(host, eq):
    n = 33
    c = np.linspace(-1.05, 1.05, n, dtype=np.float32)
    for bs in ((4, 4, 4), (8, 2, 16), (2, 2, 2)):
        for iso in (0.0, 0.1, -0.25):
            st = np.zeros(6, np.int64)
            assert host.mcoh_interval_check(eq.encode(), c.ctypes.data, c.ctypes.data, c.ctypes.data, n, *bs,
                                            C.c_float(iso), st.ctypes.data) == 0
            assert st[4] == 0 and st[5] == 0, (eq, bs, iso, st)


def _undecided(host, eq, c, bs, iso):
    st = np.zeros(6, np.int64)
    assert host.mcoh_interval_check(eq.encode(), c.ctypes.data, c.ctypes.data, c.ctypes.data, len(c), *bs, C.c_float(iso),
                                    st.ctypes.data) == 0
    assert st[4] == 0 and st[5] == 0
    return int(st[0] - st[1] - st[2]), int(st[1] + st[2])


@pytest.mark.parametrize("a,b", [("sqrt(x^2+y^2+z^2)-0.5", "sqrt((x-0.45)^2+y^2+z^2)-0.35"), ("x+y", "z-0.3"),
                                 ("sqrt(x)-0.2", "y^2-0.1"), ("abs(x)-0.5", "sin(9y)+z")])
def test_min_max_leave_no_more_boxes_undecided_than_their_arguments(host, a, b):
    c = np.linspace(-1, 1, 65, dtype=np.float32)
    ua, _ = _undecided(host, a, c, (4, 4, 4), 0.0)
    ub, _ = _undecided(host, b, c, (4, 4, 4), 0.0)
    for f in ("min", "max"):
        u, decided = _undecided(host, "%s(%s,%s)" % (f, a, b), c, (4, 4, 4), 0.0)
        assert u <= ua + ub, (f, u, ua, ub)
    _, decided = _undecided(host, CSG_BOX_SDF, c, (4, 4, 4), 0.0)
    assert decided > 0


# ---- run-time compiled kernels -------------------------------------------------------------------------------------------
def test_generated_csg_kernels_compile_without_a_gpu(mcb):
    for eq in CSG_EQUATIONS + random_csg_equations(mcb, 7, 8, max_len=80):
        nbytes, src = mcb.jit_check(eq, cap=1 << 20, grammar=F)
        assert nbytes > 1000 and src.count("__launch_bounds__") == 2, eq
    _, src = mcb.jit_check(CSG_UNION8, cap=1 << 20, grammar=F)
    assert '#include "mcb_bytecode.h"' in src and src.count("op_min(") >= 7 and "op_pow(" not in src.split("#define R(e)")[1]
    _, src = mcb.jit_check(CSG_BOX_SDF, cap=1 << 20, grammar=F)  # min / max all hoisted: nothing of them in the source
    assert "mcb_bytecode.h" not in src and "op_max" not in src


def test_generated_csg_kernel_source_executed_on_the_host_equals_the_oracle(mcb, host, tmp_path):
    """The run-time generated CUDA source of CSG programs, compiled by g++ under tests/cpp/jit_host_shim_fn.h and run lane
    by lane (both kernels), equals the oracle's field bit for bit."""
    from .test_host_logic import _HostGrid
    P = 32
    rng = np.random.default_rng(6)
    ax = [np.sort((rng.random(P, dtype=np.float32) * 3 - 1.5).astype(np.float32)) for _ in range(3)]
    eqs = [CSG_UNION2, CSG_LENS, CSG_SPHERE_MINUS_CYLINDER, CSG_UNION8, "min(x*y,z)+max(sqrt(x),y*z)"] + \
        random_csg_equations(mcb, 43, 5, max_len=80)
    shim = os.path.join(ROOT, "tests", "cpp", "jit_host_shim_fn.h")
    tail = open(os.path.join(ROOT, "tests", "cpp", "jit_host_tail.inc")).read()
    for n, eq in enumerate(eqs):
        NV, NZ, kb = ((11, 9, 0), (21, 6, 5), (16, 4, 2))[n % 3]
        Z, Y, X = np.meshgrid(ax[2][kb:kb + NZ], ax[1][:NV], ax[0][:NV], indexing="ij")
        pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
        _, src = mcb.jit_check(eq, cap=1 << 20, grammar=F)
        cpp, so = tmp_path / ("c%d.cpp" % n), tmp_path / ("c%d.so" % n)
        cpp.write_text('#include "%s"\n' % shim + src + tail)
        r = subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-w", "-shared", "-fPIC", "-I", os.path.join(ROOT, mcb.__name__, "csrc"),
                            "-DMCB_GRID_BYTES=%d" % C.sizeof(_HostGrid), "-DMCB_MAX_K=128", "-DMCB_MIN_BLOCKS=8", str(cpp), "-o", str(so)],
                           capture_output=True, text=True)
        assert r.returncode == 0, (eq, r.stderr[:2000])
        L = C.CDLL(str(so))
        L.run_fill.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_int]
        L.run_plane.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        tables = np.zeros(3 * 64 * P + 256, np.float32)
        kpool = np.zeros(128, np.float32)
        spa = host.mcoh_tables(eq.encode(), ax[0].ctypes.data, ax[1].ctypes.data, ax[2].ctypes.data, P, tables.ctypes.data,
                               len(tables) - 256, kpool.ctypes.data)
        assert spa > 0, (eq, spa)
        g = _HostGrid(M=NV - 3, NV=NV, P=P, WP=4, kb=kb, ke=kb + NZ - 3, NZ=NZ, sx=1, sy=1, sz=1, iso=0, repeat=0, rstep=0)
        ref = CsgOracle(eq).eval_points(pts).reshape(NZ, NV, NV)
        nbx, nby, nbz = P // 32, (NV + 3) // 4, (NZ + 3) // 4
        ids = np.arange(nbx * nby * nbz)
        blocks = ((ids % nbx) | ((ids // nbx % nby) << 8) | ((ids // (nbx * nby)) << 20)).astype(np.uint32)
        Fb = np.full((NZ, NV, P), np.nan, np.float32)
        S = np.zeros((NZ, NV, 4), np.uint32)
        L.run_fill(kpool.ctypes.data, C.byref(g), tables.ctypes.data, Fb.ctypes.data, S.ctypes.data, blocks.ctypes.data, len(blocks), spa)
        assert same_bits(Fb[:, :, :NV], ref), (eq, "fill")
        Fp = np.full((NZ, NV, P), np.nan, np.float32)
        S2 = np.zeros((NZ, NV, 4), np.uint32)
        L.run_plane(kpool.ctypes.data, C.byref(g), tables.ctypes.data, Fp.ctypes.data, S2.ctypes.data, spa)
        assert same_bits(Fp[:, :, :NV], ref), (eq, "plane")


# ---- emulated device pipeline ------------------------------------------------------------------------------------------
EMULATED_CSG = {"union": CSG_UNION2, "lens": CSG_LENS, "difference": CSG_SPHERE_MINUS_CYLINDER, "box": CSG_BOX_SDF}


@pytest.mark.parametrize("name", sorted(EMULATED_CSG))
@pytest.mark.parametrize("mode", ["dense", "blocks"])
def test_emulated_kernels_reproduce_the_oracle_csg_mesh(mcb_emu, name, mode):
    """The device code executed on the host (tests/emu) at step 2/32 (33^3 cubes), both field modes: per-cube codes, counts, soup
    and welded Poly_Data equal the oracle's reference pipeline on the CSG equation."""
    eq, step, scale = EMULATED_CSG[name], 2.0 / 32, 1.1
    ctx = mcb_emu.Context(0)
    try:
        ctx.set_mesh_mode(mcb_emu.MESH_SOUP | mcb_emu.MESH_INDEXED)
        ctx.set_grammar(mcb_emu.GRAMMAR_FUNCTIONS)
        assert ctx.set_equation(eq) == 0
        M = ctx.set_grid_step(step)
        ctx.set_scaling(scale, scale, scale)
        ctx.set_field_mode(mcb_emu.FIELD_DENSE if mode == "dense" else mcb_emu.FIELD_AUTO)
        ctx.set_normals(0)
        cnt = ctx.polygonise()
        code, tidx = ctx.get_cases()
        pos, _ = ctx.get_mesh(normals=False)
        vl, tl = ctx.get_indexed_mesh(normals=False)[:2]
    finally:
        ctx.close()
    o = CsgOracle(eq, step=step, scale=(scale, scale, scale))
    assert o.M == M
    sw = o.sweep()
    v, t = o.recalculate()
    assert sw["T"] > 500 and cnt.triangles == sw["T"]
    assert np.array_equal(code.ravel(), sw["code"]) and np.array_equal(tidx.ravel(), sw["table_idx"])
    assert cnt.ambiguous == sw["ambiguous"] and cnt.redirected == sw["redirected"]
    assert same_bits(pos[:, :, :3], sw["soup"])
    assert same_bits(vl, v) and np.array_equal(tl, t)
