"""CPU tier of the function grammar (MCB_GRAMMAR_FUNCTIONS: sin( cos( sqrt( abs( on top of the reference's language):
the grammar rules, the restated sinf / cosf against libm, the lowering against the independent restatement in
oracle/mc_oracle_fn.c, the interval rules against brute force, the run-time compiled kernels executed on the host and the
emulated device pipeline against the oracle's meshes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from .functions_common import (CHECKER, FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, GYROID, TORUS_SDF, FnOracle, fn_parse_ok,
                               host_fn_lib, random_function_equations, trig_exhaustive_exe)
from .helpers import same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = GRAMMAR_FUNCTIONS

# (equation, tokens or None for a parse error, postfix)
GRAMMAR_TABLE = [
    ("sin(x)", "sin( x )", "x sin"),
    ("sin (x)", "sin( x )", "x sin"),
    ("cos(y)+sqrt(z)", "cos( y ) + sqrt( z )", "y cos z sqrt +"),
    ("abs(-x)", "abs( NEG x )", "x NEG abs"),
    ("sin(-x)", "sin( NEG x )", "x NEG sin"),
    ("-sin(x)^2", "NEG sin( x ) ^ 2", "x sin NEG 2 ^"),
    ("-(x)^2", "NEG ( x ) ^ 2", "x NEG 2 ^"),
    ("2sin(x)", "2 * sin( x )", "2 x sin *"),
    ("xcos(y)", "x * cos( y )", "x y cos *"),
    ("(x)sin(y)", "( x ) * sin( y )", "x y sin *"),
    ("sin(x)cos(y)", "sin( x ) * cos( y )", "x sin y cos *"),
    ("sin(x)(y)", "sin( x ) * ( y )", "x sin y *"),
    ("sin(x)2", "sin( x ) * 2", "x sin 2 *"),
    ("sqrt(sqrt(x^2+y^2)-0.5)", "sqrt( sqrt( x ^ 2 + y ^ 2 ) - 0.5 )", "x 2 ^ y 2 ^ + sqrt 0.5 - sqrt"),
    ("x-sin(y)+z", "x - sin( y ) + z", "x y sin z + -"),
    ("sin(x+y*z)^2", "sin( x + y * z ) ^ 2", "x y z * + sin 2 ^"),
    ("abs(x)^sin(y)", "abs( x ) ^ sin( y )", "x abs y sin ^"),
    ("sin(2)", "sin( 2 )", "2 sin"),
    ("cos(-(x))", "cos( NEG ( x ) )", "x NEG cos"),
    ("sinx", None, None),
    ("sin x", None, None),
    ("SIN(x)", None, None),
    ("Sin(x)", None, None),
    ("s(x)", None, None),
    ("sin()", None, None),
    ("sin(", None, None),
    ("sin(x", None, None),
    ("sin)x(", None, None),
    ("tan(x)", None, None),
    ("exp(x)", None, None),
    ("sin(-)", None, None),
    ("sin(x+)", None, None),
    ("sqr(x)", None, None),
    ("x+a", None, None),
]


@pytest.mark.parametrize("eq,toks,pf", GRAMMAR_TABLE)
def test_grammar_table(mcb, eq, toks, pf):
    ok = toks is not None
    assert mcb.parse_ok(eq, grammar=F) == ok, eq
    assert fn_parse_ok(eq) == ok, eq  # the oracle's own restatement of the grammar
    if ok:
        assert mcb.tokens(eq, grammar=F) == toks
        assert mcb.postfix(eq, grammar=F) == pf
    has_fn = any(f in eq for f in ("sin", "cos", "sqrt", "abs", "SIN", "Sin", "tan", "exp", "sqr", "a", "s("))
    if has_fn:  # the default grammar is the reference's: every name is a parse error there
        assert not mcb.parse_ok(eq) and not mcb.parse_ok(eq, grammar=0)
        with pytest.raises(mcb.McbError):
            mcb.tokens(eq)


def test_default_grammar_rejects_every_function_equation(mcb):
    for eq in FUNCTION_EQUATIONS + random_function_equations(mcb, 5, 100):
        assert not mcb.parse_ok(eq), eq
        assert mcb.lib.mcb_parse(eq.encode()) == mcb.MCB_E_PARSE


def test_grammar_argument_is_checked(mcb):
    buf = C.create_string_buffer(64)
    assert mcb.lib.mcb_grammar_text(b"x", 2, 0, buf, 64) == mcb.MCB_E_ARG
    assert mcb.lib.mcb_grammar_text(b"x", -1, 0, buf, 64) == mcb.MCB_E_ARG
    assert mcb.lib.mcb_jit_check_grammar(b"x", 7, buf, 64) == mcb.MCB_E_ARG


def _reference_equations(golden):
    from .helpers import load_meta
    from .test_host_logic import POSTFIX_KNOWN, _random_equation
    meta = load_meta(golden)
    eqs = [c["eq"] for c in meta.values()] + [l for c in meta.values() for (l, _, _) in c.get("cons", [])] + list(POSTFIX_KNOWN)
    rng = np.random.default_rng(11)
    alphabet = "xyzXYZ0123456789.+-*/^() "
    for _ in range(1500):
        eq = _random_equation(rng, int(rng.integers(1, 6)))
        if rng.random() < 0.5:  # mutated: the accept/reject of malformed strings must agree as well
            i, ch = int(rng.integers(0, len(eq) + 1)), alphabet[rng.integers(0, len(alphabet))]
            eq = eq[:i] + ch + eq[i:]
        eqs.append(eq)
    return eqs


def test_reference_equations_are_unchanged_under_the_function_grammar(mcb, golden):
    """Every golden and fuzzed equation of the reference grammar: same accept/reject, tokens, postfix and all four
    bytecode listings under both grammars."""
    accepted = 0
    for eq in _reference_equations(golden):
        ok = mcb.parse_ok(eq)
        assert mcb.parse_ok(eq, grammar=F) == ok, eq
        try:
            t0 = mcb.tokens(eq)
        except mcb.McbError:
            t0 = None
        try:
            t1 = mcb.tokens(eq, grammar=F)
        except mcb.McbError:
            t1 = None
        assert t0 == t1, eq
        if not ok:
            continue
        accepted += 1
        assert mcb.postfix(eq) == mcb.postfix(eq, grammar=F), eq
        for which in (0, 1, 2, 3):
            assert mcb.disassemble(eq, which) == mcb.disassemble(eq, which, grammar=F), (eq, which)
    assert accepted > 500


def test_trig_restatement_equals_libm_on_1e8_random_and_edge_inputs():
    """csrc/mcb_trig.h (host build) against this machine's libm sinf / cosf; the full 2^32-input run is
    oracle/trig_exhaustive with no argument (profiles/trig_exhaustive.txt)."""
    exe = trig_exhaustive_exe()
    r = subprocess.run([exe, "1", "100000000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches_sin 0 mismatches_cos 0 out_of_range 0" in r.stdout, r.stdout
    r = subprocess.run([exe, "257"], capture_output=True, text=True)  # every 257th bit pattern, all exponents
    assert r.returncode == 0 and "mismatches_sin 0 mismatches_cos 0 out_of_range 0" in r.stdout, r.stdout


def test_exhaustive_trig_run_is_recorded():
    text = open(os.path.join(ROOT, "profiles", "trig_exhaustive.txt")).read()
    assert "inputs 4294967296 mismatches_sin 0 mismatches_cos 0 out_of_range 0" in text


@pytest.fixture(scope="module")
def host():
    """oracle/host_interp.cpp's runners of the product's bytecode, lowering under the function grammar"""
    return host_fn_lib()


def test_lowering_bit_exact_against_the_oracle(mcb, host):
    """About 500 random function equations (and the named shapes): the product's bytecode, run by the host build of its
    interpreters (folded constants, hoisted axis tables, fused grid form), against the oracle's own tokenizer and
    two-stack walk calling libm, at random points and on a tensor grid.  Each equation also serves as a constraint
    left-hand side (slot 1) of the oracle."""
    rng = np.random.default_rng(123)
    pts = (rng.random((300, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    pts[:8] = 0
    pts[8:16] = -1
    pts[16:24] = np.float32(0.5)
    cx = np.linspace(-1.1, 1.2, 9, dtype=np.float32)
    cy = np.linspace(-0.9, 1.3, 6, dtype=np.float32)
    cz = np.linspace(-1, 1, 4, dtype=np.float32)
    Z, Y, X = np.meshgrid(cz, cy, cx, indexing="ij")
    gp = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    eqs = FUNCTION_EQUATIONS + ["sin(2)+x", "cos(1.5)*sqrt(2)y", "abs(-3)z+sin(x)", "sqrt(-1)+x", "sin(100000000000000000000x)", "cos(x*1000000)+y",
                                "sqrt(x)", "abs(x)-abs(y)"] + random_function_equations(mcb, 9, 480)
    for eq in eqs:
        o = FnOracle(eq)
        assert o.set_equation(1, eq)
        out = np.empty(len(pts), np.float32)
        assert host.mcoh_eval_points(eq.encode(), pts.ctypes.data, out.ctypes.data, len(pts)) == 0, eq
        assert same_bits(out, o.eval_points(pts)), eq
        assert same_bits(out, o.eval_points(pts, slot=1)), eq
        g = np.empty(len(gp), np.float32)
        assert host.mcoh_eval_grid(eq.encode(), cx.ctypes.data, len(cx), cy.ctypes.data, len(cy), cz.ctypes.data, len(cz),
                                           g.ctypes.data) == 0, eq
        assert same_bits(g, o.eval_points(gp)), eq


def test_function_subtrees_are_folded_and_hoisted(mcb):
    """Constant-only functions fold into the constant pool; single-variable ones become axis tables, so the literal
    gyroid's grid program is products and sums of table reads."""
    fused = mcb.disassemble(GYROID, 3, grammar=F)
    assert "SIN" not in fused and "COS" not in fused and "TX" in fused and "TZ" in fused, fused
    slots = mcb.disassemble(GYROID, 2, grammar=F)
    assert slots.count("SIN") == 3 and slots.count("COS") == 3, slots
    assert "SIN" not in mcb.disassemble("sin(2)+x", 3, grammar=F)
    assert mcb.disassemble("sin(2)+x", 2, grammar=F).startswith("K")
    assert "SIN" in mcb.disassemble("sin(6(x^2+y^2+z^2))", 3, grammar=F)
    assert "SQRT" in mcb.disassemble(TORUS_SDF, 3, grammar=F)


@pytest.mark.parametrize("eq", FUNCTION_EQUATIONS + ["sqrt(x+y)-0.3", "sqrt(x*y*z)-0.1", "sin(3(x+y+z))", "cos(0.2x+0.3y)+z",
                                                     "sqrt(abs(x)-0.1)-0.2+z", "abs(x+y)-abs(z)", "sin(20(x+y+z))+0.5z"])
def test_interval_rules_never_prove_wrongly(host, eq):
    """Brute force of the interval proof on function programs, boxes of 4 x 4 x 4 and 8 x 2 x 16 vertices: zero wrong
    proofs, zero enclosure violations (sqrt of intervals that may be negative, sin / cos of narrow and wide ranges)."""
    n = 33
    c = np.linspace(-1.05, 1.05, n, dtype=np.float32)
    for bs in ((4, 4, 4), (8, 2, 16), (2, 2, 2)):
        for iso in (0.0, 0.1, -0.25):
            st = np.zeros(6, np.int64)
            assert host.mcoh_interval_check(eq.encode(), c.ctypes.data, c.ctypes.data, c.ctypes.data, n, *bs,
                                                    C.c_float(iso), st.ctypes.data) == 0
            assert st[4] == 0 and st[5] == 0, (eq, bs, iso, st)


def test_interval_proofs_decide_function_fields(host):
    n = 65
    c = np.linspace(-1, 1, n, dtype=np.float32)
    for eq in (TORUS_SDF, "abs(x)+abs(y)+abs(z)-0.7", GYROID):
        st = np.zeros(6, np.int64)
        assert host.mcoh_interval_check(eq.encode(), c.ctypes.data, c.ctypes.data, c.ctypes.data, n, 4, 4, 4, C.c_float(0.0),
                                                st.ctypes.data) == 0
        assert st[4] == 0 and st[3] > 0 and (st[1] + st[2]) >= 0.8 * st[3], (eq, st)  # most boxes that are uniform are proven so


def test_generated_kernels_compile_without_a_gpu(mcb):
    for eq in [GYROID, TORUS_SDF, "sin(6(x^2+y^2+z^2))", "cos(x*y)+sin(z*x)"] + random_function_equations(mcb, 31, 10, max_len=80):
        nbytes, src = mcb.jit_check(eq, cap=1 << 20, grammar=F)
        assert nbytes > 1000 and src.count("__launch_bounds__") == 2, eq
    _, src = mcb.jit_check("sin(6(x^2+y^2+z^2))", cap=1 << 20, grammar=F)
    assert '#include "mcb_trig.h"' in src and "op_sin(" in src
    _, src = mcb.jit_check("x^2+y^2+z^2-0.49", cap=1 << 20)
    assert "mcb_trig.h" not in src and "op_sqrt" not in src  # a reference-grammar program generates what it did before


def test_generated_kernel_source_executed_on_the_host_equals_the_oracle(mcb, host, tmp_path):
    """The run-time generated CUDA source of function programs, compiled by g++ under tests/cpp/jit_host_shim_fn.h and run
    lane by lane (both kernels), equals the oracle's field bit for bit."""
    from .test_host_logic import _HostGrid
    P = 32
    rng = np.random.default_rng(5)
    ax = [np.sort((rng.random(P, dtype=np.float32) * 3 - 1.5).astype(np.float32)) for _ in range(3)]
    eqs = [GYROID, TORUS_SDF, "sin(6(x^2+y^2+z^2))", "abs(x-y)*cos(z*x)-sqrt(abs(y))"] + random_function_equations(mcb, 41, 6, max_len=80)
    shim = os.path.join(ROOT, "tests", "cpp", "jit_host_shim_fn.h")
    tail = open(os.path.join(ROOT, "tests", "cpp", "jit_host_tail.inc")).read()
    for n, eq in enumerate(eqs):
        NV, NZ, kb = ((11, 9, 0), (21, 6, 5), (16, 4, 2))[n % 3]
        Z, Y, X = np.meshgrid(ax[2][kb:kb + NZ], ax[1][:NV], ax[0][:NV], indexing="ij")
        pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
        _, src = mcb.jit_check(eq, cap=1 << 20, grammar=F)
        cpp, so = tmp_path / ("f%d.cpp" % n), tmp_path / ("f%d.so" % n)
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
        ref = FnOracle(eq).eval_points(pts).reshape(NZ, NV, NV)
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


EMULATED_MESHES = {GYROID: (2.0 / 32, 1.1), TORUS_SDF: (2.0 / 32, 1.1), CHECKER: (0.125, 1.0)}  # equation: (step, scale)


@pytest.mark.parametrize("eq", list(EMULATED_MESHES))
@pytest.mark.parametrize("mode", ["dense", "blocks"])
def test_emulated_kernels_reproduce_the_oracle_mesh(mcb_emu, eq, mode):
    """The device code executed on the host (tests/emu), both field modes: per-cube codes, soup and welded Poly_Data equal
    the oracle's reference pipeline run on the function equation.  CHECKER makes the soup emitter split every full chunk
    into several runs, with and without normals."""
    step, scale = EMULATED_MESHES[eq]
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
        if eq == CHECKER:
            ctx.set_normals(1)
            ctx.polygonise()
            assert same_bits(ctx.get_mesh(normals=True)[0], pos)
    finally:
        ctx.close()
    o = FnOracle(eq, step=step, scale=(scale, scale, scale))
    assert o.M == M
    sw = o.sweep()
    v, t = o.recalculate()
    assert sw["T"] > 1000 and cnt.triangles == sw["T"]
    if eq == CHECKER:  # every cube active, each with 4 triangles (codes 90 / 165)
        assert cnt.active == M ** 3 and cnt.triangles == 4 * M ** 3
    assert np.array_equal(code.ravel(), sw["code"]) and np.array_equal(tidx.ravel(), sw["table_idx"])
    assert cnt.ambiguous == sw["ambiguous"] and cnt.redirected == sw["redirected"]
    assert same_bits(pos[:, :, :3], sw["soup"])
    assert same_bits(vl, v) and np.array_equal(tl, t)
