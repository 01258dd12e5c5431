"""CPU tier: host logic of the boundary (tokenizer, two-stack lowering, grid loop, slabs, tables, C-ABI exports)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Evaluator::test()'s nine cases (evaluator.h:67-77) — the only known-answer test the reference ships.
EVALUATOR_TEST_CASES = [("-(x+ -(y)* -.021)", True), ("(x(y)", False), ("(x)", True), ("(x-)", False), ("(-x)", True),
                        ("-(-x)", True), ("", False), ("xyz", True), ("xy/z^-.22", True)]

# SURVEY.md Appendix A.1: operation order of the reference's two-stack evaluator (probe-verified against the
# compiled reference) — NOT conventional precedence.
POSTFIX_KNOWN = {
    "x-y+z": "x y z + -",
    "x/y*z": "x y z * /",
    "-x^2": "x NEG 2 ^",
    "x*-y+z": "x y NEG z + *",
    "x+y*z^2+x": "x y z 2 ^ x + * +",
    "x-y*z+x": "x y z * x + -",
    "x*y-z*x+y": "x y * z x * y + -",
    "x^2-y^2-z^2": "x 2 ^ y 2 ^ z 2 ^ - -",
    "x^y^z": "x y z ^ ^",
    "(x)(y)2": "x y 2 * *",
    "-(x+ -(y)* -.021)": "x y NEG 0.021 NEG * + NEG",
    "x^2*y^2+x^2*z^2+z^2*y^2+x*y*z": "x 2 ^ y 2 ^ x 2 ^ z 2 ^ z 2 ^ y 2 ^ x y z * * + * + * + *",
}


def test_abi_exports_every_declared_symbol(mcb):
    hdr = open(os.path.join(ROOT, "include", "mcb.h")).read()
    declared = set(re.findall(r"\b(mcb_[a-z_0-9]+)\s*\(", hdr))
    declared -= {"mcb_ctx"}
    lib = C.CDLL(mcb.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), "libmcb200.so does not export " + name
    assert set(mcb.EXPORTS) == declared
    assert mcb.lib.mcb_abi_version() == 4
    import ctypes
    assert mcb.lib.mcb_struct_size(0) == ctypes.sizeof(mcb.Counts) and mcb.lib.mcb_struct_size(1) == ctypes.sizeof(mcb.StepData)
    assert mcb.lib.mcb_struct_size(7) < 0


def test_loaded_library_is_the_build_of_these_sources(mcb):
    """mcb_build_stamp(): sha256 over the sources the loaded libmcb200.so was compiled from == the sources in the tree"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mcb_build", os.path.join(ROOT, mcb.__name__, "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert mcb.lib.mcb_build_stamp().decode() == b.source_stamp()


@pytest.mark.parametrize("eq,ok", EVALUATOR_TEST_CASES)
def test_evaluator_selftest_cases(mcb, eq, ok):
    assert mcb.parse_ok(eq) == ok


def test_tokenizer_matches_reference(mcb, refbind):
    cases = [e for e, _ in EVALUATOR_TEST_CASES] + ["2..3", "3.x", "x.5", "--x", "x--y", "()", ".", "x)", "a", "X+Y*Z", "x y", "2x",
                                                     "x(y)", "(x)(y)2", "x^-y", "x*-(y)", "-", "(", "1.2.3", "x+(", "((x))", "x^2^3",
                                                     "3(x)", "x3", "x 3", ".5.5", "x*/y", "+x", "x++y", "-x-y", "(-)", "-.5x"]
    for eq in cases:
        ref_ok = refbind.parse_ok(eq)
        mine = mcb.parse_ok(eq)
        if ref_ok and not mine:
            # accepted by the reference tokenizer, refused here: only allowed when the reference would underflow its
            # operand stack (undefined behaviour), i.e. an operator with a missing operand
            assert eq in ("x+", "-", "x+(", "(", "x^-") or eq.rstrip()[-1] in "+-*/^(" or eq == "-", eq
        else:
            assert mine == ref_ok, eq


@pytest.mark.parametrize("eq,pf", sorted(POSTFIX_KNOWN.items()))
def test_two_stack_operation_order(mcb, eq, pf):
    assert mcb.postfix(eq) == pf


def test_implicit_multiplication_tokens(mcb):
    assert mcb.tokens("xyz") == "x * y * z"
    assert mcb.tokens("2x(y)3") == "2 * x * ( y ) * 3"
    assert mcb.tokens("x*-y") == "x * NEG y"
    assert mcb.tokens("xy/z^-.22") == "x * y / z ^ NEG .22"


def test_grid_loop_matches_reference(mcb, refbind):
    for step in (0.5, 0.25, 0.2, 0.1, 0.05, 0.01, 0.001, 2.0 / 256, 2.0 / 1024, 0.0123, 0.3):
        r = refbind.Ref("x", step)
        Mr, cr = r.coords()
        M, c = mcb.grid_axis(step)
        assert M == Mr and np.array_equal(c.view(np.uint32), cr.view(np.uint32)), step


def test_grid_loop_known_counts(mcb):
    # SURVEY.md Appendix A.3 (probe of the reference loop)
    for step, M in [(0.5, 5), (0.25, 9), (0.2, 11), (0.1, 21), (0.05, 41), (0.01, 201), (0.001, 2001), (2.0 / 256, 257),
                    (2.0 / 1024, 1025), (2.0 / 2048, 2049)]:
        assert mcb.grid_axis(step)[0] == M
    with pytest.raises(mcb.McbError):
        mcb.grid_axis(0.0)


def test_slab_ranges_partition(mcb):
    for M in (9, 257, 1025, 2049):
        for n in (1, 2, 3, 4, 8):
            edges = [mcb.slab_range(M, r, n) for r in range(n)]
            assert edges[0][0] == 0 and edges[-1][1] == M
            assert all(edges[i][1] == edges[i + 1][0] for i in range(n - 1))
            sizes = [b - a for a, b in edges]
            assert max(sizes) - min(sizes) <= 1


def _packed_rows():
    txt = open(os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "csrc", "mcb_tri_words.inc")).read()
    words = [int(w, 16) for w in re.findall(r"0x([0-9a-f]{16})ull", txt)]
    assert len(words) == 256
    rows = []
    for w in words:
        r = [(w >> (4 * f)) & 0xF for f in range(16)]
        rows.append([v if v != 0xF else -1 for v in r])
    return np.array(rows, np.int32)


EDGES = [[0, 1], [1, 2], [2, 3], [3, 0], [4, 5], [5, 6], [6, 7], [7, 4], [0, 4], [1, 5], [2, 6], [3, 7]]


def _golden_active_cubes(golden):
    """(case name, case, x, y, z, linear index) of every cube with triangles in the reference's golden runs, in its loop
    order (x fastest), with the offset of the cube's first triangle in the golden soup."""
    from .helpers import load_meta
    for name, case in load_meta(golden).items():
        M, t = case["M"], 0
        ntri = golden[name + "/ntri"].astype(np.int64)
        for lin in np.flatnonzero(ntri):
            yield name, case, int(lin % M), int(lin // M % M), int(lin // (M * M)), int(lin), t
            t += int(ntri[lin])


def test_packed_triangle_table_equals_reference(golden):
    """The committed packed table against the reference.  Where oracle/_ref is built: all 256 rows of its tri_table and
    its edge table.  Always: every row the reference's golden runs used (tests/golden/cases.npz) against the triangles
    the reference emitted — the row holds its triangle count, and the k-th corner of the soup lies on the row's k-th
    edge (the two fixed coordinates equal, the third between the edge's corners), which pins edges, order and winding."""
    from oracle import refbind
    rows = _packed_rows()
    if refbind.available():
        tri, _, edge = refbind.tables()
        assert np.array_equal(rows, tri)
        assert edge.tolist() == EDGES
    rows_seen = set()
    for name, case, i, j, k, lin, t in _golden_active_cubes(golden):
        c = golden[name + "/coords"]
        ti = int(golden[name + "/table_idx"][lin])
        r = rows[ti][rows[ti] >= 0]
        assert len(r) == 3 * int(golden[name + "/ntri"][lin]), (name, lin, ti)
        soup = golden[name + "/soup"][t:t + len(r) // 3].reshape(-1, 3)
        # corner v at (i,j,k) + bits 0,1,2 of v ^ ((v >> 1) & 1) (mcb_tables.h)
        P = np.array([[c[i + (o & 1)], c[j + (o >> 1 & 1)], c[k + (o >> 2 & 1)]] for o in (v ^ (v >> 1 & 1) for v in range(8))], np.float32)
        for p, e in zip(soup, r):
            a, b = P[EDGES[e][0]], P[EDGES[e][1]]
            ax = int(np.flatnonzero(a != b)[0])
            assert all(p[d] == a[d] for d in range(3) if d != ax), (name, lin, ti, e)
            assert min(a[ax], b[ax]) <= p[ax] <= max(a[ax], b[ax]) or np.isnan(p[ax]), (name, lin, ti, e)
        rows_seen.add(ti)
    assert len(rows_seen) >= 228


def test_triangle_table_invariants():
    rows = _packed_rows()
    hist = np.bincount([(r != -1).sum() // 3 for r in rows], minlength=6)
    assert hist.tolist() == [2, 16, 50, 80, 76, 32]  # SURVEY.md §8 a10
    EA = [0, 1, 2, 3, 4, 5, 6, 7, 0, 1, 2, 3]
    EB = [1, 2, 3, 0, 5, 6, 7, 4, 4, 5, 6, 7]
    for code, r in enumerate(rows):
        for e in r[r != -1]:
            assert ((code >> EA[e]) ^ (code >> EB[e])) & 1, "row references a non-crossing edge"


def test_ambiguity_faces_equal_reference(mcb, golden):
    """The derived face-per-code table (mcb_tables.h) against the reference.  Where oracle/_ref is built: all 256 rows of
    the table it ships.  Always: the reference's golden runs (tests/golden/cases.npz) — the cubes it counted as ambiguous
    are exactly the active cubes whose code has a face here, and every cube it redirected took row 255 - code."""
    from oracle import refbind
    from .helpers import load_meta
    FACE = [(0, 1, 2, 3), (1, 2, 6, 5), (4, 5, 6, 7), (0, 3, 7, 4), (3, 2, 6, 7), (0, 1, 5, 4)]
    derived = []
    for code in range(256):
        f = -1
        for fi in (0, 1, 2, 3, 5, 4):
            b = [(code >> v) & 1 for v in FACE[fi]]
            if b[0] == b[2] and b[1] == b[3] and b[0] != b[1]:
                f = fi
        derived.append([-1] if f < 0 else [255 - code] + list(FACE[f]))
    assert sum(len(d) > 1 for d in derived) == 120
    if refbind.available():
        _, amb, _ = refbind.tables()
        for code in range(256):
            assert amb[code][0] == -1 if len(derived[code]) == 1 else amb[code].tolist() == derived[code]
    redirected_seen = 0
    for name, case in load_meta(golden).items():
        code, tidx = golden[name + "/code"].astype(np.int64), golden[name + "/table_idx"].astype(np.int64)
        active = (code != 0) & (code != 255)
        has_face = np.array([len(d) > 1 for d in derived])[code]
        assert int((active & has_face).sum()) == case["ambiguous"], name
        red = tidx != code
        assert int(red.sum()) == case["redirected"] and np.all(has_face[red]) and np.array_equal(tidx[red], 255 - code[red]), name
        redirected_seen += int(red.sum())
    assert redirected_seen > 0


def test_lowering_bit_exact_on_host(mcb, refbind):
    """The bytecode the GPU interprets, run by the host build of the same interpreter (oracle/host_interp.cpp), against
    Evaluator::evaluate of the compiled reference: random points and a tensor grid (exercises folding + hoisting)."""
    so = os.path.join(ROOT, "oracle", "libmcoracle_host.so")
    if not os.path.exists(so):
        pytest.skip("oracle/libmcoracle_host.so not built")
    H = C.CDLL(so)
    H.mcoh_eval_points.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_long]
    H.mcoh_eval_grid.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    rng = np.random.default_rng(1)
    pts = (rng.random((4000, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    pts[:32] = 0
    cx = np.linspace(-1.1, 1.2, 19, dtype=np.float32)
    cy = np.linspace(-0.9, 1.3, 13, dtype=np.float32)
    cz = np.linspace(-1, 1, 7, dtype=np.float32)
    Z, Y, X = np.meshgrid(cz, cy, cx, indexing="ij")
    gp = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    eqs = list(refbind.EXAMPLE_EQUATIONS.values()) + [refbind.SPHERE, refbind.TORUS, refbind.GYR34, refbind.GYR78] + \
        list(POSTFIX_KNOWN) + ["x^0.5+y", "x/y", "1/(x*y*z)", "x^-2", "-x^0.5", "2^x+y^z", "x^y", "(1/3)^2*x+(1/3)*y", "3", "1+2*3"]
    for eq in eqs:
        ref = refbind.Ref(eq)
        out = np.empty(len(pts), np.float32)
        assert H.mcoh_eval_points(eq.encode(), pts.ctypes.data, out.ctypes.data, len(pts)) == 0
        r = ref.eval_points(pts)
        assert np.all((r.view(np.uint32) == out.view(np.uint32)) | (np.isnan(r) & np.isnan(out))), eq
        g = np.empty(len(gp), np.float32)
        assert H.mcoh_eval_grid(eq.encode(), cx.ctypes.data, len(cx), cy.ctypes.data, len(cy), cz.ctypes.data, len(cz), g.ctypes.data) == 0
        rg = ref.eval_points(gp)
        assert np.all((rg.view(np.uint32) == g.view(np.uint32)) | (np.isnan(rg) & np.isnan(g))), eq


def test_no_device_is_a_loud_failure(mcb):
    """Without a GPU the product refuses to work (no CPU fallback); with one, creation succeeds."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        mcb.Context(0).close()
    else:
        with pytest.raises(mcb.McbError) as ei:
            mcb.Context(0)
        assert ei.value.status == mcb.MCB_E_NODEVICE


def test_grid_limits(mcb):
    """M is capped at 4094 (12-bit cube indices in the active-cube records); steps outside (0, 1] are rejected."""
    assert mcb.lib.mcb_grid_axis(2.0 / 4093, None, 0) in (4093, 4094)
    assert mcb.lib.mcb_grid_axis(2.0 / 5000, None, 0) < 0
    for bad in (0.0, -0.1, 1.5, float("nan"), float("inf")):
        assert mcb.lib.mcb_grid_axis(bad, None, 0) < 0


def test_jit_source_compiles_for_every_golden_equation_without_a_gpu(mcb, golden):
    """mcb_jit_check: generate the specialised evaluator of each golden equation and compile it with NVRTC for sm_100a
    (no device needed).  The source depends on the equation's program only: same source for any constants/grid."""
    from .helpers import load_meta
    seen = {}
    for name, case in load_meta(golden).items():
        if case["eq"] in seen:
            continue
        nbytes, src = mcb.jit_check(case["eq"])
        seen[case["eq"]] = nbytes
        assert nbytes > 1000 and "mcb_eval_jit" in src and "op_" in src or "ty" in src
    assert len(seen) >= 15
    assert mcb.jit_check("x^2+y^2+z^2-0.49")[1] == mcb.jit_check("x^2+y^2+z^2-0.25")[1]   # constants are arguments
    with pytest.raises(mcb.McbError):
        mcb.jit_check("x+")                                                                 # parse error, not a crash


def test_committed_bench_lines_carry_every_contract_key():
    """The bench lines committed under profiles/ (what `python bench.py` and `bench.py --impl reference` printed on the
    B200) have every key of the measurement contract, and the numbers hang together."""
    import glob
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ours = sorted(glob.glob(os.path.join(root, "profiles", "r02_bench_n[1248].json")))
    assert len(ours) == 4
    for path in ours:
        d = json.loads(open(path).read().strip().splitlines()[-1])
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                  "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks", "changed_param", "strong_2048"):
            assert k in d, (path, k)
        assert d["metric"] == d["unit"] == "Gvoxels/s" and d["scaling"] == "weak" and d["warmup"] >= 3 and d["gpu_launches"] > 0
        assert abs(d["config"]["cubes"] / (d["ms_per_step"] * 1e-3) / 1e9 - d["value"]) < 1e-6 * d["value"]
        for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert k in d["roofline"], (path, k)
        assert abs(d["roofline"]["achieved"] / d["roofline"]["peak"] - d["roofline"]["frac"]) < 1e-9
        for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
            assert k in d["e2e"], (path, k)
        assert d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        assert abs(d["changed_param"]["value"] / d["value"] - 1.0) < 0.05     # a changed parameter costs what a repeat costs
        st = d["strong_2048"]
        assert st["resolution"] == 2048 and st["scaling"] == "strong" and len(st["per_rank"]) == d["n_gpus"]
        assert sum(r["triangles"] for r in st["per_rank"]) == st["triangles"] == 19369064
        if d["n_gpus"] == 1:
            for k in ("value", "unit", "cores", "kind", "sample"):
                assert k in d["cpu_baseline"], k
            for k in ("first_call", "variants", "workloads"):
                assert k in d, k
            assert d["e2e"]["dropin"]["value"] > 0.9 * d["e2e"]["value"] and set(d["workloads"]) == {"gyr78", "torus"}
            assert d["workloads"]["gyr78"]["redirected"] > 0
            fc = d["first_call"]   # the first mesh of a new equation came from the interpreter, before the compile had finished
            assert fc["jit_first_call"] == 0 and fc["ms_wall"] < fc["ms_until_compiled_wall"] and fc["ms_compile"] > 0
        else:
            assert 0.5 < st["efficiency_vs_n1_2048"] <= 1.0
            ms = [r["ms_kernels"] for r in st["per_rank"]]
            assert max(ms) / (sum(ms) / len(ms)) < 1.06               # the refined cut: every rank within a few per cent
    ref = json.loads(open(os.path.join(root, "profiles", "r02_bench_reference_arm.json")).read().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and ref["metric"] == "Gvoxels/s" and ref["e2e"]["h2d_bytes_per_step"] == 0
    assert ref["cpu_baseline"]["kind"] == "reference" and ref["cpu_baseline"]["cores"] >= 1


def test_jit_source_has_both_kernels(mcb):
    """One module per equation: mcb_eval_jit (plane tiles: the whole field + signs) and mcb_fill_jit (listed 32 x 4 x 4 blocks:
    field + signs, the block-field mode).  The operations are spelled with the never-contracted intrinsics."""
    _, plain = mcb.jit_check("x*y+z*(x-y)")
    _, power = mcb.jit_check("(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)")
    for src in (plain, power):
        for kernel in ("mcb_eval_jit", "mcb_fill_jit"):
            assert src.count('%s(const __grid_constant__ Consts C' % kernel) == 1 or ("define MCB_KERNEL_NAME " + kernel) in src, kernel
        assert "mcb_signs_jit" not in src
        assert "__fadd_rn" in src and "__fmul_rn" in src and "__fdiv_rn" in src and "mcb_powf" in src
    assert "op_pow(" in power and "op_pow(v" not in plain


def _random_equation(rng, depth):
    """A random string over the reference's grammar: variables, numbers, + - * / ^, brackets, unary minus and the
    implicit-multiplication forms (2x, x(y), (x)(y))."""
    r = rng.random()
    if depth <= 0 or r < 0.25:
        k = rng.integers(0, 6)
        if k < 3:
            return "xyz"[k]
        if k == 3:
            return str(int(rng.integers(0, 10)))
        if k == 4:
            return "%d.%d" % (rng.integers(0, 4), rng.integers(0, 100))
        return "XYZ"[rng.integers(0, 3)]
    if r < 0.45:
        return "(" + _random_equation(rng, depth - 1) + ")"
    if r < 0.52:
        return "-" + _random_equation(rng, depth - 1)
    if r < 0.60:
        return _random_equation(rng, depth - 1) + "(" + _random_equation(rng, depth - 1) + ")"
    if r < 0.65:
        return str(int(rng.integers(2, 5))) + "xyz"[rng.integers(0, 3)]
    return _random_equation(rng, depth - 1) + "+-*/^"[rng.integers(0, 5)] + _random_equation(rng, depth - 1)


def test_random_equations_lower_bit_exactly(mcb, refbind):
    """Fuzz of the front end against the compiled reference: 500 random (half of them mutated, so often malformed)
    equations.  Accept/reject: the product never accepts what Evaluator::tokenize rejects; it additionally rejects
    strings the reference tokenizes but cannot evaluate (a dangling operator pops its unchecked Simple_Stack empty:
    undefined behaviour there), exactly the ones the plain-C restatement flags as operand underflow.  Values: for every
    equation both accept, the bytecode run by the host build of the interpreter equals Evaluator::evaluate bit for
    bit at random points and on a tensor grid (folding, hoisting, fusion)."""
    from oracle import oraclebind
    so = os.path.join(ROOT, "oracle", "libmcoracle_host.so")
    if not os.path.exists(so) or not oraclebind.available():
        pytest.skip("oracle libraries not built")
    H = C.CDLL(so)
    H.mcoh_eval_points.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_long]
    H.mcoh_eval_grid.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    rng = np.random.default_rng(20261018)
    pts = (rng.random((200, 3), dtype=np.float32) * 3 - 1.5).astype(np.float32)
    pts[:8] = 0
    pts[8:16] = 1
    cx = np.linspace(-1.1, 1.2, 7, dtype=np.float32)
    cy = np.linspace(-0.9, 1.3, 5, dtype=np.float32)
    cz = np.linspace(-1, 1, 3, dtype=np.float32)
    Z, Y, X = np.meshgrid(cz, cy, cx, indexing="ij")
    gp = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    alphabet = "xyzXYZ0123456789.+-*/^() "
    both = stricter = rejected = 0
    for _ in range(500):
        eq = _random_equation(rng, int(rng.integers(1, 6)))
        if rng.random() < 0.5:
            for _m in range(int(rng.integers(1, 3))):
                i, k, ch = int(rng.integers(0, len(eq) + 1)), rng.integers(0, 3), alphabet[rng.integers(0, len(alphabet))]
                eq = eq[:i] + eq[i + 1:] if k == 0 else eq[:i] + ch + eq[i:] if k == 1 else eq[:i] + ch + eq[i + 1:]
        if not eq or len(eq) > 120:
            continue
        ref_ok, ours_ok = refbind.parse_ok(eq), mcb.parse_ok(eq)
        assert ref_ok or not ours_ok, eq
        if not ref_ok:
            rejected += 1
            continue
        if not ours_ok:
            assert not oraclebind.lib().mco_parse_ok(eq.encode()), eq
            stricter += 1
            continue
        both += 1
        ref = refbind.Ref(eq)
        out = np.empty(len(pts), np.float32)
        assert H.mcoh_eval_points(eq.encode(), pts.ctypes.data, out.ctypes.data, len(pts)) == 0, eq
        r = ref.eval_points(pts)
        assert np.all((r.view(np.uint32) == out.view(np.uint32)) | (np.isnan(r) & np.isnan(out))), eq
        g = np.empty(len(gp), np.float32)
        assert H.mcoh_eval_grid(eq.encode(), cx.ctypes.data, len(cx), cy.ctypes.data, len(cy), cz.ctypes.data, len(cz), g.ctypes.data) == 0, eq
        rg = ref.eval_points(gp)
        assert np.all((rg.view(np.uint32) == g.view(np.uint32)) | (np.isnan(rg) & np.isnan(g))), eq
    assert both > 300 and rejected > 30 and stricter > 3, (both, rejected, stricter)


def test_random_equations_compile_at_run_time(mcb):
    """The kernel generator takes whatever the lowering produces (deep stacks, NEG, reversed operators, powers): 25 random
    well-formed equations go through generation and NVRTC without a device."""
    rng = np.random.default_rng(77)
    done = 0
    while done < 25:
        eq = _random_equation(rng, int(rng.integers(2, 6)))
        if len(eq) > 100 or not mcb.parse_ok(eq):
            continue
        nbytes, src = mcb.jit_check(eq, cap=1 << 20)
        assert nbytes > 1000 and src.count("__launch_bounds__") == 2, eq
        done += 1


class _HostGrid(C.Structure):  # mcbk::Grid / the Grid struct of the generated source (52 bytes)
    _fields_ = [(n, C.c_int) for n in ("M", "NV", "P", "WP", "kb", "ke", "NZ")] + \
               [(n, C.c_float) for n in ("sx", "sy", "sz", "iso")] + [("repeat", C.c_int), ("rstep", C.c_float)]


def test_generated_kernel_source_executed_on_the_host_equals_the_reference(mcb, refbind, tmp_path):
    """The CUDA source mcb_jit.cpp generates is also valid C++ under a small shim (tests/cpp/jit_host_shim.h): g++ compiles
    it with -ffp-contract=off and both kernels run lane by lane over a small grid with random coordinates (warp
    ballots emulated by a two-pass trick).  The field they write equals Evaluator::evaluate of the compiled reference
    bit for bit and the sign words equal `value > iso`, for the bench equations and for random ones (deep stacks,
    reversed operators, powers, unary minus)."""
    import subprocess
    so_host = os.path.join(ROOT, "oracle", "libmcoracle_host.so")
    if not os.path.exists(so_host):
        pytest.skip("oracle/libmcoracle_host.so not built")
    H = C.CDLL(so_host)
    H.mcoh_tables.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    P = 32
    rng = np.random.default_rng(3)
    ax = [np.sort((rng.random(P, dtype=np.float32) * 3 - 1.5).astype(np.float32)) for _ in range(3)]
    eqs = [refbind.SPHERE, refbind.TORUS, refbind.EXAMPLE_EQUATIONS[8], refbind.GYR34, "x*y-z/(x+2.5)", "-x^2-(y-1)(z+2)/3", "2^x+y^z"]
    while len(eqs) < 17:
        eq = _random_equation(rng, int(rng.integers(2, 6)))
        if len(eq) <= 100 and mcb.parse_ok(eq):
            eqs.append(eq)
    shim = os.path.join(ROOT, "tests", "cpp", "jit_host_shim.h")
    tail = open(os.path.join(ROOT, "tests", "cpp", "jit_host_tail.inc")).read()
    for n, eq in enumerate(eqs):
        # geometry: vertices per axis, planes, first cube layer of the slab (the z tables are indexed by plane + kb)
        NV, NZ, kb = ((11, 9, 0), (21, 6, 5), (16, 4, 2))[n % 3]
        Z, Y, X = np.meshgrid(ax[2][kb:kb + NZ], ax[1][:NV], ax[0][:NV], indexing="ij")
        pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
        _, src = mcb.jit_check(eq, cap=1 << 20)
        cpp, so = tmp_path / ("k%d.cpp" % n), tmp_path / ("k%d.so" % n)
        cpp.write_text('#include "%s"\n' % shim + src + tail)
        r = subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-w", "-shared", "-fPIC", "-I", os.path.join(ROOT, mcb.__name__, "csrc"),
                            "-DMCB_GRID_BYTES=%d" % C.sizeof(_HostGrid), "-DMCB_MAX_K=128", "-DMCB_MIN_BLOCKS=8", str(cpp), "-o", str(so)],
                           capture_output=True, text=True)
        assert r.returncode == 0, (eq, r.stderr[:2000])
        L = C.CDLL(str(so))
        L.run_fill.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_int]
        tables = np.zeros(3 * 64 * P + 256, np.float32)
        kpool = np.zeros(128, np.float32)
        spa = H.mcoh_tables(eq.encode(), ax[0].ctypes.data, ax[1].ctypes.data, ax[2].ctypes.data, P, tables.ctypes.data, len(tables) - 256,
                            kpool.ctypes.data)
        assert spa > 0, (eq, spa)
        g = _HostGrid(M=NV - 3, NV=NV, P=P, WP=4, kb=kb, ke=kb + NZ - 3, NZ=NZ, sx=1, sy=1, sz=1, iso=0, repeat=0, rstep=0)
        ref = refbind.Ref(eq).eval_points(pts).reshape(NZ, NV, NV)
        g.iso = float(np.float32(np.nanmedian(ref[np.isfinite(ref)]))) if np.isfinite(ref).any() else 0.0
        with np.errstate(invalid="ignore"):
            want = ref > np.float32(g.iso)   # sign bit = value > iso, strict, NaN -> 0
        xs = np.arange(NV)
        nbx, nby, nbz = P // 32, (NV + 3) // 4, (NZ + 3) // 4
        ids = np.arange(nbx * nby * nbz)
        blocks = ((ids % nbx) | ((ids // nbx % nby) << 8) | ((ids // (nbx * nby)) << 20)).astype(np.uint32)  # bx | by << 8 | bz << 20
        # mcb_fill_jit: every block listed; field and sign words (warp ballots emulated by the shim)
        F = np.full((NZ, NV, P), np.nan, np.float32)
        S = np.zeros((NZ, NV, 4), np.uint32)
        L.run_fill(kpool.ctypes.data, C.byref(g), tables.ctypes.data, F.ctypes.data, S.ctypes.data, blocks.ctypes.data, len(blocks), spa)
        got = F[:, :, :NV]
        assert np.all((ref.view(np.uint32) == got.view(np.uint32)) | (np.isnan(ref) & np.isnan(got))), eq
        bits = ((S[:, :, xs >> 5] >> (xs & 31).astype(np.uint32)) & 1).astype(bool)
        assert np.array_equal(bits, want), (eq, "fill")
        # mcb_eval_jit: 128 x 4 tile in registers, field + sign words
        L.run_plane.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        F2 = np.full((NZ, NV, P), np.nan, np.float32)
        S2 = np.zeros((NZ, NV, 4), np.uint32)
        L.run_plane(kpool.ctypes.data, C.byref(g), tables.ctypes.data, F2.ctypes.data, S2.ctypes.data, spa)
        bits = ((S2[:, :, xs >> 5] >> (xs & 31).astype(np.uint32)) & 1).astype(bool)
        assert np.array_equal(bits, want), (eq, "plane")
        got2 = F2[:, :, :NV]
        assert np.all((ref.view(np.uint32) == got2.view(np.uint32)) | (np.isnan(ref) & np.isnan(got2))), eq
