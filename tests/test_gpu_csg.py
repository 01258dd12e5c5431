"""-m gpu: min( max( of the function grammar (unions, intersections, differences of shapes) on the device against
oracle/mc_oracle_csg.c, whose own tokenizer and walk restate min / max in plain C: fields, cases, counts, soups and welded
meshes bit for bit, in both field modes, interpreted and run-time compiled; the special values of minimumNumber /
maximumNumber; the interval proof's block counts; seed mode; mcb_headless; a 1024^3 union."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from . import mc_numpy
from .csg_common import CSG_BOX_SDF, CSG_LENS, CSG_SPHERE_MINUS_CYLINDER, CSG_UNION2, CSG_UNION8, CsgOracle
from .functions_common import GRAMMAR_FUNCTIONS
from .helpers import rel_close, same_bits
from .test_csg_host import definition, special_pairs
from .test_gpu_parity import tri_rows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = GRAMMAR_FUNCTIONS

# (equation, step, scale, iso, constraints).  Not min(sqrt(x^2+y^2+z^2)-0.5,z+0.3+0.1sin(9x)cos(7y)) at step 0.05: there the
# reference's vertex set keeps 20 duplicate vertices (3799 against the weld's 3779), the documented deviation of the weld
# (DESIGN.md §5); its field, cases and soup are bit-exact.
CASES = {
    "union2": (CSG_UNION2, 0.05, (1.0, 1.0, 1.0), 0.0, []),
    "lens": (CSG_LENS, 0.04, (1.0, 1.0, 1.0), 0.0, []),
    "sphere_minus_cylinder": (CSG_SPHERE_MINUS_CYLINDER, 0.05, (1.0, 1.0, 1.0), 0.0, []),
    "box_sdf": (CSG_BOX_SDF, 0.05, (1.1, 1.1, 1.1), 0.0, []),
    "union8": (CSG_UNION8, 0.04, (1.0, 1.0, 1.0), 0.0, []),
    "sphere_cons": ("x^2+y^2+z^2-0.5", 0.06, (1.0, 1.0, 1.0), 0.0, [("max(abs(x),abs(y))", "<", 0.6), ("min(x,z)", ">", -0.5)]),
    "mixed_sin": ("min(sqrt(x^2+y^2+z^2)-0.5,z+0.35+0.1sin(8x))", 0.05, (1.0, 1.0, 1.0), 0.0, []),
}


def _configure(ctx, eq, step, scale, iso, cons):
    ctx.set_grammar(F)
    assert ctx.set_equation(eq) == 0
    M = ctx.set_grid_step(step)
    ctx.set_scaling(*scale)
    ctx.set_surface_constant(iso)
    for i in range(3):
        ctx.set_constraint(i, ">", 0.0, False)
    for i, (lhs, op, rhs) in enumerate(cons):
        assert ctx.set_equation(lhs, slot=i + 1) == 0
        assert ctx.set_constraint(i, op, rhs, True) == 0
    return M


@pytest.fixture(scope="module")
def ctx(mcb):
    c = mcb.Context(0)
    c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
    yield c
    c.close()


@pytest.mark.parametrize("jit", [0, 1])
@pytest.mark.parametrize("name", sorted(CASES))
def test_csg_dense_mode_bit_exact_against_the_oracle(mcb, ctx, name, jit):
    eq, step, scale, iso, cons = CASES[name]
    ctx.set_jit(mcb.JIT_ON if jit else mcb.JIT_OFF)
    ctx.set_field_mode(mcb.FIELD_DENSE)
    ctx.set_normals(1)
    M = _configure(ctx, eq, step, scale, iso, cons)
    cnt = ctx.polygonise()
    assert cnt.jit == jit
    o = CsgOracle(eq, step=step, scale=scale, iso=iso, cons=cons)
    Mo, c = o.coords()
    assert Mo == M
    Z, Y, X = np.meshgrid(c, c, c, indexing="ij")
    pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    assert same_bits(ctx.get_field().ravel(), o.eval_points(pts, scaled=True)), "field at every vertex"
    sw = o.sweep(grad_normals=False)
    code, tidx = ctx.get_cases()
    assert np.array_equal(code.ravel(), sw["code"]) and np.array_equal(tidx.ravel(), sw["table_idx"])
    assert (cnt.active, cnt.triangles, cnt.ambiguous, cnt.redirected) == (sw["active"], sw["T"], sw["ambiguous"], sw["redirected"])
    assert cnt.triangles > 1000
    pos, nrm = ctx.get_mesh(normals=True)
    assert same_bits(pos[:, :, :3], sw["soup"])
    v, t = o.recalculate()
    vl, tl = ctx.get_indexed_mesh(normals=False)[:2]
    assert same_bits(vl, v) and np.array_equal(tl, t)
    cs = mc_numpy.apron_coords(c, step)
    Z, Y, X = np.meshgrid(cs, cs, cs, indexing="ij")
    ext = o.eval_points(np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32), scaled=True).reshape(len(cs), len(cs), len(cs))
    rec, _ = ctx.get_active()
    cubes = [(int(r & 0xFFF), int((r >> 12) & 0xFFF), int((r >> 24) & 0xFFF), int((r >> 36) & 0xFF), int((r >> 44) & 0xFF)) for r in rec]
    nref = mc_numpy.soup_gradient_normals(ext, cs, iso, cubes, tri_rows())
    ok = np.isfinite(nref).all(axis=2)
    assert rel_close(nrm[:, :, :3][ok], nref[ok], 1e-5)


@pytest.mark.parametrize("name", sorted(CASES))
def test_csg_field_modes_and_jit_are_byte_identical(mcb, name):
    """Dense, block-field with and without the interval proof ($MCB_NO_INTERVAL) and the compiled kernels: the same
    bytes in every mesh output."""
    eq, step, scale, iso, cons = CASES[name]
    outs = []
    for field, jit, nointerval in ((mcb.FIELD_DENSE, mcb.JIT_OFF, False), (mcb.FIELD_SPARSE, mcb.JIT_OFF, False),
                                   (mcb.FIELD_SPARSE, mcb.JIT_OFF, True), (mcb.FIELD_SPARSE, mcb.JIT_ON, False),
                                   (mcb.FIELD_DENSE, mcb.JIT_ON, False)):
        if nointerval:
            os.environ["MCB_NO_INTERVAL"] = "1"
        try:
            c = mcb.Context(0)
        finally:
            os.environ.pop("MCB_NO_INTERVAL", None)
        try:
            c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
            c.set_normals(1)
            c.set_jit(jit)
            c.set_field_mode(field)
            _configure(c, eq, step, scale, iso, cons)
            cnt = c.polygonise()
            assert cnt.jit == (jit == mcb.JIT_ON) and cnt.field_mode == field
            code, tidx = c.get_cases()
            pos, nrm = c.get_mesh(normals=True)
            vl, tl, vn = c.get_indexed_mesh(normals=True)
            outs.append((code.tobytes(), tidx.tobytes(), pos.tobytes(), nrm.tobytes(), vl.tobytes(), tl.tobytes(), vn.tobytes(),
                         (cnt.active, cnt.triangles, cnt.ambiguous, cnt.redirected, cnt.vertices)))
        finally:
            c.close()
    for o in outs[1:]:
        assert o == outs[0]


def test_eval_points_on_special_values_equals_the_definition(mcb, ctx):
    """mcb_eval_points of min(x,y) / max(x,y) (scale 1: the coordinates reach the interpreter unchanged) on every pair of
    {+-0, +-denormal, +-1, +-FLT_MAX, +-inf, NaN, ...} and on 1e6 random bit pairs: minimumNumber / maximumNumber exactly"""
    a, b = special_pairs()
    rng = np.random.default_rng(5)
    ra = rng.integers(0, 1 << 32, 10 ** 6, dtype=np.uint64).astype(np.uint32).view(np.float32)
    rb = rng.integers(0, 1 << 32, 10 ** 6, dtype=np.uint64).astype(np.uint32).view(np.float32)
    a, b = np.concatenate([a, ra]), np.concatenate([b, rb])
    pts = np.stack([a, b, np.zeros_like(a)], 1).astype(np.float32)
    ctx.set_grammar(F)
    ctx.set_scaling(1.0, 1.0, 1.0)
    for name, is_max in (("min", False), ("max", True)):
        assert ctx.set_equation("%s(x,y)" % name) == 0
        got = ctx.eval_points(pts)
        assert same_bits(got, definition(a, b, is_max)), name
        z = np.array([[0.0, -0.0, 0], [-0.0, 0.0, 0]], np.float32)
        assert (np.signbit(ctx.eval_points(z)) == (not is_max)).all(), name


def _field_blocks(mcb, eq, res=256):
    c = mcb.Context(0)
    try:
        c.set_mesh_mode(mcb.MESH_SOUP)
        c.set_field_mode(mcb.FIELD_SPARSE)
        c.set_jit(mcb.JIT_OFF)
        c.set_grammar(F)
        assert c.set_equation(eq) == 0
        c.set_grid_step(2.0 / res)
        cnt = c.polygonise()
        return int(cnt.field_blocks)
    finally:
        c.close()


@pytest.mark.parametrize("a,b", [("sqrt(x^2+y^2+z^2)-0.5", "sqrt((x-0.45)^2+y^2+z^2)-0.35"),
                                 ("sqrt((x-0.3)^2+y^2+z^2)-0.6", "sqrt((x+0.3)^2+y^2+z^2)-0.6"),
                                 ("sqrt(x^2+y^2+z^2)-0.7", "-(sqrt(x^2+y^2)-0.3)"), ("abs(x)-0.5", "sin(9y)+z")])
def test_interval_proof_leaves_no_more_blocks_for_min_max_than_for_the_arguments(mcb, a, b):
    fa, fb = _field_blocks(mcb, a), _field_blocks(mcb, b)
    for f in ("min", "max"):
        fm = _field_blocks(mcb, "%s(%s,%s)" % (f, a, b))
        assert 0 < fm <= fa + fb, (f, fm, fa, fb)


def test_seed_mode_on_a_union_keeps_the_seeded_sphere(mcb):
    """Two disjoint spheres joined by min, seeded in a surface cube of one: the soup is that sphere's polygonised alone,
    byte for byte (near it min returns its field bit for bit); without the seed the union has both spheres."""
    left = "(x+0.45)^2+y^2+z^2-0.09"
    right = "(x-0.45)^2+y^2+z^2-0.09"
    outs = []
    for eq, seed in (("min(%s,%s)" % (left, right), True), (left, False), ("min(%s,%s)" % (left, right), False)):
        c = mcb.Context(0)
        try:
            c.set_mesh_mode(mcb.MESH_SOUP)
            c.set_normals(0)
            c.set_grammar(F)
            assert c.set_equation(eq) == 0
            c.set_grid_step(0.04)
            if seed:
                assert c.set_seed(True, -0.74, 0.01, 0.02) == 0
            cnt = c.polygonise()
            outs.append((cnt.triangles, c.get_mesh(normals=False)[0][:, :, :3].tobytes()))
        finally:
            c.close()
    assert outs[0][0] > 1000 and outs[0] == outs[1]
    assert outs[2][0] == 2 * outs[0][0]


def test_headless_functions_flag_gives_the_ctypes_csg_mesh(mcb, tmp_path):
    exe = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "mcb_headless")
    dump = tmp_path / "c.bin"
    out = subprocess.check_output([exe, "--eq", CSG_BOX_SDF, "--functions", "--res", "96", "--scale", "1", "1", "1", "--dump", str(dump)], text=True)
    info = json.loads(out.strip().splitlines()[-1])
    raw = dump.read_bytes()
    nv, nt = struct.unpack("<QQ", raw[:16])
    v = np.frombuffer(raw, np.float32, nv * 3, 16).reshape(-1, 3)
    t = np.frombuffer(raw, np.uint32, nt * 3, 16 + nv * 12).reshape(-1, 3)
    m = mcb.Marching()
    e = mcb.Evaluator()
    e.set_function_grammar(True)
    assert e.set_equation(CSG_BOX_SDF)
    m.set_evaluator(e)
    assert m.set_grid_resolution(96)
    assert m.recalculate()
    pd = m.get_poly_data()
    assert info["triangles"] == nt and nt > 5000
    assert same_bits(pd.vertex_list.reshape(-1, 3), v) and np.array_equal(pd.tri_list.reshape(-1, 3), t)
    assert subprocess.run([exe, "--eq", CSG_BOX_SDF], capture_output=True).returncode == 1  # the default grammar rejects it


def test_union8_1024_is_deterministic_and_one_layer_equals_the_oracle(mcb):
    c = mcb.Context(0)
    try:
        c.set_grammar(F)
        assert c.set_equation(CSG_UNION8) == 0
        M = c.set_grid_step(2.0 / 1024)
        c.set_mesh_mode(mcb.MESH_SOUP)
        c.set_normals(0)
        a = c.polygonise()
        pa = c.get_mesh(normals=False)[0].tobytes()
        b = c.polygonise()
        assert a.triangles > 10 ** 6
        assert (a.triangles, a.active, a.ambiguous, a.redirected) == (b.triangles, b.active, b.ambiguous, b.redirected)
        assert c.get_mesh(normals=False)[0].tobytes() == pa
        k = 700
        c.set_slab(k, k + 1)
        c.set_field_mode(mcb.FIELD_DENSE)
        cnt = c.polygonise()
        code, tidx = c.get_cases()
        pos = c.get_mesh(normals=False)[0]
    finally:
        c.close()
    o = CsgOracle(CSG_UNION8, step=2.0 / 1024)
    assert o.M == M
    sw = o.sweep(k0=k, k1=k + 1)
    assert cnt.triangles == sw["T"] > 1000
    assert np.array_equal(code.ravel(), sw["code"]) and np.array_equal(tidx.ravel(), sw["table_idx"])
    assert same_bits(pos[:, :, :3], sw["soup"])
