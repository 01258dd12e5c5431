"""-m gpu: the function grammar (MCB_GRAMMAR_FUNCTIONS) on the device against oracle/mc_oracle_fn.c, whose own tokenizer and
two-stack walk call libm sinf / cosf / sqrtf / fabsf: fields, cases, counts, soups and welded meshes bit for bit, in both
field modes, interpreted and run-time compiled."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from . import mc_numpy
from .functions_common import CHECKER, FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, GYROID, TORUS_SDF, FnOracle, random_function_equations
from .helpers import rel_close, same_bits
from .test_gpu_parity import tri_rows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = GRAMMAR_FUNCTIONS

# (equation, step, scale, iso, constraints); the steps of gyroid and nonhoist are coarse enough for the face-centre test to
# redirect cubes (REDIRECTS), the smooth distance fields have no ambiguous faces that flip at any step tried; checker has
# only ambiguous cubes and makes the soup emitter split its chunks into several runs
CASES = {
    "checker": (CHECKER, 0.125, (1.0, 1.0, 1.0), 0.0, []),
    "gyroid": (GYROID, 0.1, (1.1, 1.1, 1.1), 0.0, []),
    "torus_sdf": (TORUS_SDF, 0.05, (1.0, 1.0, 1.0), 0.0, []),
    "nonhoist": ("sin(6(x^2+y^2+z^2))", 0.15, (1.0, 1.0, 1.0), 0.1, []),
    "octahedron_cons": ("abs(x)+abs(y)+abs(z)-0.7", 0.07, (1.0, 1.0, 1.0), 0.0, [("sin(3x)+cos(2y)", ">", 0.2), ("sqrt(abs(z))", "<", 0.8)]),
    "schwarz_cons": (FUNCTION_EQUATIONS[4], 0.09, (1.2, 1.0, 0.9), 0.3, [("abs(x-y)", "<=", 0.9)]),
    "mixed": (FUNCTION_EQUATIONS[5], 0.06, (1.0, 1.0, 1.0), 0.0, []),
}
REDIRECTS = {"checker", "gyroid", "nonhoist"}


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


def _oracle(eq, step, scale, iso, cons):
    return FnOracle(eq, step=step, scale=scale, iso=iso, cons=cons)


@pytest.fixture(scope="module")
def ctx(mcb):
    c = mcb.Context(0)
    c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
    yield c
    c.close()


@pytest.mark.parametrize("jit", [0, 1])
@pytest.mark.parametrize("name", sorted(CASES))
def test_dense_mode_bit_exact_against_the_oracle(mcb, ctx, name, jit):
    eq, step, scale, iso, cons = CASES[name]
    ctx.set_jit(mcb.JIT_ON if jit else mcb.JIT_OFF)
    ctx.set_field_mode(mcb.FIELD_DENSE)
    ctx.set_normals(1)
    M = _configure(ctx, eq, step, scale, iso, cons)
    cnt = ctx.polygonise()
    assert cnt.jit == jit
    o = _oracle(eq, step, scale, iso, cons)
    Mo, c = o.coords()
    assert Mo == M
    Z, Y, X = np.meshgrid(c, c, c, indexing="ij")
    pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    assert same_bits(ctx.get_field().ravel(), o.eval_points(pts, scaled=True)), "field at every vertex"
    sw = o.sweep(grad_normals=False)
    code, tidx = ctx.get_cases()
    assert np.array_equal(code.ravel(), sw["code"]) and np.array_equal(tidx.ravel(), sw["table_idx"])
    assert (cnt.active, cnt.triangles, cnt.ambiguous, cnt.redirected) == (sw["active"], sw["T"], sw["ambiguous"], sw["redirected"])
    if name in REDIRECTS:
        assert cnt.redirected > 0, "a coarse grid should redirect some ambiguous cubes"
    pos, nrm = ctx.get_mesh(normals=True)
    assert same_bits(pos[:, :, :3], sw["soup"])
    v, t = o.recalculate()
    vl, tl = ctx.get_indexed_mesh(normals=False)[:2]
    assert same_bits(vl, v) and np.array_equal(tl, t)
    # gradient normals: the numpy restatement of their definition on the oracle's field over the apron grid
    cs = mc_numpy.apron_coords(c, step)
    Z, Y, X = np.meshgrid(cs, cs, cs, indexing="ij")
    ext = o.eval_points(np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32), scaled=True).reshape(len(cs), len(cs), len(cs))
    rec, _ = ctx.get_active()
    cubes = [(int(r & 0xFFF), int((r >> 12) & 0xFFF), int((r >> 24) & 0xFFF), int((r >> 36) & 0xFF), int((r >> 44) & 0xFF)) for r in rec]
    nref = mc_numpy.soup_gradient_normals(ext, cs, iso, cubes, tri_rows())
    ok = np.isfinite(nref).all(axis=2)
    assert rel_close(nrm[:, :, :3][ok], nref[ok], 1e-5)


@pytest.mark.parametrize("name", sorted(CASES))
def test_block_field_and_jit_outputs_are_byte_identical(mcb, name):
    """Block-field mode with and without the interval proof ($MCB_NO_INTERVAL) and the compiled kernels against the
    interpreted dense field: the same bytes in every mesh output."""
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


def test_eval_points_and_inspect_cube_equal_the_oracle(mcb, ctx):
    rng = np.random.default_rng(8)
    pts = (rng.random((5000, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    for eq in FUNCTION_EQUATIONS + random_function_equations(mcb, 77, 40):
        ctx.set_grammar(F)
        assert ctx.set_equation(eq) == 0, eq
        ctx.set_scaling(1.0, 1.0, 1.0)
        o = _oracle(eq, 0.25, (1.0, 1.0, 1.0), 0.0, [])
        assert same_bits(ctx.eval_points(pts), o.eval_points(pts)), eq
    eq, step, scale, iso, cons = CASES["octahedron_cons"]
    ctx.set_field_mode(mcb.FIELD_DENSE)
    M = _configure(ctx, eq, step, scale, iso, cons)
    ctx.polygonise()
    o = _oracle(eq, step, scale, iso, cons)
    _, c = o.coords()
    sw = o.sweep(soup=False)
    code = sw["code"].reshape(M, M, M)
    for (k, j, i) in [tuple(int(q) for q in a) for a in np.argwhere((code != 0) & (code != 255))[:40]]:
        sd = ctx.inspect_cube(float(c[i]), float(c[j]), float(c[k]))
        assert sd.skipped == 0 and sd.cube_code == code[k, j, i]
        assert sd.table_idx == sw["table_idx"].reshape(M, M, M)[k, j, i]
        corners = np.array(sd.corner_coords, np.float32).reshape(8, 3)
        assert same_bits(np.array(sd.corner_values, np.float32), o.eval_points(corners, scaled=True))


def test_reference_grammar_equations_are_byte_identical_under_the_function_grammar(mcb):
    from .test_emu_pipeline import GYR78
    outs = {}
    for grammar in (0, F):
        for eq in ("x^2+y^2+z^2-0.49", GYR78):
            c = mcb.Context(0)
            try:
                c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
                c.set_grammar(grammar)
                assert c.set_equation(eq) == 0
                c.set_grid_step(2.0 / 200)
                cnt = c.polygonise()
                outs[(grammar, eq)] = (c.get_mesh(normals=True)[0].tobytes(), c.get_indexed_mesh()[1].tobytes(),
                                       (cnt.triangles, cnt.vertices, cnt.jit))
            finally:
                c.close()
    for eq in ("x^2+y^2+z^2-0.49", GYR78):
        assert outs[(0, eq)] == outs[(F, eq)]


def test_gyroid_1024_is_deterministic_and_one_layer_equals_the_oracle(mcb):
    c = mcb.Context(0)
    try:
        c.set_grammar(F)
        assert c.set_equation(GYROID) == 0
        M = c.set_grid_step(2.0 / 1024)
        c.set_mesh_mode(mcb.MESH_SOUP)
        c.set_normals(0)
        a = c.polygonise()
        pa = c.get_mesh(normals=False)[0].tobytes()
        b = c.polygonise()
        assert (a.triangles, a.active, a.ambiguous, a.redirected) == (b.triangles, b.active, b.ambiguous, b.redirected)
        assert c.get_mesh(normals=False)[0].tobytes() == pa
        k = 517
        c.set_slab(k, k + 1)
        c.set_field_mode(mcb.FIELD_DENSE)
        c.polygonise()
        code, tidx = c.get_cases()
        pos = c.get_mesh(normals=False)[0]
    finally:
        c.close()
    o = _oracle(GYROID, 2.0 / 1024, (1.0, 1.0, 1.0), 0.0, [])
    assert o.M == M
    sw = o.sweep(k0=k, k1=k + 1)
    assert np.array_equal(code.ravel(), sw["code"]) and np.array_equal(tidx.ravel(), sw["table_idx"])
    assert same_bits(pos[:, :, :3], sw["soup"])


def test_headless_functions_flag_gives_the_ctypes_mesh(mcb, tmp_path):
    exe = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "mcb_headless")
    dump = tmp_path / "g.bin"
    out = subprocess.check_output([exe, "--eq", GYROID, "--functions", "--res", "96", "--scale", "1", "1", "1", "--dump", str(dump)], text=True)
    info = json.loads(out.strip().splitlines()[-1])
    raw = dump.read_bytes()
    nv, nt = struct.unpack("<QQ", raw[:16])
    v = np.frombuffer(raw, np.float32, nv * 3, 16).reshape(-1, 3)
    t = np.frombuffer(raw, np.uint32, nt * 3, 16 + nv * 12).reshape(-1, 3)
    m = mcb.Marching()
    e = mcb.Evaluator()
    e.set_function_grammar(True)
    assert e.set_equation(GYROID)
    m.set_evaluator(e)
    assert m.set_grid_resolution(96)
    assert m.recalculate()
    pd = m.get_poly_data()
    assert info["triangles"] == nt and nt > 10000
    assert same_bits(pd.vertex_list.reshape(-1, 3), v) and np.array_equal(pd.tri_list.reshape(-1, 3), t)
    assert subprocess.run([exe, "--eq", GYROID], capture_output=True).returncode == 1  # the default grammar rejects it
