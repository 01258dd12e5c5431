"""-m gpu: analytic normals (mcb_set_normals 3, mcb_eval_gradients) on the B200.  The device's normals equal the host build's
bit for bit at every soup and welded vertex; they are byte-identical across field modes, interpreted and compiled runs,
slabs, seed mode and repeating-surface mode, while positions, indices and counts stay those of mode 0; on smooth fields they
agree with the central differences of mode 1, on kinked fields they do not; mcb_headless and the C++ drop-in deliver the
same bytes; a 1024^3 run is deterministic."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_UNION2, CSG_UNION8
from .functions_common import FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, GYROID, TORUS_SDF
from .helpers import configure, load_meta, same_bits
from .normals_common import NORMALS_ANALYTIC, SPECIAL, counts_tuple, host_eval, run_mesh, soup_matches_welded
from .test_normals_host import _check_box_faces

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "mcb_headless")
F = GRAMMAR_FUNCTIONS
A = NORMALS_ANALYTIC
NAMED = {"gyroid": (GYROID, 0.05), "torus_sdf": (TORUS_SDF, 0.04), "mixed": (FUNCTION_EQUATIONS[5], 0.05),
         "union2": (CSG_UNION2, 0.05), "box_sdf": (CSG_BOX_SDF, 0.05), "union8": (CSG_UNION8, 0.04)}
SEEDS = {"gyroid": (-0.01, 0.01, 0.012), "union8": (0.7, 0.41, 0.41), "box_sdf": (0.57, 0.47, 0.01)}  # in an active cube
GOLDEN_NAMES = ["sphere_17", "eq3_gui", "eq8_ctor", "gyr78_17", "quirk_div", "quirk_neg", "nonuniform_scale", "constraint_2"]


def _assert_normals_are_the_host_ones(m, eq, scale, grammar):
    p = m["pos"][:, :, :3].reshape(-1, 3)
    assert same_bits(m["nrm"][:, :, :3].reshape(-1, 3), host_eval(eq, p, scale, grammar)[3])
    assert not m["nrm"][:, :, 3].any()
    assert same_bits(m["vn"], host_eval(eq, m["vl"], scale, grammar)[3])
    a, b, k = soup_matches_welded(m)
    assert same_bits(a, b) and k > 0


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_golden_cases_device_equals_host(mcb, golden, name):
    case = load_meta(golden)[name]
    c = mcb.Context(0)
    try:
        c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        configure(c, case)
        out = {}
        for mode in (0, A):
            c.set_normals(mode)
            cnt = c.polygonise()
            pos, nrm = c.get_mesh(normals=mode == A)
            r = c.get_indexed_mesh(normals=mode == A)
            out[mode] = dict(counts=cnt, pos=pos, nrm=nrm, vl=r[0], tl=r[1], vn=r[2] if mode else None)
    finally:
        c.close()
    m3, m0 = out[A], out[0]
    assert counts_tuple(m3["counts"]) == counts_tuple(m0["counts"]) and m3["counts"].triangles > 0
    assert same_bits(m3["pos"], m0["pos"]) and same_bits(m3["vl"], m0["vl"]) and np.array_equal(m3["tl"], m0["tl"])
    _assert_normals_are_the_host_ones(m3, case["eq"], tuple(case["scale"]), 0)


@pytest.mark.parametrize("name", sorted(NAMED))
def test_function_and_csg_cases_device_equals_host(mcb, name):
    eq, step = NAMED[name]
    m3 = run_mesh(mcb, eq, step, (1.1, 1.1, 1.1), A)
    m0 = run_mesh(mcb, eq, step, (1.1, 1.1, 1.1), 0)
    assert counts_tuple(m3["counts"]) == counts_tuple(m0["counts"]) and m3["counts"].triangles > 1000
    assert same_bits(m3["pos"], m0["pos"]) and same_bits(m3["vl"], m0["vl"]) and np.array_equal(m3["tl"], m0["tl"])
    _assert_normals_are_the_host_ones(m3, eq, (1.1, 1.1, 1.1), F)


def test_eval_gradients_on_special_values_equals_the_host(mcb):
    a, b, c3 = np.meshgrid(SPECIAL, SPECIAL, SPECIAL, indexing="ij")
    pts = np.stack([a.ravel(), b.ravel(), c3.ravel()], axis=1)
    pts = np.concatenate([pts, np.random.default_rng(9).uniform(-2, 2, (5000, 3)).astype(np.float32)])
    c = mcb.Context(0)
    try:
        c.set_grammar(F)
        c.set_scaling(1.1, 0.9, 1.3)
        for eq in FUNCTION_EQUATIONS + [CSG_UNION2, CSG_BOX_SDF, "x^y+z", "(x-1)^y/z", "min(x,y)*max(z,x)", "abs(x)-sqrt(y)+1/z"]:
            assert c.set_equation(eq, slot=2) == 0
            assert same_bits(c.eval_gradients(pts, slot=2), host_eval(eq, pts)[2]), eq
            assert same_bits(c.eval_gradients(pts, slot=2, apply_scale=True), host_eval(eq, pts, (1.1, 0.9, 1.3))[2]), eq
        with pytest.raises(mcb.McbError):
            c.eval_gradients(pts, slot=3)
    finally:
        c.close()


@pytest.mark.parametrize("name", ["gyroid", "union8", "box_sdf"])
def test_mode3_bytes_across_field_modes_jit_slabs_seed_and_levels(mcb, name):
    eq, step = NAMED[name]
    runs = [run_mesh(mcb, eq, step, normals=A, field_mode=fm, jit=jit)
            for fm in (mcb.FIELD_DENSE, mcb.FIELD_SPARSE) for jit in (mcb.JIT_OFF, mcb.JIT_ON)]
    assert sorted((r["field_mode"], r["jit"]) for r in runs) == [(0, 0), (0, 1), (1, 0), (1, 1)]
    for r in runs[1:]:
        for k in ("pos", "nrm", "vl", "tl", "vn"):
            assert r[k].tobytes() == runs[0][k].tobytes(), k
    full = runs[0]
    by_pos = {full["pos"][t, i, :3].tobytes(): full["nrm"][t, i].tobytes() for t in range(len(full["pos"])) for i in range(3)}
    M = full["counts"].M
    sl = run_mesh(mcb, eq, step, normals=A, slab=(M // 3, M // 3 + 5))
    sl0 = run_mesh(mcb, eq, step, normals=0, slab=(M // 3, M // 3 + 5))
    assert 0 < sl["counts"].triangles < full["counts"].triangles
    assert counts_tuple(sl["counts"]) == counts_tuple(sl0["counts"]) and sl["pos"].tobytes() == sl0["pos"].tobytes()
    assert all(by_pos[sl["pos"][t, i, :3].tobytes()] == sl["nrm"][t, i].tobytes() for t in range(len(sl["pos"])) for i in range(3))
    seed = run_mesh(mcb, eq, step, normals=A, seed=SEEDS[name])
    lev = run_mesh(mcb, eq, step, normals=A, levels=0.3)
    lev0 = run_mesh(mcb, eq, step, normals=0, levels=0.3)
    assert counts_tuple(lev["counts"]) == counts_tuple(lev0["counts"]) and lev["vl"].tobytes() == lev0["vl"].tobytes()
    for m in (seed, lev):
        assert m["counts"].triangles > 0
        _assert_normals_are_the_host_ones(m, eq, (1.0, 1.0, 1.0), F)
    assert all(by_pos[seed["pos"][t, i, :3].tobytes()] == seed["nrm"][t, i].tobytes() for t in range(len(seed["pos"])) for i in range(3))


def _max_angle_deg(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    ok = (np.linalg.norm(a, axis=1) > 0.5) & (np.linalg.norm(b, axis=1) > 0.5)
    cos = np.clip(np.sum(a[ok] * b[ok], axis=1) / np.linalg.norm(a[ok], axis=1) / np.linalg.norm(b[ok], axis=1), -1, 1)
    return float(np.degrees(np.arccos(cos)).max())


def test_smooth_fields_agree_with_mode1_and_kinked_fields_do_not(mcb, golden):
    gyr78 = load_meta(golden)["gyr78_17"]["eq"]
    step = 2.0 / 256
    # (equation, grammar, bound in degrees): mode 1's error shrinks with step^2; the degree-7 gyroid curves fastest
    smooth = {"sphere": ("x^2+y^2+z^2-0.49", 0, 0.01), "torus_sdf": (TORUS_SDF, F, 0.1), "gyr78": (gyr78, 0, 5.0)}
    for name, (eq, grammar, bound) in smooth.items():
        m3 = run_mesh(mcb, eq, step, normals=A, grammar=grammar)
        m1 = run_mesh(mcb, eq, step, normals=1, grammar=grammar)
        ang = _max_angle_deg(m3["vn"], m1["vn"])
        print("%s at step 2/256: largest angle between mode 3 and mode 1 normals %.4f degrees" % (name, ang))
        assert ang < bound, (name, ang)
    # the union's seam is a kink of the surface: mode 1 averages the two spheres' normals there at any step.  The rounded
    # box is smooth but its curvature jumps where a face meets an edge, and the field has a kink 0.1 inside the surface
    for name, eq, least in (("box_sdf", CSG_BOX_SDF, 0.5), ("union2", CSG_UNION2, 10.0)):
        m3 = run_mesh(mcb, eq, step, normals=A)
        m1 = run_mesh(mcb, eq, step, normals=1)
        ang = _max_angle_deg(m3["vn"], m1["vn"])
        print("%s at step 2/256: largest angle between mode 3 and mode 1 normals %.2f degrees" % (name, ang))
        assert ang > least, (name, ang)
        if name == "box_sdf":
            flat, dev1 = _check_box_faces(m3["vl"], m3["vn"], m1["vn"])
            assert flat > 10000 and dev1 > 1e-2


def _headless(tmp_path, extra):
    dump, nd = tmp_path / "m.bin", tmp_path / "n.bin"
    out = subprocess.check_output([EXE, "--eq", CSG_BOX_SDF, "--functions", "--res", "96", "--scale", "1", "1", "1", "--dump", str(dump),
                                   "--dump-normals", str(nd)] + extra, text=True)
    raw = dump.read_bytes()
    nv, nt = struct.unpack("<QQ", raw[:16])
    v = np.frombuffer(raw, np.float32, nv * 3, 16).reshape(-1, 3)
    t = np.frombuffer(raw, np.uint32, nt * 3, 16 + nv * 12).reshape(-1, 3)
    return json.loads(out.strip().splitlines()[-1]), v, t, np.frombuffer(nd.read_bytes(), np.float32)


def test_headless_and_dropin_give_the_ctypes_bytes(mcb, tmp_path):
    info, v, t, n = _headless(tmp_path, ["--analytic-normals"])
    m = mcb.Marching()
    e = mcb.Evaluator()
    e.set_function_grammar(True)
    assert e.set_equation(CSG_BOX_SDF)
    m.set_evaluator(e)
    assert m.set_grid_resolution(96)
    m.set_normals(A)
    assert m.recalculate()
    pd = m.get_poly_data()
    assert info["triangles"] == len(t) > 5000
    assert same_bits(pd.vertex_list.reshape(-1, 3), v) and np.array_equal(pd.tri_list.reshape(-1, 3), t)
    assert same_bits(pd.vertex_normals.reshape(-1), n)
    assert same_bits(n.reshape(-1, 3), host_eval(CSG_BOX_SDF, v)[3])
    # the soup path of the drop-in (set_weld(false)): 3 float4 normals per triangle
    _, vs, ts, ns = _headless(tmp_path, ["--analytic-normals", "--soup"])
    assert len(ts) == len(t) and len(ns) == 12 * len(t)
    assert same_bits(ns.reshape(-1, 4)[:, :3], host_eval(CSG_BOX_SDF, vs)[3])
    _, _, _, n1 = _headless(tmp_path, [])
    assert n1.shape == n.shape and not same_bits(n1, n)


def test_1024_gyroid_is_deterministic(mcb):
    c = mcb.Context(0)
    try:
        c.set_grammar(F)
        assert c.set_equation(GYROID) == 0
        c.set_grid_step(2.0 / 1024)
        c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        c.set_normals(A)
        a = c.polygonise()
        na = c.get_mesh()[1].tobytes()
        va = c.get_indexed_mesh(normals=True)[2].tobytes()
        b = c.polygonise()
        assert a.triangles > 10 ** 6 and counts_tuple(a) == counts_tuple(b)
        assert c.get_mesh()[1].tobytes() == na and c.get_indexed_mesh(normals=True)[2].tobytes() == va
    finally:
        c.close()
