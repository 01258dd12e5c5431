"""-m gpu: refined vertices (mcb_set_refine_vertices) on the B200.  The device's refined positions equal the host build's
refinement of the unrefined positions bit for bit at every soup and welded vertex, with indices and counts unchanged; they
are byte-identical across field modes, interpreted and compiled runs, slabs, seed mode and constraints; corners on one grid
edge carry one position; normals modes 3 and 2 run at the refined positions; mcb_headless gives the ctypes bytes; a 1024^3
run is deterministic."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_UNION2, CSG_UNION8
from .functions_common import FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, GYROID, TORUS_SDF
from .helpers import configure, load_meta, same_bits
from .normals_common import host_eval
from .refine_common import SAME_SIGN, counts_tuple, host_refine, run_refined

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "mcb_headless")
F = GRAMMAR_FUNCTIONS
NAMED = {"gyroid": (GYROID, 0.05), "torus_sdf": (TORUS_SDF, 0.04), "mixed": (FUNCTION_EQUATIONS[5], 0.05),
         "union2": (CSG_UNION2, 0.05), "box_sdf": (CSG_BOX_SDF, 0.05), "union8": (CSG_UNION8, 0.04)}
SEEDS = {"gyroid": (-0.01, 0.01, 0.012), "union8": (0.7, 0.41, 0.41), "box_sdf": (0.57, 0.47, 0.01)}  # in an active cube
GOLDEN_NAMES = ["sphere_17", "eq3_gui", "eq8_ctor", "gyr78_17", "quirk_div", "quirk_neg", "nonuniform_scale", "constraint_2"]


def _assert_refined_is_the_host_refinement(mcb, m1, m0, eq, step, scale, grammar, iso=0.0):
    assert counts_tuple(m1["counts"]) == counts_tuple(m0["counts"]) and m1["counts"].triangles > 0
    assert np.array_equal(m1["tl"], m0["tl"])
    M, c = mcb.grid_axis(step)
    want, ev, _ = host_refine(eq, c, m0["pos"][:, :, :3].reshape(-1, 3), iso, scale, grammar)
    assert not (ev == SAME_SIGN).any()
    assert same_bits(m1["pos"][:, :, :3].reshape(-1, 3), want) and (m1["pos"][:, :, 3] == 1).all()
    wv, evv, _ = host_refine(eq, c, m0["vl"], iso, scale, grammar)
    assert not (evv == SAME_SIGN).any() and same_bits(m1["vl"], wv)
    return ev


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_golden_cases_device_equals_host(mcb, golden, name):
    case = load_meta(golden)[name]
    c = mcb.Context(0)
    try:
        c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        configure(c, case)
        c.set_normals(0)
        out = {}
        for refine in (False, True):
            c.set_refine_vertices(refine)
            cnt = c.polygonise()
            pos, _ = c.get_mesh(normals=False)
            vl, tl = c.get_indexed_mesh()
            out[refine] = dict(counts=cnt, pos=pos, vl=vl, tl=tl)
    finally:
        c.close()
    _assert_refined_is_the_host_refinement(mcb, out[True], out[False], case["eq"], case["step"], tuple(case["scale"]), 0,
                                           case.get("iso", 0.0))


@pytest.mark.parametrize("name", sorted(NAMED))
def test_function_and_csg_cases_device_equals_host(mcb, name):
    eq, step = NAMED[name]
    m1 = run_refined(mcb, eq, step, (1.1, 1.1, 1.1), True)
    m0 = run_refined(mcb, eq, step, (1.1, 1.1, 1.1), False)
    assert m1["counts"].triangles > 1000
    ev = _assert_refined_is_the_host_refinement(mcb, m1, m0, eq, step, (1.1, 1.1, 1.1), F)
    print("%s: evaluations per refined soup vertex mean %.2f max %d" % (name, ev[ev > 0].mean(), ev.max()))


def _edge_keys(c, p):
    """per point: (axis, i, j, k) of the grid edge whose interior holds it (i, j, k = the lower end's indices), or -1s"""
    idx = np.searchsorted(c, p, side="left")
    idx_c = np.clip(idx, 0, len(c) - 1)
    on = c[idx_c] == p
    inside = (p > c[0]) & (p < c[-1]) & ~on
    ok = (on.sum(axis=1) == 2) & (inside.sum(axis=1) == 1)
    ax = np.argmax(inside, axis=1)
    lower = np.where(on, idx_c, idx - 1)
    keys = np.concatenate([ax[:, None], lower], axis=1).astype(np.int64)
    keys[~ok] = -1
    return keys


@pytest.mark.parametrize("name", ["gyroid", "union8", "box_sdf"])
def test_refined_bytes_across_field_modes_jit_slabs_seed_and_constraints(mcb, name):
    eq, step = NAMED[name]
    runs = [run_refined(mcb, eq, step, field_mode=fm, jit=jit) for fm in (mcb.FIELD_DENSE, mcb.FIELD_SPARSE) for jit in (mcb.JIT_OFF, mcb.JIT_ON)]
    assert sorted((r["field_mode"], r["jit"]) for r in runs) == [(0, 0), (0, 1), (1, 0), (1, 1)]
    for r in runs[1:]:
        for k in ("pos", "vl", "tl"):
            assert r[k].tobytes() == runs[0][k].tobytes(), k
    full, full0 = runs[0], run_refined(mcb, eq, step, refine=False)
    # a refined position is a function of the unrefined one: slab and seed mode refine their vertices to the same bits
    by_pos = {full0["pos"][t, i, :3].tobytes(): full["pos"][t, i].tobytes() for t in range(len(full["pos"])) for i in range(3)}
    M = full["counts"].M
    for kw in (dict(slab=(M // 3, M // 3 + 5)), dict(seed=SEEDS[name])):
        m1, m0 = run_refined(mcb, eq, step, **kw), run_refined(mcb, eq, step, refine=False, **kw)
        assert 0 < m1["counts"].triangles and counts_tuple(m1["counts"]) == counts_tuple(m0["counts"])
        assert all(by_pos[m0["pos"][t, i, :3].tobytes()] == m1["pos"][t, i].tobytes() for t in range(len(m1["pos"])) for i in range(3))
        _assert_refined_is_the_host_refinement(mcb, m1, m0, eq, step, (1.0, 1.0, 1.0), F)
    cons = [("x+y", "<", 0.3), ("z", ">", -0.4)]
    m1, m0 = run_refined(mcb, eq, step, cons=cons), run_refined(mcb, eq, step, refine=False, cons=cons)
    assert 0 < m1["counts"].triangles < full["counts"].triangles
    _assert_refined_is_the_host_refinement(mcb, m1, m0, eq, step, (1.0, 1.0, 1.0), F)


@pytest.mark.parametrize("name", ["gyroid", "torus_sdf", "box_sdf"])
def test_one_position_per_grid_edge(mcb, name):
    """Soup corners on the same grid edge carry identical refined bits, and a soup corner equals its welded vertex wherever
    both lie on the same edge.  The exceptions are the weld's near-vertex merges (a welded vertex within the tolerance
    comparator of a corner on another edge, next to a grid vertex); they are counted."""
    eq, step = NAMED[name]
    m1, m0 = run_refined(mcb, eq, step), run_refined(mcb, eq, step, refine=False)
    M, c = mcb.grid_axis(step)
    p0, p1 = m0["pos"][:, :, :3].reshape(-1, 3), m1["pos"][:, :, :3].reshape(-1, 3)
    keys = _edge_keys(c, p0)
    on = keys[:, 0] >= 0
    _, inv = np.unique(keys[on], axis=0, return_inverse=True)
    first = np.zeros(inv.max() + 1, np.int64)
    first[inv[::-1]] = np.arange(len(inv))[::-1]
    assert same_bits(p1[on], p1[on][first[inv]])
    idx = m0["tl"].reshape(-1).astype(np.int64)
    wkeys = _edge_keys(c, m0["vl"])[idx]
    same_edge = (wkeys == keys).all(axis=1) & on
    assert same_bits(p1[same_edge], m1["vl"][idx][same_edge])
    other = ~same_edge & on
    print("%s: %d soup corners on edge interiors, %d of them welded to a vertex on another edge" % (name, int(on.sum()), int(other.sum())))
    # each is a corner within the weld's 1.5e-6 of a grid vertex, merged with another edge's point near the same vertex
    assert (np.abs(p0[other] - m0["vl"][idx][other]) <= 3e-6).all()


def test_normals_at_the_refined_positions(mcb):
    eq, step = NAMED["torus_sdf"]
    m3 = run_refined(mcb, eq, step, normals=3)
    m0 = run_refined(mcb, eq, step)
    assert same_bits(m3["pos"], m0["pos"]) and same_bits(m3["vl"], m0["vl"])
    p = m3["pos"][:, :, :3].reshape(-1, 3)
    assert same_bits(m3["nrm"][:, :, :3].reshape(-1, 3), host_eval(eq, p)[3])
    assert same_bits(m3["vn"], host_eval(eq, m3["vl"])[3])
    m2 = run_refined(mcb, eq, step, normals=2)
    m2u = run_refined(mcb, eq, step, normals=2, refine=False)
    assert same_bits(m2["vl"], m0["vl"]) and np.array_equal(m2["tl"], m2u["tl"]) and not same_bits(m2["vn"], m2u["vn"])
    assert np.abs(np.linalg.norm(m2["vn"], axis=1) - 1).max() < 1e-5


def _headless(tmp_path, extra):
    dump = tmp_path / "m.bin"
    out = subprocess.check_output([EXE, "--eq", CSG_BOX_SDF, "--functions", "--res", "96", "--scale", "1", "1", "1", "--dump", str(dump)] + extra,
                                  text=True)
    raw = dump.read_bytes()
    nv, nt = struct.unpack("<QQ", raw[:16])
    v = np.frombuffer(raw, np.float32, nv * 3, 16).reshape(-1, 3)
    t = np.frombuffer(raw, np.uint32, nt * 3, 16 + nv * 12).reshape(-1, 3)
    return json.loads(out.strip().splitlines()[-1]), v, t


def test_headless_gives_the_ctypes_bytes(mcb, tmp_path):
    m1 = run_refined(mcb, CSG_BOX_SDF, 2.0 / 96)
    m0 = run_refined(mcb, CSG_BOX_SDF, 2.0 / 96, refine=False)
    info, v, t = _headless(tmp_path, ["--refine-vertices"])
    assert info["triangles"] == len(t) > 5000
    assert same_bits(v, m1["vl"]) and np.array_equal(t, m1["tl"])
    _, vs, ts = _headless(tmp_path, ["--refine-vertices", "--soup"])
    assert len(ts) == len(t) and same_bits(vs.reshape(-1, 3), m1["pos"][:, :, :3].reshape(-1, 3))
    _, v0, _ = _headless(tmp_path, [])
    assert same_bits(v0, m0["vl"]) and not same_bits(v0, v)


def test_1024_gyroid_is_deterministic(mcb):
    c = mcb.Context(0)
    try:
        c.set_grammar(F)
        assert c.set_equation(GYROID) == 0
        c.set_grid_step(2.0 / 1024)
        c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        c.set_normals(0)
        c.set_refine_vertices(True)
        a = c.polygonise()
        pa = c.get_mesh(normals=False)[0].tobytes()
        va = c.get_indexed_mesh()[0].tobytes()
        b = c.polygonise()
        assert a.triangles > 10 ** 6 and counts_tuple(a) == counts_tuple(b)
        assert c.get_mesh(normals=False)[0].tobytes() == pa and c.get_indexed_mesh()[0].tobytes() == va
    finally:
        c.close()
