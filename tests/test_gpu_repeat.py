"""-m gpu: repeating-surface mode (Marching::repeating_surface_mode + set_surface_repeat_step_distance,
marching.cpp:156-170, 481-494: every cube is polygonised with its own iso level) against the UNMODIFIED reference
(tests/golden/repeat_cases.npz, made by tests/golden/make_repeat_golden.py).

Bar: cube_code (against the cube's own level), tri_table row, per-cube triangle counts and the triangle soup byte for
byte; the welded Poly_Data expands to the reference's triangles, and is identical to it (with its normal.h normals)
wherever the reference does not merge coincident points of unrelated edges (see the comment in the test).
"""
import json
import os

import numpy as np
import pytest

from .helpers import load_repeat_golden, same_bits

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def rep():
    return load_repeat_golden(os.path.join(ROOT, "tests", "golden", "repeat_cases.npz"))


@pytest.fixture(scope="module")
def meta(rep):
    return json.loads(bytes(rep["meta_json"]).decode())


NAMES = ["rep_sphere_20", "rep_sphere_iso", "rep_eq1_ctor", "rep_eq1_gui", "rep_torus_24", "rep_eq8_gui", "rep_gyr78_17",
         "rep_quirk_div", "rep_testdrawer", "rep_cons"]


def setup(mcb, c, case, on=True):
    assert c.set_equation(case["eq"]) == 0
    assert c.set_grid_step(case["step"]) == case["M"]
    c.set_scaling(*case["scale"])
    c.set_surface_constant(case["iso"])
    for i in range(3):
        c.set_constraint(i, ">", 0.0, False)
    for i, (lhs, op, rhs) in enumerate(case["cons"]):
        assert c.set_equation(lhs, slot=i + 1) == 0
        assert c.set_constraint(i, op, rhs, True) == 0
    assert c.set_repeat(on, case["dist"]) == 0


@pytest.mark.parametrize("name", NAMES)
def test_repeating_surface_mode_equals_the_reference(mcb, rep, meta, name):
    case = meta[name]
    c = mcb.Context(0)
    c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
    c.set_normals(2)
    setup(mcb, c, case)
    cnt = c.polygonise()
    assert cnt.M == case["M"]
    code, tidx = c.get_cases()
    gcode = rep[name + "/code"]
    act = (gcode != 0) & (gcode != 255)
    assert np.array_equal((code != 0) & (code != 255), act), "active set"
    assert np.array_equal(code[act], gcode[act]), "cube_code of the active cubes"
    assert np.array_equal(tidx[act], rep[name + "/table_idx"][act]), "table_idx"
    assert (cnt.active, cnt.triangles, cnt.ambiguous, cnt.redirected) == (case["active"], case["T"], case["ambiguous"], case["redirected"])
    pos, _ = c.get_mesh(normals=False)
    assert same_bits(pos[:, :, :3], rep[name + "/soup"]), "soup"
    vl, tl, vn = c.get_indexed_mesh(normals=True)
    # Welded mesh.  Marching::interp keeps interpolating towards the surface constant itself (marching.cpp:437-446), so in
    # this mode the crossing points are extrapolated along their edges, and on regular grids points of unrelated, distant
    # edges happen to coincide; the reference's std::set merges those too.  The GPU weld is local (cubes sharing a grid
    # edge, and the neighbourhood of a grid vertex): it never merges more than the reference, every triangle has the
    # reference's corner positions, and where no such coincidence exists the meshes are identical.
    gv, gt = rep[name + "/vertex_list"], rep[name + "/tri_list"].astype(np.int64)
    # (the other way round, the reference's non-transitive tolerance comparator sometimes misses an equal element and
    #  keeps a duplicate — the deviation documented for the plain mode in DESIGN.md; those are the near-pairs counted here)
    from scipy.spatial import cKDTree
    finite = gv[~np.isnan(gv).any(axis=1)].astype(np.float64)
    kept_duplicates = len(cKDTree(finite).query_pairs(1e-6, p=np.inf)) if len(finite) else 0
    assert cnt.vertices >= case["V"] - kept_duplicates
    assert tl.shape == gt.shape
    if len(gt):
        # first-inserted-wins under a 1e-6 per-axis tolerance that is not transitive: a corner can sit a few 1e-6 from the
        # representative the reference's set happened to keep
        assert np.abs(vl[tl.astype(np.int64)].astype(np.float64) - gv[gt].astype(np.float64)).max() <= 4e-6
    if cnt.vertices == case["V"]:
        assert same_bits(vl, gv), "vertex_list"
        assert np.array_equal(tl, gt), "tri_list"
        assert same_bits(vn, rep[name + "/normals"]), "normal.h normals"
    # gradient normals still work (no parity target in the reference: just finite where the field is)
    c.set_normals(1)
    c.polygonise()
    _, nrm = c.get_mesh(normals=True)
    assert nrm.shape == pos.shape
    # and the mode switches off cleanly
    assert c.set_repeat(False) == 0
    off = c.polygonise()
    assert off.triangles != cnt.triangles or off.active != cnt.active or cnt.triangles == 0
    c.close()


def test_repeat_argument_and_state_errors(mcb):
    c = mcb.Context(0)
    assert c.set_repeat(True, 0.0) == mcb.MCB_E_ARG and c.set_repeat(True, -1.0) == mcb.MCB_E_ARG
    assert c.set_repeat(True, 0.5) == 0
    assert c.set_seed(True, 0.0, 0.0, 0.0) == 0
    with pytest.raises(mcb.McbError):
        c.polygonise()
    c.set_seed(False)
    c.set_field_mode(mcb.FIELD_SPARSE)  # ignored while every cube reads the field
    cnt = c.polygonise()
    assert cnt.field_mode == mcb.FIELD_DENSE
    c.close()


def test_inspect_cube_reports_the_cube_level(mcb, rep, meta):
    case = meta["rep_sphere_20"]
    c = mcb.Context(0)
    setup(mcb, c, case)
    M, axis = mcb.grid_axis(case["step"])
    gcode = rep["rep_sphere_20/code"].reshape(M, M, M)
    rng = np.random.default_rng(5)
    for _ in range(40):
        i, j, k = (int(v) for v in rng.integers(0, M, 3))
        sd = c.inspect_cube(float(axis[i]), float(axis[j]), float(axis[k]))
        vals = np.array(sd.corner_values[:], np.float32)
        lvl = np.float32(sd.surf_constant)
        a = np.floor((vals.max() - np.float32(case["iso"])) / np.float32(case["dist"]))
        assert lvl == np.float32(case["iso"]) + np.float32(case["dist"]) * np.float32(a)
        if gcode[k, j, i] not in (0, 255):
            assert sd.cube_code == gcode[k, j, i]
    c.close()
