"""GPU tier of dual contouring (MCB_MESH_DC, DESIGN.md §14): the device mesh equals the host build (tests/cpp/dc_host.cpp)
bit for bit, and stays byte-identical across field modes, field kernels, stage timing, $MCB_DEBUG_SYNC, a changed surface
constant and buffer growth; constraints, both normals modes, mcb_headless / the C++ drop-in and the Python mirror."""
import hashlib
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_UNION2, CSG_UNION8
from .dc_common import BOX, MESH_DC, SPHERE, host_dc, run_dc
from .functions_common import GYROID, TORUS_SDF
from .helpers import same_bits
from .normals_common import host_normalise

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "mcb_headless")
TORUS_GOLDEN = "(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)"
CASES = [SPHERE, TORUS_GOLDEN, TORUS_SDF, GYROID, BOX, CSG_UNION2, CSG_BOX_SDF, CSG_UNION8]


def _digest(r):
    h = hashlib.sha256()
    for a in (r["vl"], r["tl"]) + ((r["vn"],) if r.get("vn") is not None else ()):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _same_as_host(r, d):
    return r["counts"].vertices == r["counts"].active == len(d["vl"]) and same_bits(r["vl"], d["vl"]) and np.array_equal(r["tl"], d["tl"])


@pytest.mark.parametrize("eq", CASES)
def test_device_equals_host(mcb, eq):
    d = host_dc(eq, 2 / 64)
    r = run_dc(mcb, eq, 2 / 64)
    assert r["counts"].mesh_mode == MESH_DC and r["counts"].triangles == len(d["tl"]) > 0
    assert _same_as_host(r, d), eq


@pytest.mark.parametrize("eq", [SPHERE, GYROID, CSG_UNION2])
def test_bytes_do_not_depend_on_field_mode_field_kernel_or_timing(mcb, eq):
    runs = {}
    for fm in (mcb.FIELD_DENSE, mcb.FIELD_SPARSE, mcb.FIELD_AUTO):
        for jit in (mcb.JIT_OFF, mcb.JIT_ON):
            for timing in (True, False):
                runs[(fm, jit, timing)] = _digest(run_dc(mcb, eq, 2 / 96, normals=3, field_mode=fm, jit=jit, timing=timing))
    assert len(set(runs.values())) == 1, runs


def test_changed_surface_constant_and_buffer_growth(mcb):
    ctx = mcb.Context(0)
    try:
        ctx.set_mesh_mode(MESH_DC)
        ctx.set_grammar(mcb.GRAMMAR_FUNCTIONS)
        grew = False
        for eq, n, iso in ((SPHERE, 24, 0.0), (SPHERE, 24, 0.1), (GYROID, 80, 0.0), (GYROID, 80, 0.3), (SPHERE, 160, -0.2)):
            assert ctx.set_equation(eq) == 0
            ctx.set_grid_step(2 / n)
            ctx.set_surface_constant(iso)
            ctx.set_normals(0)
            cnt = ctx.polygonise()
            grew |= cnt.reruns > 0
            vl, tl = ctx.get_indexed_mesh()
            d = host_dc(eq, 2 / n, iso=iso)
            assert _same_as_host({"counts": cnt, "vl": vl, "tl": tl}, d), (eq, n, iso)
        assert grew
    finally:
        ctx.close()


_DEBUG_CASES = [(SPHERE, 80), (GYROID, 64), (CSG_UNION8, 64)]


def _worker():
    mcb = __import__("importlib").import_module("marching-cube-for-implicit-surfaces_b200")
    out = {}
    for eq, n in _DEBUG_CASES:
        for fm in (mcb.FIELD_DENSE, mcb.FIELD_AUTO):
            out["%s/%d/%d" % (eq, n, fm)] = _digest(run_dc(mcb, eq, 2 / n, normals=2, field_mode=fm))
    sys.stdout.write(json.dumps(out) + "\n")


def test_debug_sync_gives_the_same_bytes():
    res = []
    for sync in (False, True):
        env = dict(os.environ)
        env.pop("MCB_DEBUG_SYNC", None)
        if sync:
            env["MCB_DEBUG_SYNC"] = "1"
        r = subprocess.run([sys.executable, "-c", "from tests.test_gpu_dc import _worker; _worker()"], cwd=ROOT, env=env,
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        assert "MCB_DEBUG_SYNC: kernel" not in r.stderr
        res.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert res[0] == res[1]


@pytest.mark.parametrize("eq,cons", [(SPHERE, (("x+0.3y", "<", 0.25),)), (GYROID, (("z", ">=", -0.3), ("x^2", "<", 0.5))),
                                     (BOX, (("x-y", "<=", 0.1),))])
def test_constraints_drop_the_quads_the_host_drops(mcb, eq, cons):
    d = host_dc(eq, 2 / 64, cons=cons)
    free = host_dc(eq, 2 / 64)
    assert len(d["tl"]) < len(free["tl"])
    for fm in (mcb.FIELD_DENSE, mcb.FIELD_AUTO):
        assert _same_as_host(run_dc(mcb, eq, 2 / 64, cons=cons, field_mode=fm), d), (eq, fm)


def _normal_h(vl, tl):
    """CalculateNormal (normal.h:3-42) restated in fp32: face normals glm::cross(B-A, C-A), summed per vertex in triangle
    order, x * (1 / sqrt(dot))"""
    v = vl.astype(np.float32)
    a, b, c = v[tl[:, 0]], v[tl[:, 1]] - v[tl[:, 0]], v[tl[:, 2]] - v[tl[:, 0]]
    fn = np.stack([b[:, 1] * c[:, 2] - c[:, 1] * b[:, 2], b[:, 2] * c[:, 0] - c[:, 2] * b[:, 0], b[:, 0] * c[:, 1] - c[:, 0] * b[:, 1]], 1)
    acc = np.zeros_like(v)
    for t in range(len(tl)):
        for s in range(3):
            acc[tl[t, s]] = fn[t] + acc[tl[t, s]]
    with np.errstate(all="ignore"):
        dot = (acc[:, 0] * acc[:, 0] + acc[:, 1] * acc[:, 1]) + acc[:, 2] * acc[:, 2]
        return acc * (np.float32(1) / np.sqrt(dot))[:, None]


@pytest.mark.parametrize("eq", [SPHERE, BOX, CSG_UNION2])
def test_normals_modes_2_and_3(mcb, eq):
    r3 = run_dc(mcb, eq, 2 / 48, normals=3)
    ctx = mcb.Context(0)
    try:
        ctx.set_grammar(mcb.GRAMMAR_FUNCTIONS)
        ctx.set_equation(eq)
        g = ctx.eval_gradients(r3["vl"], apply_scale=True)
    finally:
        ctx.close()
    assert same_bits(r3["vn"], host_normalise(g))
    r2 = run_dc(mcb, eq, 2 / 48, normals=2)
    assert same_bits(r2["vl"], r3["vl"]) and np.array_equal(r2["tl"], r3["tl"])
    used = np.unique(r2["tl"])
    assert same_bits(r2["vn"][used], _normal_h(r2["vl"], r2["tl"])[used])


def test_headless_and_cpp_dropin_give_the_ctypes_bytes(mcb, tmp_path):
    dump, nrm = tmp_path / "m.bin", tmp_path / "n.bin"
    subprocess.check_call([EXE, "--functions", "--eq", BOX, "--res", "64", "--scale", "1", "1", "1", "--dual-contouring", "--dump", str(dump),
                           "--dump-normals", str(nrm)], stdout=subprocess.DEVNULL)
    b = dump.read_bytes()
    nv, nt = struct.unpack("<QQ", b[:16])
    vl = np.frombuffer(b[16:16 + 12 * nv], np.float32).reshape(-1, 3)
    tl = np.frombuffer(b[16 + 12 * nv:], np.uint32).reshape(-1, 3)
    r = run_dc(mcb, BOX, 2 / 64, normals=3)
    assert nt == len(r["tl"]) and same_bits(vl, r["vl"]) and np.array_equal(tl, r["tl"])
    assert same_bits(np.fromfile(str(nrm), np.float32).reshape(-1, 3), r["vn"])
    bad = subprocess.run([EXE, "--functions", "--eq", BOX, "--res", "64", "--dual-contouring", "--devices", "2"], capture_output=True, text=True)
    assert bad.returncode == 1 and "dual contouring runs on one device" in bad.stderr


def test_python_marching_mirror(mcb):
    m = mcb.Marching()
    e = mcb.Evaluator()
    e.set_function_grammar(True)
    assert e.set_equation(BOX)
    m.set_evaluator(e)
    m.set_grid_resolution(64)
    m.set_dual_contouring(True)
    m.set_normals(0)
    assert m.recalculate()
    p = m.get_poly_data()
    r = run_dc(mcb, BOX, 2 / 64)
    assert same_bits(p.vertex_list, r["vl"].reshape(-1)) and np.array_equal(p.tri_list, r["tl"].reshape(-1))


def test_literal_gyroid_at_1024_is_deterministic(mcb):
    a = run_dc(mcb, GYROID, 2 / 1024, normals=3, field_mode=mcb.FIELD_AUTO)
    b = run_dc(mcb, GYROID, 2 / 1024, normals=3, field_mode=mcb.FIELD_AUTO)
    assert a["counts"].triangles > 10 ** 7
    assert _digest(a) == _digest(b)
