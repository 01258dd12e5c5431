"""-m gpu: the kernels of one polygonisation overlap their neighbours on the stream (programmatic dependent launch, DESIGN.md
§5 "The wait rule") and the tile scan is part of compact_kernel.  Every output must be the bytes a fully serialised run
gives: $MCB_DEBUG_SYNC=1 waits for each kernel right after its launch, so no kernel can start before the previous one has
finished.  The variable is read once per process, hence one worker process per setting, running the same scenarios."""
import hashlib
import importlib
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "marching-cube-for-implicit-surfaces_b200"

SPHERE = "x^2+y^2+z^2-0.49"
TORUS = "(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)"
GYR78 = ("((x*(-7+x^2*(56+x^2*(-112+64*x^2))))*(1+y^2*(-32+y^2*(160+y^2*(-256+128*y^2)))))"
         "+((y*(-7+y^2*(56+y^2*(-112+64*y^2))))*(1+z^2*(-32+z^2*(160+z^2*(-256+128*z^2)))))"
         "+((z*(-7+z^2*(56+z^2*(-112+64*z^2))))*(1+x^2*(-32+x^2*(160+x^2*(-256+128*x^2)))))")
CSG = "max(sqrt(x^2+y^2+z^2)-0.7,-(sqrt(x^2+y^2)-0.3))"  # sphere minus a cylinder (function grammar)
HEADLINE_LAUNCHES = 12  # axis_tables, bounds, super/block classes, decided signs, block fill, classify, ambiguity, compact, field list, apron fill, emit


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(a.tobytes())
    return h.hexdigest()


def _run(ctx, out, name, soup=True, indexed=False):
    """one polygonisation: its counts and the digests of the soup (positions, normals) and the welded mesh"""
    c = ctx.polygonise()
    rec = {k: int(getattr(c, k)) for k in ("active", "triangles", "ambiguous", "redirected", "vertices", "reruns", "launches", "field_mode")}
    if soup:
        rec["soup"] = _digest(*ctx.get_mesh())
    if indexed:
        rec["indexed"] = _digest(*ctx.get_indexed_mesh(normals=True))
    out[name] = rec


def worker():
    """every scenario once, in this process; prints {scenario: counts and output digests} as one JSON line"""
    sys.path.insert(0, ROOT)
    mcb = importlib.import_module(PKG)
    out = {}

    def fresh(eq, n, normals=1, mode=None, field=None, grammar=None):
        ctx = mcb.Context(0)
        if grammar is not None:
            ctx.set_grammar(grammar)
        assert ctx.set_equation(eq) == 0
        ctx.jit_wait()
        ctx.set_grid_step(2.0 / n)
        ctx.set_field_mode(mcb.FIELD_AUTO if field is None else field)
        ctx.set_mesh_mode(mcb.MESH_SOUP if mode is None else mode)
        ctx.set_normals(normals)
        ctx.set_stage_timing(False)  # as bench.py's timed loop: no events between the kernels
        return ctx

    ctx = fresh(SPHERE, 256)  # the headline configuration, smaller
    _run(ctx, out, "headline_sphere")
    ctx.close()
    for name, eq in (("sphere", SPHERE), ("torus", TORUS), ("gyr78", GYR78)):
        for field in (mcb.FIELD_AUTO, mcb.FIELD_DENSE):
            ctx = fresh(eq, 128, field=field)
            _run(ctx, out, "%s_%s" % (name, "blocks" if field == mcb.FIELD_AUTO else "dense"))
            ctx.close()
    ctx = fresh(CSG, 128, grammar=mcb.GRAMMAR_FUNCTIONS)
    _run(ctx, out, "csg")
    ctx.close()
    ctx = fresh(SPHERE, 128)
    assert ctx.set_equation("x-0.1", slot=1) == 0 and ctx.set_constraint(0, ">", 0.0, True) == 0
    _run(ctx, out, "constraint")
    ctx.close()
    ctx = fresh(TORUS, 128)
    assert ctx.set_seed(True, 0.74, 0.0, 0.0) == 0
    _run(ctx, out, "seed", indexed=False)
    ctx.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
    _run(ctx, out, "seed_indexed", indexed=True)
    ctx.close()
    ctx = fresh(SPHERE, 128)
    assert ctx.set_repeat(True, 0.25) == 0
    _run(ctx, out, "repeat")
    ctx.close()
    ctx = fresh(GYR78, 128, mode=mcb.MESH_SOUP | mcb.MESH_INDEXED)
    _run(ctx, out, "indexed", indexed=True)
    ctx.set_normals(2)
    _run(ctx, out, "indexed_normal_h", soup=False, indexed=True)
    ctx.close()
    ctx = fresh(TORUS, 128, normals=3, mode=mcb.MESH_SOUP | mcb.MESH_INDEXED)
    ctx.set_refine_vertices(True)
    _run(ctx, out, "refined_analytic_normals", indexed=True)
    ctx.close()
    ctx = fresh(GYR78, 128)
    M = ctx.set_grid_step(2.0 / 128)
    ctx.set_slab(M // 3, 2 * M // 3)
    _run(ctx, out, "slab")
    ctx.close()
    # one context, the surface constant changing and a buffer growing in the middle: the re-run path
    ctx = fresh(SPHERE, 128, mode=mcb.MESH_SOUP | mcb.MESH_INDEXED)
    for i, (eq, iso) in enumerate(((SPHERE, -0.45), (GYR78, 0.0), (GYR78, 0.05), (SPHERE, 0.2), (SPHERE, -0.3))):
        assert ctx.set_equation(eq) == 0
        ctx.jit_wait()
        ctx.set_surface_constant(iso)
        _run(ctx, out, "sequence_%d" % i, indexed=True)
    ctx.close()
    sys.stdout.write(json.dumps(out) + "\n")


def _worker_output(debug_sync):
    env = dict(os.environ)
    env.pop("MCB_DEBUG_SYNC", None)
    if debug_sync:
        env["MCB_DEBUG_SYNC"] = "1"
    r = subprocess.run([sys.executable, "-m", "tests.test_gpu_launch_chain"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert "MCB_DEBUG_SYNC: kernel" not in r.stderr, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.fixture(scope="module")
def runs():
    return _worker_output(False), _worker_output(True)


SCENARIOS = ["headline_sphere", "sphere_blocks", "sphere_dense", "torus_blocks", "torus_dense", "gyr78_blocks", "gyr78_dense", "csg",
             "constraint", "seed", "seed_indexed", "repeat", "indexed", "indexed_normal_h", "refined_analytic_normals", "slab"] + \
            ["sequence_%d" % i for i in range(5)]


@pytest.mark.parametrize("name", SCENARIOS)
def test_outputs_equal_serialised_run(runs, name):
    overlapped, serialised = runs
    assert overlapped[name]["triangles"] > 0
    assert overlapped[name] == serialised[name]


def test_sequence_grows_a_buffer(runs):
    assert any(runs[0]["sequence_%d" % i]["reruns"] > 0 for i in range(5))


def test_headline_launch_count(runs):
    assert runs[0]["headline_sphere"]["launches"] == HEADLINE_LAUNCHES


if __name__ == "__main__":
    worker()
