"""-m "not gpu": who owns a context's device and pinned memory, checked on the emulated runtime (tests/emu), which counts
the live allocations and can make the n-th following cudaMalloc / cudaMallocHost fail.

One scripted session on a small grid touches every buffer of the context: soup and indexed mesh, the normals modes,
refined vertices, the dense and block-field modes, seed mode, dual contouring, a grid step that makes the buffers grow,
and the queries with temporaries of their own.  Checked: close() gives every allocation back; a repeated identical
polygonise() allocates nothing once the buffers have settled; and an allocation that fails anywhere in the session makes
exactly the call that met it return MCB_E_NOMEM, after which the same context finishes the session with the bytes a
fresh context produces, also when it first polygonises a grid smaller than the one that failed to grow."""
import ctypes as C
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from .helpers import same_bits

GYR78 = ("((x*(-7+x^2*(56+x^2*(-112+64*x^2))))*(1+y^2*(-32+y^2*(160+y^2*(-256+128*y^2)))))"
         "+((y*(-7+y^2*(56+y^2*(-112+64*y^2))))*(1+z^2*(-32+z^2*(160+z^2*(-256+128*z^2)))))"
         "+((z*(-7+z^2*(56+z^2*(-112+64*z^2))))*(1+x^2*(-32+x^2*(160+x^2*(-256+128*x^2)))))")
PTS = np.array([[0.1, -0.2, 0.3], [0.5, 0.5, -0.5], [-0.9, 0.0, 0.7]], np.float32)


def alloc_stats(m):
    live, calls = C.c_longlong(), C.c_longlong()
    m.lib.mcb_emu_alloc_stats(C.byref(live), C.byref(calls))
    return live.value, calls.value


def fail_alloc(m, n):
    m.lib.mcb_emu_fail_alloc(C.c_longlong(n))


def set_grid(ctx, step):
    ctx.grid_step = step  # remembered: the failure sweep returns to it after visiting a smaller grid
    return ctx.set_grid_step(step)


def final_config(m, ctx):
    """the configuration the session ends in, as steps"""
    return [
        lambda: ctx.set_mesh_mode(m.MESH_SOUP | m.MESH_INDEXED),
        lambda: ctx.set_equation(GYR78),
        lambda: ctx.set_equation("x+y", slot=1),
        lambda: ctx.set_constraint(0, "<", 1.2),
        lambda: set_grid(ctx, 0.125),
        lambda: ctx.set_field_mode(m.FIELD_AUTO),
        lambda: ctx.set_normals(3),
        lambda: ctx.set_refine_vertices(True),
    ]


def session(m, ctx):
    """one API call per step, in order; the last step leaves the session's final configuration polygonised"""
    poly = ctx.polygonise
    ctx.grid_step = 0.25  # mcb_create's
    return [
        lambda: ctx.set_mesh_mode(m.MESH_SOUP | m.MESH_INDEXED),
        lambda: ctx.set_equation(GYR78),
        lambda: ctx.set_equation("x+y", slot=1),
        lambda: ctx.set_constraint(0, "<", 1.2),
        lambda: set_grid(ctx, 0.25),
        poly,                                               # soup + indexed mesh, normals mode 1
        lambda: ctx.set_normals(2), poly,
        lambda: ctx.set_normals(3), poly,
        lambda: ctx.set_refine_vertices(True), poly,
        lambda: ctx.set_refine_vertices(False),
        lambda: ctx.set_field_mode(m.FIELD_AUTO), poly,     # block-field mode
        lambda: ctx.set_field_mode(m.FIELD_DENSE), poly,
        lambda: ctx.set_seed(True, -0.75, -0.92, -0.75), poly,
        lambda: ctx.set_seed(False),
        lambda: ctx.set_mesh_mode(m.MESH_DC), poly,
        lambda: ctx.set_mesh_mode(m.MESH_SOUP | m.MESH_INDEXED),
        lambda: set_grid(ctx, 0.125),                       # M 9 -> 17: every buffer grows
        lambda: ctx.set_normals(2),
        lambda: ctx.set_seed(True, -0.75, -0.92, -0.75), poly,
        lambda: ctx.set_seed(False),
        lambda: ctx.set_field_mode(m.FIELD_AUTO), poly,
        lambda: ctx.set_mesh_mode(m.MESH_DC),
        lambda: ctx.set_normals(3), poly,
        ctx.get_cases,
        lambda: ctx.eval_points(PTS),
        lambda: ctx.eval_gradients(PTS),
        lambda: ctx.inspect_cube(-0.5, -0.25, 0.0),
        ctx.layer_triangles,
    ] + final_config(m, ctx) + [poly]


def status(m, step):
    """the status of one step: the negative code it returned or raised, else 0"""
    try:
        r = step()
    except m.McbError as e:
        return e.status
    return r if isinstance(r, int) and r < 0 else 0


def outputs(ctx):
    pos, nrm = ctx.get_mesh()
    return (pos, nrm) + ctx.get_indexed_mesh(normals=True)


def same_outputs(a, b):
    return len(a) == len(b) and all(x.shape == y.shape and (same_bits(x, y) if x.dtype == np.float32 else np.array_equal(x, y))
                                    for x, y in zip(a, b))


@pytest.fixture(scope="module")
def reference(mcb_emu):
    """the final configuration's outputs on a fresh context, and the session's allocation calls"""
    m = mcb_emu
    ctx = m.Context(0)
    for step in final_config(m, ctx):
        assert status(m, step) == 0
    ctx.polygonise()
    ref = outputs(ctx)
    ctx.close()
    calls0 = alloc_stats(m)[1]
    ctx = m.Context(0)
    for step in session(m, ctx):
        assert status(m, step) == 0
    assert same_outputs(outputs(ctx), ref)
    n = alloc_stats(m)[1] - calls0
    ctx.close()
    return ref, n


def test_session_returns_every_allocation(mcb_emu, reference):
    m = mcb_emu
    live0 = alloc_stats(m)[0]
    ctx = m.Context(0)
    for step in session(m, ctx):
        assert status(m, step) == 0
    assert alloc_stats(m)[0] > live0
    ctx.close()
    assert alloc_stats(m)[0] == live0


# Allocation calls of the first repeat once the M 17 grid has made the records grow: that repeat still grows the indexed
# mesh to the size prepare_buffers estimates from the grown records, and with it the normal.h scratch sized by the mesh.
FIRST_REPEAT_ALLOCS = {"dense": 6, "blocks": 6, "seed": 6, "dc": 9}


@pytest.mark.parametrize("mode", sorted(FIRST_REPEAT_ALLOCS))
def test_repeated_polygonise_allocates_nothing(mcb_emu, mode):
    m = mcb_emu
    ctx = m.Context(0)
    ctx.set_mesh_mode(m.MESH_DC if mode == "dc" else m.MESH_SOUP | m.MESH_INDEXED)
    assert ctx.set_equation(GYR78) == 0
    ctx.set_normals(2)
    ctx.set_field_mode(m.FIELD_AUTO if mode == "blocks" else m.FIELD_DENSE)
    assert ctx.set_seed(mode == "seed", -0.75, -0.92, -0.75) == 0
    for step, first in ((0.25, 0), (0.125, FIRST_REPEAT_ALLOCS[mode])):
        ctx.set_grid_step(step)
        grew = ctx.polygonise().reruns > 0
        assert grew == (first > 0)
        for expect in (first, 0, 0):
            calls = alloc_stats(m)[1]
            ctx.polygonise()
            assert alloc_stats(m)[1] - calls == expect
    ctx.close()


def _sweep(ns, ref, shrink):
    """the failure sweep over the allocations numbered ns, in a process of its own (its own allocation counts).  shrink:
    after the failure, polygonise on a grid smaller than any before, where the old sizes of every buffer suffice, and
    come back, before the failed step is re-issued"""
    from tests import emu
    m = emu.load()
    live0 = alloc_stats(m)[0]
    for n in ns:
        fail_alloc(m, n)
        target = alloc_stats(m)[1] + n
        try:
            ctx = m.Context(0)
        except m.McbError as e:
            assert e.status == m.MCB_E_NOMEM, n
            assert alloc_stats(m)[1] >= target and alloc_stats(m)[0] == live0, n
            continue
        assert alloc_stats(m)[1] < target, n  # a creation that met the failure raised above
        met = False
        for i, step in enumerate(session(m, ctx)):
            rc = status(m, step)
            if not met and alloc_stats(m)[1] >= target:
                met = True
                assert rc == m.MCB_E_NOMEM, (n, i, rc)
                if shrink:
                    back = ctx.grid_step
                    for s in (lambda: ctx.set_grid_step(0.5), ctx.polygonise, lambda: ctx.set_grid_step(back), ctx.polygonise):
                        assert status(m, s) == 0, (n, i)
                rc = status(m, step)  # re-issued: the failure fires once
            assert rc == 0, (n, i, rc)
        assert met, n
        assert same_outputs(outputs(ctx), ref), n
        ctx.close()
        assert alloc_stats(m)[0] == live0, n
    return len(ns)


@pytest.mark.parametrize("shrink", [False, True])
def test_every_failed_allocation_is_reported_and_recovered(reference, shrink):
    ref, n_alloc = reference
    workers = min(8, os.cpu_count() or 1)
    with ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn")) as ex:
        done = ex.map(_sweep, [range(1 + w, n_alloc + 1, workers) for w in range(workers)], [ref] * workers, [shrink] * workers)
        assert sum(done) == n_alloc
