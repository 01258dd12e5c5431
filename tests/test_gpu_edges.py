"""-m gpu: edge cases of the path — the finest step the reference accepts (0.001: the fp32-accumulated grid drifts by
1.9e-5, SURVEY.md A.3), a step below it (2048^3, SURVEY.md D4), the coarsest grids, empty and all-NaN fields,
capacity growth on the first call, and slabs that do not start at layer 0.  The reference (or, where oracle/_ref is not
built, its restatement: see the `refbind` fixture) is executed live on the same layers."""
import numpy as np
import pytest

from .helpers import same_bits

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("eq,step,force", [("x+y", 0.001, False), ("x*y-z", 0.001, False), ("x+y", 2.0 / 2048, True)])
def test_finest_grids_one_layer_against_live_reference(mcb, refbind, eq, step, force):
    r = refbind.Ref(eq, step, force_step=force)
    M, coords = r.coords()
    Mg, cg = mcb.grid_axis(step)
    assert Mg == M and same_bits(cg, coords)  # the accumulated loop coordinates, not -1 + i*h
    c = mcb.Context(0)
    c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
    assert c.set_equation(eq) == 0 and c.set_grid_step(step) == M
    for k0 in (0, M // 2, M - 1):
        c.set_slab(k0, k0 + 1)
        cnt = c.polygonise()
        sw = r.sweep(k0, k0 + 1, soup=True)
        code, tidx = c.get_cases()
        assert np.array_equal(code, sw["code"]) and np.array_equal(tidx, sw["table_idx"])
        assert cnt.triangles == sw["T"] and cnt.active == sw["active"]
        pos, _ = c.get_mesh()
        assert same_bits(pos[:, :, :3], sw["soup"])
        vl, tl = c.get_indexed_mesh()
        if len(tl):
            assert np.abs(vl[tl.astype(np.int64)].astype(np.float64) - sw["soup"].astype(np.float64)).max() < 1e-6
    c.close()


@pytest.mark.parametrize("step,M", [(1.0, 3), (0.5, 5), (0.3, 8)])
def test_coarsest_grids(mcb, refbind, step, M):
    """Steps above the reference's 0.5 limit are accepted by the C ABI (the class clamps); a handful of cubes."""
    c = mcb.Context(0)
    c.set_mesh_mode(3)
    assert c.set_equation("x^2+y^2+z^2-0.49") == 0 and c.set_grid_step(step) == M
    cnt = c.polygonise()
    if refbind.available():
        r = refbind.Ref("x^2+y^2+z^2-0.49", step, force_step=True)
        sw = r.sweep(soup=True)
        assert cnt.triangles == sw["T"]
        pos, _ = c.get_mesh()
        assert same_bits(pos[:, :, :3], sw["soup"])
    assert cnt.cubes == M ** 3
    c.close()


@pytest.mark.parametrize("eq", ["x^2+y^2+z^2+1", "(x-x)/(y-y)", "0*x-1"])
def test_empty_and_nan_fields(mcb, eq):
    c = mcb.Context(0)
    c.set_mesh_mode(3)
    assert c.set_equation(eq) == 0 and c.set_grid_step(0.05) == 41
    cnt = c.polygonise()
    assert (cnt.active, cnt.triangles, cnt.vertices) == (0, 0, 0)
    pos, nrm = c.get_mesh()
    vl, tl = c.get_indexed_mesh()
    assert pos.shape[0] == 0 and vl.shape[0] == 0 and tl.shape[0] == 0
    code, tidx = c.get_cases()
    assert not code.any() or set(np.unique(code)) <= {0, 255}
    c.close()


def test_first_call_grows_buffers_then_settles(mcb):
    """A dense surface on a fresh context: the first call has to grow the record / soup / vertex buffers (reruns > 0),
    the second one does not, and both give the same mesh."""
    from oracle.refbind import GYR78
    c = mcb.Context(0)
    c.set_mesh_mode(3)
    assert c.set_equation(GYR78) == 0 and c.set_grid_step(2.0 / 128) == 129
    a = c.polygonise()
    pa, _ = c.get_mesh()
    va, ta = c.get_indexed_mesh()
    b = c.polygonise()
    pb, _ = c.get_mesh()
    vb, tb = c.get_indexed_mesh()
    assert a.reruns > 0 and b.reruns == 0
    assert (a.triangles, a.active, a.vertices) == (b.triangles, b.active, b.vertices)
    assert same_bits(pa, pb) and same_bits(va, vb) and np.array_equal(ta, tb)
    c.close()


def test_slab_in_the_middle_equals_the_same_layers_of_the_full_grid(mcb):
    c = mcb.Context(0)
    assert c.set_equation("(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)") == 0 and c.set_grid_step(2.0 / 64) == 65
    full = c.polygonise()
    code_f, tidx_f = c.get_cases()
    rec_f, off_f = c.get_active()
    pos_f, nrm_f = c.get_mesh()
    k0, k1 = 20, 41
    c.set_slab(k0, k1)
    s = c.polygonise()
    code_s, tidx_s = c.get_cases()
    pos_s, nrm_s = c.get_mesh()
    M = full.M
    assert np.array_equal(code_s, code_f[k0 * M * M:k1 * M * M]) and np.array_equal(tidx_s, tidx_f[k0 * M * M:k1 * M * M])
    kk = ((rec_f >> 24) & 0xFFF).astype(np.int64)
    first = int(off_f[np.argmax(kk >= k0)])
    assert same_bits(pos_s, pos_f[first:first + s.triangles]) and same_bits(nrm_s, nrm_f[first:first + s.triangles])
    c.close()


def test_truncated_passes_are_harmless(mcb):
    """A grid that outgrows every buffer: the first pass of the call runs with too small record, soup and mesh buffers and is
    repeated by the host.  Its kernels must stay inside their buffers whatever the truncated state looks like (weld_emit once
    took the end of a truncated chunk from shared memory another warp was still writing: an intermittent illegal access).
    Many fresh contexts, so that the truncated pass meets many different leftovers in shared and global memory."""
    ref = None
    for rep in range(24):
        c = mcb.Context(0)
        c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        c.set_normals(1)
        c.set_field_mode(mcb.FIELD_DENSE if rep % 2 else mcb.FIELD_AUTO)
        assert c.set_equation("x^2+y^2+z^2-0.49") == 0
        c.set_grid_step(2.0 / (12 + rep))                 # small buffers
        c.polygonise()
        c.set_scaling(1.1, 0.9, 1.0)
        c.set_surface_constant(0.01)
        c.set_grid_step(2.0 / 257)                        # every buffer too small: truncated pass + repeat
        cnt = c.polygonise()
        assert cnt.reruns >= 1
        got = (cnt.triangles, cnt.active, cnt.vertices)
        ref = ref or got
        assert got == ref
        v, t, n = c.get_indexed_mesh(normals=True)
        assert len(v) == cnt.vertices and len(t) == cnt.triangles and int(t.max()) == cnt.vertices - 1
        c.close()


def test_contexts_on_several_host_threads(mcb):
    """One context per host thread (how Marching::set_devices drives several GPUs, and how the reference's "movie" thread
    calls recalculate(), drawer.cpp:135): contexts share nothing but the lazily loaded NVRTC / NCCL entry points, so four
    threads polygonising different equations at once — new equations, i.e. background compiles included — must each get
    what a single thread gets."""
    import threading
    from oracle.refbind import GYR78
    eqs = ["x^2+y^2+z^2-0.49", GYR78, "(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)", "x*y*z+0.05*x-0.01"]
    grids = [96, 64, 80, 72]

    def run(eq, n, out, reps):
        c = mcb.Context(0)
        c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
        c.set_normals(1)
        assert c.set_equation(eq) == 0
        c.set_grid_step(2.0 / n)
        res = None
        for r in range(reps):
            c.set_surface_constant(0.001 * (r % 3))
            cnt = c.polygonise()
            if r % 3 == 0:
                pos, nrm = c.get_mesh(normals=True)
                v, t, vn = c.get_indexed_mesh(normals=True)
                cur = (cnt.triangles, cnt.active, cnt.vertices, pos.tobytes(), nrm.tobytes(), v.tobytes(), t.tobytes())
                assert res is None or cur == res      # interpreter before, compiled kernels after: the same bytes
                res = cur
        c.close()
        out.append(res)

    single = []
    for eq, n in zip(eqs, grids):
        run(eq, n, single, 1)
    outs = [[] for _ in eqs]
    threads = [threading.Thread(target=run, args=(eq, n, o, 30)) for eq, n, o in zip(eqs, grids, outs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for s, o in zip(single, outs):
        assert len(o) == 1 and o[0] == s and s[0] > 0
