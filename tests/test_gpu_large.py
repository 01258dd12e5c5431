"""-m gpu: larger grids.  256^3 (M=257): counts against SURVEY.md Appendix B (made with the unmodified reference) for
all eight example equations, plus live per-cube comparison against the `refbind` fixture on a few z-layers.  1024^3: size-
independent properties (slab additivity, determinism, symmetric-field symmetry)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# SURVEY.md Appendix B, step 2/256, scale 1, iso 0: triangles of the reference's full run
T257 = {1: 263682, 2: 266244, 3: 153868, 4: 240532, 5: 369792, 6: 186060, 7: 78928, 8: 370672}


@pytest.mark.parametrize("n", range(1, 9))
def test_examples_at_256(mcb, n):
    from oracle.refbind import EXAMPLE_EQUATIONS
    c = mcb.Context(0)
    assert c.set_equation(EXAMPLE_EQUATIONS[n]) == 0
    assert c.set_grid_step(2.0 / 256) == 257
    cnt = c.polygonise()
    assert cnt.triangles == T257[n]
    c.close()


@pytest.mark.parametrize("eq,T", [("x^2+y^2+z^2-0.49", 302792), ("(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)", 232128)])
def test_sphere_torus_at_256(mcb, eq, T):
    c = mcb.Context(0)
    assert c.set_equation(eq) == 0
    assert c.set_grid_step(2.0 / 256) == 257
    assert c.polygonise().triangles == T
    c.close()


@pytest.mark.parametrize("n", [2, 3, 8])
def test_layers_against_live_reference_at_256(mcb, refbind, n):
    """Per-cube cube_code / table_idx / soup for a handful of z-layers of the 257^3 grid, reference executed live."""
    from .helpers import same_bits
    eq = refbind.EXAMPLE_EQUATIONS[n]
    r = refbind.Ref(eq, 2.0 / 256)
    c = mcb.Context(0)
    assert c.set_equation(eq) == 0 and c.set_grid_step(2.0 / 256) == 257
    for (k0, k1) in [(0, 1), (127, 130), (200, 201), (256, 257)]:
        c.set_slab(k0, k1)
        cnt = c.polygonise()
        code, tidx = c.get_cases()
        sw = r.sweep(k0, k1, soup=True)
        assert np.array_equal(code, sw["code"]) and np.array_equal(tidx, sw["table_idx"])
        assert cnt.triangles == sw["T"]
        pos, _ = c.get_mesh()
        assert same_bits(pos[:, :, :3], sw["soup"])
    c.close()


def test_1024_properties(mcb):
    """1025^3 cubes: determinism, slab additivity and mirror symmetry of the sphere's triangle count."""
    c = mcb.Context(0)
    assert c.set_equation("x^2+y^2+z^2-0.49") == 0
    assert c.set_grid_step(2.0 / 1024) == 1025
    a = c.polygonise()
    b = c.polygonise()
    assert (a.triangles, a.active) == (b.triangles, b.active) and a.cubes == 1025 ** 3
    assert b.reruns == 0
    T, A = 0, 0
    for r in range(4):
        k0, k1 = mcb.slab_range(1025, r, 4)
        c.set_slab(k0, k1)
        s = c.polygonise()
        T += s.triangles; A += s.active
    assert (T, A) == (a.triangles, a.active)
    c.close()


LIVE_1024 = [
    ("x^2+y^2+z^2-0.49", (154, 512, 870)),                       # BASELINE.json configs[2]
    ("(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)", (512,)),           # configs[2], torus: `^` of a three-variable sum
]   # (the polynomial gyroid has its own test below: its layer is spread over the host threads)


@pytest.mark.parametrize("eq,layers", LIVE_1024)
def test_layers_against_live_reference_at_1024(mcb, refbind, eq, layers):
    """BASELINE.json configs[2] at full size: z-layers of the 1025^3-cube grid (1.05 M cubes each), cube codes,
    table rows and the triangle soup bit-exact against the reference executed live; plus the welded layer."""
    from .helpers import same_bits
    r = refbind.Ref(eq, 2.0 / 1024)
    c = mcb.Context(0)
    c.set_mesh_mode(mcb.MESH_SOUP | mcb.MESH_INDEXED)
    assert c.set_equation(eq) == 0 and c.set_grid_step(2.0 / 1024) == 1025
    for k0 in layers:
        c.set_slab(k0, k0 + 1)
        cnt = c.polygonise()
        sw = r.sweep(k0, k0 + 1, soup=True)
        code, tidx = c.get_cases()
        assert np.array_equal(code, sw["code"]) and np.array_equal(tidx, sw["table_idx"])
        assert cnt.triangles == sw["T"] and cnt.triangles > 0
        assert (cnt.ambiguous, cnt.redirected) == (sw["ambiguous"], sw["redirected"])
        pos, _ = c.get_mesh()
        assert same_bits(pos[:, :, :3], sw["soup"])
        vl, tl = c.get_indexed_mesh()
        assert np.abs(vl[tl.astype(np.int64)].astype(np.float64) - sw["soup"].astype(np.float64)).max() < 1e-6
    c.close()


def test_gyr78_layer_against_live_reference_at_1024(mcb, refbind):
    """BASELINE.json configs[3] at full size: one z-layer of the 1025^3-cube grid of the polynomial gyroid — the field that
    exercises the ambiguity redirect at scale — per cube against the UNMODIFIED reference run live (marching.cpp:456-595,
    redirect :521-549), its 1.05 M calculate_step calls spread over the host threads: cube codes, table rows, ambiguous and
    redirected counts and the triangle soup, bit for bit."""
    from .helpers import same_bits
    eq = refbind.GYR78
    c = mcb.Context(0)
    c.set_field_mode(mcb.FIELD_AUTO)
    c.set_normals(0)
    assert c.set_equation(eq) == 0 and c.set_grid_step(2.0 / 1024) == 1025
    # the whole grid first: which layers hold cubes whose triangles come from the redirected row 255 - code?
    full = c.polygonise()
    assert full.redirected > 0 and full.ambiguous >= full.redirected
    rec, _ = c.get_active()
    redirected = rec[((rec >> 36) & 0xFF) != ((rec >> 44) & 0xFF)]
    assert len(redirected) == full.redirected
    layers = sorted(set(int(k) for k in ((redirected >> 24) & 0xFFF)))
    seen_amb = seen_red = 0
    for k0 in (512, layers[0], layers[len(layers) // 2]):
        c.set_slab(k0, k0 + 1)
        cnt = c.polygonise()
        sw = refbind.sweep_rows_mt(eq, 2.0 / 1024, k0 * 1025, (k0 + 1) * 1025)
        code, tidx = c.get_cases()
        assert np.array_equal(code, sw["code"]) and np.array_equal(tidx, sw["table_idx"])
        assert cnt.triangles == sw["T"] and cnt.triangles > 10000
        assert (cnt.active, cnt.ambiguous, cnt.redirected) == (sw["active"], sw["ambiguous"], sw["redirected"])
        pos, _ = c.get_mesh(normals=False)
        assert same_bits(pos[:, :, :3], sw["soup"])
        seen_amb += cnt.ambiguous; seen_red += cnt.redirected
    assert seen_amb > 0 and seen_red > 0   # the redirect itself was exercised against the reference at full size
    c.close()


@pytest.mark.parametrize("nranks", [2, 4, 8])
def test_2048_slabs_against_live_reference(mcb, refbind, nranks):
    """BASELINE.json configs[4]: the 2049^3-cube sphere cut into the z-slabs of an nranks-GPU run (mcb_slab_range).  A whole
    slab is polygonised under mcb_set_slab; its first and its last cube layer — the ones next to the recomputed halo planes —
    are compared per active cube (position, code, table row, triangle offsets) and triangle by triangle with the unmodified
    reference run live on those layers."""
    from .helpers import same_bits
    eq = "x^2+y^2+z^2-0.49"
    step = 2.0 / 2048
    c = mcb.Context(0)
    c.set_field_mode(mcb.FIELD_AUTO)
    c.set_normals(0)
    assert c.set_equation(eq) == 0 and c.set_grid_step(step) == 2049
    M = 2049
    r = nranks // 2                       # a slab through the sphere with neighbours on both sides
    k0, k1 = mcb.slab_range(M, r, nranks)
    c.set_slab(k0, k1)
    cnt = c.polygonise()
    assert cnt.cubes == (k1 - k0) * M * M and cnt.triangles > 0
    rec, off = c.get_active()
    pos, _ = c.get_mesh(normals=False)
    layer = ((rec >> 24) & 0xFFF).astype(np.int64)
    compared = 0
    for k in (k0, k1 - 1):
        sw = refbind.sweep_rows_mt(eq, step, k * M, (k + 1) * M)
        act = np.flatnonzero((sw["code"] != 0) & (sw["code"] != 255))
        sel = np.flatnonzero(layer == k)
        assert len(sel) == len(act) == sw["active"]
        if len(sel) == 0:   # the last layer of the last slab lies outside the sphere: both sides agree that it is empty
            continue
        compared += 1
        lin = (rec[sel] & 0xFFF).astype(np.int64) + M * ((rec[sel] >> 12) & 0xFFF).astype(np.int64)
        assert np.array_equal(lin, act)
        assert np.array_equal(((rec[sel] >> 36) & 0xFF).astype(np.uint8), sw["code"][act])
        assert np.array_equal(((rec[sel] >> 44) & 0xFF).astype(np.uint8), sw["table_idx"][act])
        t0 = int(off[sel[0]])
        t1 = int(off[sel[-1] + 1]) if sel[-1] + 1 < len(off) else int(cnt.triangles)
        assert t1 - t0 == sw["T"]
        assert np.array_equal(off[sel].astype(np.int64) - t0, np.concatenate([[0], np.cumsum(sw["ntri"][act].astype(np.int64))[:-1]]))
        assert same_bits(pos[t0:t1, :, :3], sw["soup"])
    assert compared >= 1
    c.close()
