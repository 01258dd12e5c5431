"""-m gpu: the CUDA path, called through the C ABI, against the golden vectors produced by the unmodified reference
(tests/golden/cases.npz, made by tests/golden/make_golden.py) and against the reference executed live (its
restatement where oracle/_ref is not built: see the `refbind` fixture).

Bars (north_star): cube_code, table_idx and per-cube triangle counts BIT-EXACT; positions within 1e-5 relative
(they are in fact required bit-exact here, the tolerance test is the weaker fallback assertion); normals within
1e-5 of the CPU restatement of the central-difference definition.
"""
import numpy as np
import pytest

from .helpers import configure, load_meta, rel_close, same_bits
from . import mc_numpy

pytestmark = pytest.mark.gpu


def _cases(golden):
    return load_meta(golden)


def tri_rows():
    import importlib
    # decode the product's packed table on the host side (pure bit twiddling, no compute path involved)
    import re, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    txt = open(os.path.join(root, "marching-cube-for-implicit-surfaces_b200", "csrc", "mcb_tri_words.inc")).read()
    words = [int(w, 16) for w in re.findall(r"0x([0-9a-f]{16})ull", txt)]
    rows = []
    for w in words:
        r = []
        for f in range(16):
            v = (w >> (4 * f)) & 0xF
            if v == 0xF:
                break
            r.append(v)
        rows.append(r)
    return rows


CASE_NAMES = ["eq%d_%s" % (n, k) for n in range(1, 9) for k in ("gui", "ctor")] + [
    "sphere_17", "sphere_33_iso", "torus_33", "saddle_17", "gyr34_9", "gyr78_17", "quirk_div", "quirk_neg",
    "nonuniform_scale", "constraint_x", "constraint_2"]


@pytest.fixture(scope="module")
def ctx(mcb):
    c = mcb.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("name", CASE_NAMES)
def test_case_against_golden(mcb, ctx, golden, name):
    case = _cases(golden)[name]
    configure(ctx, case)
    ctx.set_normals(1)
    cnt = ctx.polygonise()
    M = case["M"]
    assert cnt.M == M and cnt.cubes == M ** 3
    # --- field values at the grid vertices: bit-exact (powf restated exactly, no FMA contraction)
    F = ctx.get_field()
    Fg = golden[name + "/field_ext"][1:-1, 1:-1, 1:-1]
    assert same_bits(F, Fg), "field differs from the reference evaluator"
    # --- cases: bit-exact
    code, tidx = ctx.get_cases()
    assert np.array_equal(code, golden[name + "/code"]), "cube_code"
    assert np.array_equal(tidx, golden[name + "/table_idx"]), "table_idx"
    assert cnt.triangles == case["T"] and cnt.active == case["active"]
    assert cnt.ambiguous == case["ambiguous"] and cnt.redirected == case["redirected"]
    # --- compacted records are in loop order and carry the per-cube triangle counts
    rec, off = ctx.get_active()
    lin = (rec & 0xFFF).astype(np.int64) + M * (((rec >> 12) & 0xFFF).astype(np.int64) + M * ((rec >> 24) & 0xFFF).astype(np.int64))
    assert np.all(np.diff(lin) > 0)
    ntri_g = golden[name + "/ntri"].astype(np.int64)
    act = np.flatnonzero((golden[name + "/code"] != 0) & (golden[name + "/code"] != 255))
    assert np.array_equal(lin, act)
    assert np.array_equal(off.astype(np.int64), np.concatenate([[0], np.cumsum(ntri_g[act])[:-1]]) if len(act) else off)
    # --- triangle soup: same order, same positions
    pos, nrm = ctx.get_mesh(normals=True)
    soup = golden[name + "/soup"]
    assert pos.shape[0] == soup.shape[0]
    if len(soup):
        assert rel_close(pos[:, :, :3], soup, 1e-5)
        assert same_bits(pos[:, :, :3], soup), "positions are within tolerance but not bit-exact"
        assert np.all(pos[:, :, 3] == 1.0)
        # --- welded expansion of the reference's Poly_Data is the same soup up to its 1e-6 weld
        v, t = golden[name + "/vertex_list"], golden[name + "/tri_list"]
        assert rel_close(pos[:, :, :3], v[t.astype(np.int64)], 1e-5)
        # --- normals: CPU restatement of the central-difference definition on the reference's field values
        cubes = [(int(r & 0xFFF), int((r >> 12) & 0xFFF), int((r >> 24) & 0xFFF), int((r >> 36) & 0xFF), int((r >> 44) & 0xFF)) for r in rec]
        cs = mc_numpy.apron_coords(golden[name + "/coords"], case["step"])
        nref = mc_numpy.soup_gradient_normals(golden[name + "/field_ext"], cs, case["iso"], cubes, tri_rows())
        ok = np.isfinite(nref).all(axis=2)
        assert rel_close(nrm[:, :, :3][ok], nref[ok], 1e-5)
        # where the restatement's normal is not finite (zero or overflowing gradient) the device's is not a number either
        assert not np.isfinite(nrm[:, :, :3][~ok]).all(axis=-1).any() if (~ok).any() else True


def test_eval_points_against_reference(mcb, ctx, refbind):
    rng = np.random.default_rng(7)
    pts = (rng.random((50000, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    pts[:64] = 0
    eqs = list(refbind.EXAMPLE_EQUATIONS.values()) + [refbind.SPHERE, refbind.TORUS, refbind.GYR34, refbind.GYR78,
                                                       "x-y+z", "x/y*z", "-x^2", "x*-y+z", "x^y^z", "x^0.5+y", "2^x+y^z", "xy/z^-.22"]
    for eq in eqs:
        assert ctx.set_equation(eq) == 0
        out = ctx.eval_points(pts)
        ref = refbind.Ref(eq).eval_points(pts)
        assert same_bits(out, ref), eq


def test_powf_device_matches_libm(mcb, ctx, refbind):
    """`^` on the device against glibc powf through the reference evaluator: random bases/exponents incl. edge cases."""
    rng = np.random.default_rng(11)
    n = 200000
    x = rng.random(n, dtype=np.float32) * 6 - 3
    y = rng.random(n, dtype=np.float32) * 16 - 8
    x[:8] = [0, -0.0, 1, -1, np.inf, -np.inf, np.nan, 1e-40]
    y[:8] = [0.5, 3, np.inf, 2, -1, 3, 0, 2]
    y[8:1000] = np.round(y[8:1000])
    pts = np.stack([x, y, np.zeros(n, np.float32)], 1).astype(np.float32)
    assert ctx.set_equation("x^y") == 0
    assert same_bits(ctx.eval_points(pts), refbind.Ref("x^y").eval_points(pts))


def test_slabs_concatenate_to_full_grid(mcb, golden):
    """z-slab decomposition (SURVEY.md §8e): concatenating the slabs' soups in rank order is the single-GPU result."""
    meta = load_meta(golden)
    for name in ("gyr78_17", "eq8_ctor", "sphere_33_iso"):
        case = meta[name]
        full = mcb.Context(0)
        configure(full, case)
        full.polygonise()
        pos_full, nrm_full = full.get_mesh()
        code_full, tidx_full = full.get_cases()
        for nranks in (2, 3, 4):
            parts_p, parts_n, parts_c, T = [], [], [], 0
            for r in range(nranks):
                k0, k1 = mcb.slab_range(case["M"], r, nranks)
                c = mcb.Context(0)
                configure(c, case)
                c.set_slab(k0, k1)
                cnt = c.polygonise()
                p, n_ = c.get_mesh()
                parts_p.append(p); parts_n.append(n_); parts_c.append(c.get_cases()[0]); T += cnt.triangles
                c.close()
            assert T == case["T"]
            assert same_bits(np.concatenate(parts_p), pos_full)
            assert same_bits(np.concatenate(parts_n), nrm_full)
            assert np.array_equal(np.concatenate(parts_c), code_full)
        full.close()


def test_error_paths(mcb, ctx):
    assert ctx.set_equation("(x(y)") == mcb.MCB_E_PARSE
    assert ctx.set_equation("x+") == mcb.MCB_E_PARSE
    assert ctx.set_equation("x+y") == 0
    assert ctx.set_grid_step(0.0) == mcb.MCB_E_ARG
    assert ctx.set_grid_step(-1.0) == mcb.MCB_E_ARG
    assert ctx.set_grid_step(0.25) == 9
    with pytest.raises(mcb.McbError):
        ctx.get_mesh()  # nothing polygonised since the last change


def test_buffer_growth_rerun(mcb, golden):
    """A dense field overflows the initial record/soup guesses: the call must grow and repeat, not truncate."""
    c = mcb.Context(0)
    assert c.set_equation("x*y*z") == 0   # crossings everywhere
    assert c.set_grid_step(2.0 / 48) > 0
    cnt = c.polygonise()
    rec, off = c.get_active()
    pos, _ = c.get_mesh()
    assert len(rec) == cnt.active and pos.shape[0] == cnt.triangles
    cnt2 = c.polygonise()
    assert cnt2.reruns == 0 and cnt2.triangles == cnt.triangles
    c.close()
