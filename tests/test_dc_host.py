"""CPU tier of dual contouring (MCB_MESH_DC, csrc/mcb_qef.h, DESIGN.md §14): the QEF against float64, the quads against an
independent integer statement, sharp corners and seams, closed shapes, orientation, the documented errors, and the
emulated device pipeline (tests/emu) against the host build."""
import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_EQUATIONS, CSG_UNION2
from .dc_common import (BOX, MESH_DC, QEF_CUT, QEF_SWEEPS, SPHERE, euler, grid_axis, host_dc, nonmanifold_edges, python_quads, qef,
                        run_dc, signed_volume)
from .functions_common import GYROID, TORUS_SDF
from .helpers import same_bits
from .refine_common import host_refine

TORUS_GOLDEN = "(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)"
CASES = [(SPHERE, 2 / 24), (TORUS_GOLDEN, 2 / 24), (TORUS_SDF, 2 / 24), (GYROID, 2 / 24), (BOX, 2 / 22)] + [(e, 2 / 24) for e in CSG_EQUATIONS]


def _box_step():
    """a step whose grid planes all lie at least step/4 from the box's face planes"""
    for n in range(40, 90):
        step = 2.0 / n
        c = grid_axis(step).astype(np.float64)
        if all(np.abs(c - f).min() >= step / 4 for f in (0.5, -0.5, 0.4, -0.4, 0.3, -0.3)):
            return step
    raise AssertionError("no step")


def _qef64(p, n, lo, hi):
    """the same rule in float64 with numpy.linalg.eigh: (x, rank, eigenvalues)"""
    p, n = p.astype(np.float64), n.astype(np.float64)
    c = p.mean(axis=0)
    keep = np.abs(n).sum(axis=1) > 0
    A = n[keep].T @ n[keep]
    r = (n[keep] * ((p[keep] - c) * n[keep]).sum(axis=1)[:, None]).sum(axis=0)
    lam, V = np.linalg.eigh(A)
    x = c.copy()
    rank = 0
    if lam.max() > 0:
        for i in range(3):
            if lam[i] >= QEF_CUT * lam.max():
                x += (V[:, i] @ r) / lam[i] * V[:, i]
                rank += 1
    return np.clip(x, lo, hi), rank, lam


def _cells(d):
    c = d["c"]
    M = d["M"]
    s = d["field"] > np.float32(d["iso"])
    idx = np.flatnonzero((np.logical_or.reduce([s[a:a + M, b:b + M, e:e + M] for a in (0, 1) for b in (0, 1) for e in (0, 1)]) &
                          ~np.logical_and.reduce([s[a:a + M, b:b + M, e:e + M] for a in (0, 1) for b in (0, 1) for e in (0, 1)])).ravel())
    k, j, i = idx // (M * M), (idx // M) % M, idx % M
    lo = np.stack([c[i], c[j], c[k]], 1)
    hi = np.stack([c[i + 1], c[j + 1], c[k + 1]], 1)
    return lo, hi


@pytest.mark.parametrize("eq,step", CASES)
def test_qef_against_float64_and_vertices_in_their_cubes(eq, step):
    d = host_dc(eq, step)
    lo, hi = _cells(d)
    vl = d["vl"]
    assert len(vl) == len(lo) > 0
    assert ((vl >= lo) & (vl <= hi)).all(), eq  # a DC vertex never leaves its cube
    compared = 0
    for q in range(len(vl)):
        m = d["cell_m"][q]
        x64, rank64, lam = _qef64(d["cell_p"][q, :m], d["cell_n"][q, :m], lo[q].astype(np.float64), hi[q].astype(np.float64))
        cut = QEF_CUT * lam.max()
        if lam.max() > 0 and np.any((lam > cut / 2) & (lam < 2 * cut)):
            continue  # an eigenvalue near the cut: fp32 and fp64 may keep different ranks there
        assert d["rank"][q] == rank64, (eq, q)
        assert np.abs(vl[q] - x64).max() <= 1e-5, (eq, q, vl[q], x64)
        compared += 1
    assert compared >= len(vl) // 10, (eq, compared, len(vl))  # curved cells often have an eigenvalue near the cut


def test_qef_rank_on_random_planes():
    """one, two and three random planes through random points of a unit cell: rank 1, 2, 3 and the float64 solution"""
    rng = np.random.default_rng(7)
    for _ in range(300):
        nplanes = int(rng.integers(1, 4))
        while True:
            N = rng.normal(size=(nplanes, 3))
            N /= np.linalg.norm(N, axis=1, keepdims=True)
            if nplanes == 1 or np.linalg.svd(N, compute_uv=False).min() > 0.3:
                break
        target = rng.uniform(0.2, 0.8, 3)
        pts, nrm = [], []
        for pl in range(nplanes):
            for _ in range(int(rng.integers(2, 5))):
                # a point on the plane through `target`
                t = rng.normal(size=3)
                t -= (t @ N[pl]) * N[pl]
                pts.append(target + 0.2 * t)
                nrm.append(N[pl])
        pts, nrm = np.float32(pts), np.float32(nrm)
        lo, hi = np.zeros(3, np.float32) - 1, np.ones(3, np.float32) + 1
        x, rk, mat, _ = qef(pts, nrm, lo, hi)
        x64, r64, _ = _qef64(pts, nrm, lo.astype(np.float64), hi.astype(np.float64))
        assert rk == nplanes == r64
        assert np.abs(x - x64).max() <= 1e-5
        if nplanes == 3:
            assert np.abs(x - target).max() <= 1e-5


@pytest.mark.parametrize("eq,step", CASES)
def test_jacobi_has_converged_after_the_pinned_sweeps(eq, step):
    """on every cell: after MCB_QEF_SWEEPS the off-diagonal entries are below 1e-6 of the largest eigenvalue"""
    d = host_dc(eq, step)
    lo, hi = _cells(d)
    worst = 0.0
    for q in range(len(d["vl"])):
        m = d["cell_m"][q]
        _, _, mat, _ = qef(d["cell_p"][q, :m], d["cell_n"][q, :m], lo[q], hi[q])
        lmax = np.abs(np.diag(mat)).max()
        if lmax == 0:
            continue
        off = np.abs(mat - np.diag(np.diag(mat))).max()
        worst = max(worst, off / lmax)
    assert worst <= 1e-6, (eq, worst)
    assert QEF_SWEEPS == 6


@pytest.mark.parametrize("eq,step,cons", [(SPHERE, 2 / 20, ()), (TORUS_SDF, 2 / 24, ()), (GYROID, 2 / 16, ()), (CSG_UNION2, 2 / 24, ()),
                                          (SPHERE, 2 / 20, (("x+0.3y", "<", 0.25),)), (GYROID, 2 / 16, (("z", ">=", -0.3), ("x^2", "<", 0.5)))])
def test_quads_equal_an_independent_integer_statement(eq, step, cons):
    d = host_dc(eq, step, cons=cons)
    assert len(d["tl"]) > 0
    assert np.array_equal(python_quads(d), d["tl"]), eq


def test_box_corners_are_sharp():
    step = _box_step()
    d = host_dc(BOX, step)
    vl = d["vl"].astype(np.float64)
    corners = np.array([(sx * 0.5, sy * 0.4, sz * 0.3) for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)])
    for cpt in corners:
        assert np.abs(vl - cpt).max(axis=1).min() <= 1e-5, cpt
    f = np.maximum(np.maximum(np.abs(vl[:, 0]) - 0.5, np.abs(vl[:, 1]) - 0.4), np.abs(vl[:, 2]) - 0.3)
    assert np.abs(f).max() <= 1e-5  # |f| is the L-infinity distance to the box here
    # the refined marching-cubes mesh cuts every corner off
    from .csg_common import CsgOracle
    o = CsgOracle(BOX, step)
    mv, _ = o.recalculate()
    r, _, _ = host_refine(BOX, d["c"], mv)
    for cpt in corners:
        assert np.linalg.norm(r.astype(np.float64) - cpt, axis=1).min() > step / 4, cpt


def _seg_dist(p, a, b):
    ab = b - a
    t = np.clip(((p - a) @ ab) / (ab @ ab), 0, 1)
    return np.linalg.norm(p - (a + t[:, None] * ab), axis=1)


def test_straight_seams_of_a_box_union_are_exact():
    """a cross of two boxes: the concave seams where B's faces meet A's faces y = +-0.3 are straight, so every vertex of a
    cube one of them crosses lies on it"""
    eq = "min(max(max(abs(x)-0.5,abs(y)-0.3),abs(z)-0.3),max(max(abs(x)-0.2,abs(y)-0.5),abs(z)-0.2))"
    step = None
    for n in range(40, 90):
        c = grid_axis(2.0 / n).astype(np.float64)
        if all(np.abs(c - f).min() >= 0.4 / n for f in (0.5, 0.3, 0.2, -0.5, -0.3, -0.2)):
            step = 2.0 / n
            break
    d = host_dc(eq, step)
    lo, hi = _cells(d)
    segs = []
    for y in (0.3, -0.3):
        for s in (0.2, -0.2):
            segs.append((np.array([s, y, -0.2]), np.array([s, y, 0.2])))  # along z, on B's faces x = +-0.2
            segs.append((np.array([-0.2, y, s]), np.array([0.2, y, s])))  # along x, on B's faces z = +-0.2
    n_checked = 0
    for a, b in segs:
        ts = np.linspace(0, 1, 2001)[:, None]
        pts = a + ts * (b - a)
        crossed = np.zeros(len(lo), bool)
        for p in pts:
            crossed |= np.all((lo <= p) & (p <= hi), axis=1)
        dist = _seg_dist(d["vl"][crossed].astype(np.float64), a, b)
        assert len(dist) > 0 and dist.max() <= 1e-5, (a, b, dist.max())
        n_checked += len(dist)
    assert n_checked > 40


def _sphere_union_seam(d, vl_mc):
    """(largest distance of a seam cube's DC vertex from the seam circle, the same for the refined MC mesh's vertices
    nearest the circle in each seam cube)"""
    x0 = (0.25 - 0.1225 + 0.45 ** 2) / 0.9
    r0 = np.sqrt(0.25 - x0 ** 2)
    th = np.linspace(0, 2 * np.pi, 20000, endpoint=False)
    circle = np.stack([np.full_like(th, x0), r0 * np.cos(th), r0 * np.sin(th)], 1)
    c = d["c"].astype(np.float64)
    lo, hi = _cells(d)
    key = {tuple(v): q for q, v in enumerate(np.round(lo.astype(np.float64), 7))}
    ijk = np.searchsorted(c, circle, side="right") - 1
    cubes = set(key.get(tuple(np.round(c[list(idx)], 7))) for idx in map(tuple, ijk))
    cubes.discard(None)

    def dist(p):
        p = np.asarray(p, np.float64).reshape(-1, 3)
        return np.hypot(p[:, 0] - x0, np.hypot(p[:, 1], p[:, 2]) - r0)
    dc = max(dist(d["vl"][q])[0] for q in cubes)
    mc = 0.0
    v = vl_mc.astype(np.float64)
    for q in cubes:
        inside = np.all((v >= lo[q] - 1e-7) & (v <= hi[q] + 1e-7), axis=1)
        if inside.any():
            mc = max(mc, dist(v[inside]).min())
    return dc, mc


def test_curved_seam_of_a_sphere_union_converges():
    from .csg_common import CsgOracle
    res = []
    for n in (64, 128):
        d = host_dc(CSG_UNION2, 2.0 / n)
        mv, _ = CsgOracle(CSG_UNION2, 2.0 / n).recalculate()
        r, _, _ = host_refine(CSG_UNION2, d["c"], mv)
        res.append(_sphere_union_seam(d, r))
    for dc, mc in res:
        assert dc < mc, res
    assert res[0][0] >= 3 * res[1][0], res  # second order


@pytest.mark.parametrize("eq,chi", [(SPHERE, 2), (BOX, 2), (CSG_BOX_SDF, 2), (TORUS_SDF, 0)])
def test_closed_shapes_are_closed_manifolds(eq, chi):
    d = host_dc(eq, 2 / 64)
    assert nonmanifold_edges(d["tl"]) == 0, eq
    assert euler(d["tl"]) == chi, eq


@pytest.mark.parametrize("eq", [SPHERE, TORUS_SDF, CSG_BOX_SDF, CSG_UNION2])
def test_orientation_and_volume_match_marching_cubes(eq):
    from .csg_common import CsgOracle
    d = host_dc(eq, 2 / 64)
    mv, mt = CsgOracle(eq, 2 / 64).recalculate()
    v_dc, v_mc = signed_volume(d["vl"], d["tl"]), signed_volume(mv, mt)
    assert v_dc * v_mc > 0 and abs(v_dc - v_mc) <= 0.02 * abs(v_mc), (eq, v_dc, v_mc)


def test_documented_errors(mcb_emu):
    m = mcb_emu
    ctx = m.Context(0)
    try:
        for mode in (MESH_DC | m.MESH_SOUP, MESH_DC | m.MESH_INDEXED, MESH_DC | 3, 8):
            with pytest.raises(m.McbError) as e:
                ctx.set_mesh_mode(mode)
            assert e.value.status == m.MCB_E_ARG
        ctx.set_mesh_mode(MESH_DC)
        ctx.set_equation(SPHERE)
        ctx.set_grid_step(2 / 16)

        def state(msg):
            with pytest.raises(m.McbError) as e:
                ctx.polygonise()
            assert e.value.status == m.MCB_E_STATE and msg in str(e.value)
        ctx.set_normals(1)
        state("normals mode 1")
        ctx.set_normals(0)
        assert ctx.set_seed(True, 0.7, 0, 0) == 0
        state("seed mode")
        ctx.set_seed(False)
        ctx.set_repeat(True, 0.1)
        state("repeating-surface mode")
        ctx.set_repeat(False, 0.1)
        ctx.set_slab(0, 8)
        state("full grid")
        ctx.set_grid_step(2 / 16)
        cnt = ctx.polygonise()
        assert cnt.mesh_mode == MESH_DC and cnt.vertices == cnt.active > 0
        with pytest.raises(m.McbError):
            ctx.get_mesh()
        assert not m.lib.mcb_host_output_filled(ctx.h)
    finally:
        ctx.close()


@pytest.mark.parametrize("eq,step,cons", [(SPHERE, 2 / 32, ()), (TORUS_SDF, 2 / 32, ()), (BOX, 2 / 32, ()), (GYROID, 2 / 32, ()),
                                          (CSG_UNION2, 2 / 32, (("x", "<", 0.3),))])
@pytest.mark.parametrize("mode", ["dense", "blocks"])
def test_emulated_pipeline_equals_the_host_build(mcb_emu, eq, step, cons, mode):
    d = host_dc(eq, step, cons=cons)
    r = run_dc(mcb_emu, eq, step, cons=cons, field_mode=mcb_emu.FIELD_DENSE if mode == "dense" else mcb_emu.FIELD_SPARSE)
    assert r["counts"].vertices == r["counts"].active == len(d["vl"])
    assert same_bits(r["vl"], d["vl"]) and np.array_equal(r["tl"], d["tl"])
