"""CPU tier of the refined vertices (mcb_set_refine_vertices, csrc/mcb_refine.h): the rule's properties on crossing edges of
named and random equations, accuracy against an independent float64 root, hard one-dimensional fields, and the emulated
device pipeline (tests/emu) against the host build."""
import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_EQUATIONS, random_csg_equations
from .functions_common import FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, TORUS_SDF, random_function_equations
from .helpers import load_meta, same_bits
from .normals_common import postfix_program
from .refine_common import (REFINE_EVALS, SAME_SIGN, counts_tuple, crossing_edges, host_f, host_refine, linear_points, root64,
                            run_refined, well_conditioned_root)

F = GRAMMAR_FUNCTIONS
SPHERE = "x^2+y^2+z^2-0.49"


def _golden_equations(golden):
    return sorted(set(c["eq"] for c in load_meta(golden).values()))


def _check_rule(mcb, eq, grammar, step, scale, rng, n=200):
    """The rule's properties on up to n crossing edges: returns (edges, evaluations)"""
    M, c = mcb.grid_axis(step)
    lo, ax, ilo, flo, fhi = crossing_edges(eq, c, n, rng, 0.0, scale, grammar)
    if len(lo) == 0:
        return 0, np.zeros(0, np.int32)
    fwd, bwd = linear_points(lo, ax, ilo, flo, fhi, c)
    r, ev, _ = host_refine(eq, c, fwd, 0.0, scale, grammar)
    assert not (ev == SAME_SIGN).any(), eq
    assert (ev <= REFINE_EVALS).all(), eq
    on_vertex = ev == 0  # the linear point fell on a grid vertex (t = 0 or 1): unchanged
    assert same_bits(r[on_vertex], fwd[on_vertex]), eq
    k = np.arange(len(r))
    other = np.ones((len(r), 3), bool)
    other[k, ax] = False
    assert same_bits(r[other], fwd[other]), eq  # the two fixed coordinates keep their bits
    assert ((r[k, ax] >= c[ilo]) & (r[k, ax] <= c[ilo + 1])).all(), eq
    d0 = np.abs(host_f(eq, fwd, scale, grammar).astype(np.float64))
    d1 = np.abs(host_f(eq, r, scale, grammar).astype(np.float64))
    fin = np.isfinite(d0)
    assert (d1[fin] <= d0[fin]).all(), eq
    # the edge function: a cube interpolating from the upper end gets the same refined bits
    rb, evb, _ = host_refine(eq, c, bwd, 0.0, scale, grammar)
    moved = (ev > 0) & (evb > 0)
    assert same_bits(rb[moved], r[moved]), eq
    return len(r), ev[ev > 0]


def test_rule_properties_on_named_and_random_equations(mcb, golden):
    """Golden, function and CSG equations and 200 random function / CSG equations, at several steps and scales: two
    coordinates bit-unchanged and the third in [c_i, c_i+1], never farther from the level than the linear point, vertices on
    grid vertices unchanged, the same bits from both directions of an edge, the same-sign branch never taken."""
    rng = np.random.default_rng(5)
    named = [(eq, 0) for eq in _golden_equations(golden)] + [(eq, F) for eq in FUNCTION_EQUATIONS + CSG_EQUATIONS]
    rand = [(eq, F) for eq in random_function_equations(mcb, 21, 100) + random_csg_equations(mcb, 22, 100)]
    steps = (0.2, 0.125, 2.0 / 64, 2.0 / 200)
    edges, evals = 0, []
    for i, (eq, grammar) in enumerate(named + rand):
        scale = (1.0, 1.0, 1.0) if i % 2 else (1.1, 0.9, 1.3)
        n, ev = _check_rule(mcb, eq, grammar, steps[i % len(steps)], scale, rng, 200 if i < len(named) else 60)
        edges += n
        evals.append(ev)
    ev = np.concatenate(evals)
    print("rule properties: %d crossing edges of %d equations; evaluations per refined vertex mean %.2f, max %d (cap %d)"
          % (edges, len(named) + len(rand), ev.mean(), ev.max(), REFINE_EVALS))
    assert edges > 2000


def test_points_off_the_edges_are_unchanged(mcb):
    M, c = mcb.grid_axis(0.2)
    pts = np.array([[c[1], c[2], c[3]],                      # a grid vertex
                    [0.05, 0.05, c[4]],                      # two coordinates off the grid
                    [c[1], c[2], 1.5], [c[1], c[2], -1.5],   # outside the table
                    [c[1], c[2], np.nan]], np.float32)
    r, ev, _ = host_refine(SPHERE, c, pts, grammar=0)
    assert (ev == 0).all() and same_bits(r, pts)


def test_sphere_radius_against_linear_points(mcb):
    """x^2+y^2+z^2-0.49 at the reference GUI's step 0.2: every refined vertex's radius is within 1e-6 of 0.7; the linear
    points' error is printed beside it."""
    M, c = mcb.grid_axis(0.2)
    lo, ax, ilo, flo, fhi = crossing_edges(SPHERE, c, 100000, np.random.default_rng(1), grammar=0)
    fwd, _ = linear_points(lo, ax, ilo, flo, fhi, c)
    r, ev, _ = host_refine(SPHERE, c, fwd, grammar=0)
    rr = np.abs(np.linalg.norm(r.astype(np.float64), axis=1) - 0.7)
    rl = np.abs(np.linalg.norm(fwd.astype(np.float64), axis=1) - 0.7)
    print("sphere at step 0.2, %d crossing edges: radius error refined max %.2e mean %.2e; linear max %.2e mean %.2e"
          % (len(r), rr.max(), rr.mean(), rl.max(), rl.mean()))
    assert len(r) > 100 and rr.max() <= 1e-6 and rl.max() > 1e-3


def test_accuracy_against_the_float64_root(mcb):
    """On crossing edges of the torus SDF, the mixed function, the gyroid and the box SDF at step 0.2 and 2/64: the refined
    coordinate is within 2^-22 + 4 * bound of the float64 root, where the edge is kept when its root is well-conditioned
    (refine_common.well_conditioned_root: fp32 evaluation noise over |df/daxis| at most 1e-6)."""
    rng = np.random.default_rng(3)
    kept = total = 0
    worst_r = worst_l = 0.0
    for eq in (TORUS_SDF, FUNCTION_EQUATIONS[5], FUNCTION_EQUATIONS[0], CSG_BOX_SDF):
        prog = postfix_program(mcb, eq, F)
        for step in (0.2, 2.0 / 64):
            M, c = mcb.grid_axis(step)
            lo, ax, ilo, flo, fhi = crossing_edges(eq, c, 40, rng)
            fwd, _ = linear_points(lo, ax, ilo, flo, fhi, c)
            r, ev, _ = host_refine(eq, c, fwd)
            for i in range(len(r)):
                total += 1
                if ev[i] <= 0:
                    continue
                root = root64(prog, r[i], ax[i], c[ilo[i]], c[ilo[i] + 1])
                if root is None:
                    continue
                ok, bound = well_conditioned_root(prog, root, r[i], ax[i])
                if not ok:
                    continue
                kept += 1
                err = abs(float(r[i, ax[i]]) - root)
                worst_r = max(worst_r, err)
                worst_l = max(worst_l, abs(float(fwd[i, ax[i]]) - root))
                assert err <= 2.0 ** -22 + 4 * bound, (eq, step, i, err, bound)
    print("float64 root: %d of %d edges kept as well-conditioned; largest error refined %.2e, linear %.2e" % (kept, total, worst_r, worst_l))
    assert kept > total // 2


# ---- hard one-dimensional fields -----------------------------------------------------------------------------------------
def _one(eq, a, b, x, iso=0.0):
    """refine the point (x, 0, 0) on the coordinate table [0, a, b]: its edge is (a, b) along x, y = z = 0 grid coordinates"""
    c = np.array([0.0, a, b], np.float32)
    r, ev, br = host_refine(eq, c, np.array([[x, 0.0, 0.0]], np.float32), iso)
    return r[0, 0], int(ev[0]), br[0]


def test_triple_root():
    x, ev, _ = _one("(x-0.31)^3", 0.25, 0.375, 0.3)
    assert 2 < ev <= REFINE_EVALS and abs(x - 0.31) < 1e-5, (x, ev)


def test_field_equal_to_the_level_on_an_interval():
    # the lower end lies on the plateau f == iso: the search stops there, f == iso exactly
    x, ev, _ = _one("max(x-0.3,0)", 0.25, 0.375, 0.3)
    assert ev == 2 and x == np.float32(0.25) and host_f("max(x-0.3,0)", [[x, 0, 0]])[0] == 0
    # the plateau strictly inside the edge: the linear point lands on it
    eq = "max(x-0.3,0)-max(0.28-x,0)"
    x, ev, _ = _one(eq, 0.25, 0.375, 0.3)
    assert ev == 3 and 0.28 <= x <= 0.3 and host_f(eq, [[x, 0, 0]])[0] == 0


def test_infinite_slope():
    eq = "sqrt(max(x-0.31,0))-sqrt(max(0.31-x,0))"
    x, ev, br = _one(eq, 0.25, 0.375, 0.3)
    assert ev <= REFINE_EVALS and abs(x - 0.31) < 1e-6 and br[1] - br[0] <= 2.0 ** -24 * 2, (x, ev, br)


def test_nan_inside_the_edge():
    """f is NaN on (0.30, 0.32) (the square root of a negative number) and changes sign inside that interval.  s(NaN) is
    false, so the classifier's sign change, and the search's, is at 0.32; the result is the finite point nearest the level."""
    eq = "x-0.31+0*sqrt(abs(x-0.31)-0.01)"
    x, ev, br = _one(eq, 0.25, 0.375, 0.3)
    fx = host_f(eq, [[x, 0, 0]])[0]
    assert 2 < ev <= REFINE_EVALS and np.isfinite(fx) and abs(fx) < 0.0101, (x, ev, fx)
    assert abs(float(br[0]) - 0.32) < 1e-6 and br[1] - br[0] <= 2.0 ** -23, br


def test_pole_converges_to_the_sign_change():
    """1/(x-0.31): the sign changes at the pole.  The bracket closes on the pole; the returned point is the evaluated point
    with the smallest |f|, far from the pole (documented in DESIGN.md §13)."""
    x, ev, br = _one("1/(x-0.31)", 0.25, 0.375, 0.3)
    assert ev <= REFINE_EVALS and br[0] < 0.31 < br[1] + 1e-7 and br[1] - br[0] <= 2.0 ** -23, (x, ev, br)
    assert abs(x - 0.31) > 0.01


# ---- emulated device pipeline --------------------------------------------------------------------------------------------
EMULATED = {"sphere": (SPHERE, 0), "torus_sdf": (TORUS_SDF, F), "union": (CSG_EQUATIONS[0], F), "box": (CSG_BOX_SDF, F),
            "mixed": (FUNCTION_EQUATIONS[5], F)}


@pytest.mark.parametrize("name", sorted(EMULATED))
@pytest.mark.parametrize("mode", ["dense", "blocks"])
def test_emulated_pipeline_refined(mcb_emu, name, mode):
    """The device code executed on the host at step 2/32 (33^3 cubes): refined soup and welded positions equal the host
    refinement of the unrefined run's positions bit for bit; tri_list and counts are those of the unrefined run."""
    eq, grammar = EMULATED[name]
    scale = (1.1, 1.1, 1.1)
    fm = mcb_emu.FIELD_DENSE if mode == "dense" else mcb_emu.FIELD_AUTO
    m1 = run_refined(mcb_emu, eq, 2.0 / 32, scale, True, field_mode=fm, grammar=grammar)
    m0 = run_refined(mcb_emu, eq, 2.0 / 32, scale, False, field_mode=fm, grammar=grammar)
    assert m1["counts"].triangles > 200
    assert counts_tuple(m1["counts"]) == counts_tuple(m0["counts"]) and np.array_equal(m1["tl"], m0["tl"])
    M, c = mcb_emu.grid_axis(2.0 / 32)
    p0 = m0["pos"][:, :, :3].reshape(-1, 3)
    want, ev, _ = host_refine(eq, c, p0, 0.0, scale, grammar)
    assert same_bits(m1["pos"][:, :, :3].reshape(-1, 3), want) and (m1["pos"][:, :, 3] == 1).all()
    assert not (ev == SAME_SIGN).any() and (ev > 0).sum() > len(ev) // 2
    wv, evv, _ = host_refine(eq, c, m0["vl"], 0.0, scale, grammar)
    assert same_bits(m1["vl"], wv) and not (evv == SAME_SIGN).any()


def test_emulated_repeat_mode_and_host_output(mcb_emu):
    ctx = mcb_emu.Context(0)
    try:
        ctx.set_mesh_mode(mcb_emu.MESH_INDEXED)
        assert ctx.set_equation(SPHERE) == 0
        ctx.set_grid_step(2.0 / 32)
        ctx.set_refine_vertices(True)
        assert ctx.set_repeat(True, 0.3) == 0
        with pytest.raises(mcb_emu.McbError) as e:
            ctx.polygonise()
        assert e.value.status == mcb_emu.MCB_E_STATE
        assert ctx.set_repeat(False) == 0
        ctx.polygonise()
        V, T = int(ctx.counts.vertices), int(ctx.counts.triangles)
        vl, tl = np.zeros((V + 16, 3), np.float32), np.zeros((T + 16, 3), np.uint32)
        ctx.set_host_output(vl.ctypes.data, tl.ctypes.data, 0, V + 16, T + 16)
        ctx.set_normals(0)
        ctx.polygonise()
        assert not ctx.host_output_filled() and not vl.any()
        want = ctx.get_indexed_mesh()
        ctx.set_refine_vertices(False)
        ctx.polygonise()
        assert ctx.host_output_filled() and not same_bits(vl[:V], want[0])
    finally:
        ctx.close()


def test_emulated_marching_mirror(mcb_emu):
    """Marching.set_refined_vertices of the Python mirror delivers the refined Poly_Data of the Context path."""
    m = mcb_emu.Marching()
    m.set_evaluator(mcb_emu.Evaluator(SPHERE))
    assert m.set_grid_resolution(32)
    m.set_refined_vertices(True)
    assert m.recalculate()
    want = run_refined(mcb_emu, SPHERE, 2.0 / 32, grammar=0)
    assert same_bits(m.get_poly_data().vertex_list.reshape(-1, 3), want["vl"])
    assert np.array_equal(m.get_poly_data().tri_list.reshape(-1, 3), want["tl"])
