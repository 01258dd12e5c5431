"""CPU tier of the analytic normals (mcb_set_normals 3, mcb_eval_gradients): the host build of mcb_interp_grad_scalar
against an independent float64 forward-mode evaluator, its value part against mcb_interp_scalar, exact cases bit for bit,
the kink conventions, and the emulated device pipeline (tests/emu) against the host build."""
import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_EQUATIONS, random_csg_equations
from .functions_common import FUNCTION_EQUATIONS, GRAMMAR_FUNCTIONS, random_function_equations
from .helpers import load_meta, same_bits
from .normals_common import (NORMALS_ANALYTIC, SPECIAL, counts_tuple, host_eval, host_normalise, normalise32, postfix_program,
                             run_mesh, soup_matches_welded, well_conditioned)

F = GRAMMAR_FUNCTIONS


def _golden_equations(golden):
    return sorted(set(c["eq"] for c in load_meta(golden).values()))


def _agree(mcb, eq, pts, scale, grammar=F):
    """max |fp32 normal - float64 normal| over the well-conditioned points, and how many points were excluded"""
    _, _, _, n = host_eval(eq, pts, scale, grammar)
    ok, u = well_conditioned(postfix_program(mcb, eq, grammar), pts, scale)
    err = float(np.abs(n.astype(np.float64) - u)[ok].max()) if ok.any() else 0.0
    return err, int((~ok).sum())


def test_host_gradient_agrees_with_the_float64_evaluator(mcb, golden):
    """Golden, function and CSG equations plus 200 random function / CSG equations at random points: every normalised
    component within 1e-5 of the float64 forward-mode evaluator, on the points the conditioning rule keeps
    (normals_common.well_conditioned)."""
    rng = np.random.default_rng(7)
    named = [(eq, 0) for eq in _golden_equations(golden)] + [(eq, F) for eq in FUNCTION_EQUATIONS + CSG_EQUATIONS]
    rand = [(eq, F) for eq in random_function_equations(mcb, 11, 100) + random_csg_equations(mcb, 12, 100)]
    total = excluded = 0
    worst = (0.0, None)
    for i, (eq, grammar) in enumerate(named + rand):
        pts = rng.uniform(-1.2, 1.2, (400 if i < len(named) else 100, 3)).astype(np.float32)
        scale = (1.0, 1.0, 1.0) if i % 2 else (1.1, 0.9, 1.3)
        err, ex = _agree(mcb, eq, pts, scale, grammar)
        total += len(pts)
        excluded += ex
        worst = max(worst, (err, eq), key=lambda t: t[0])
        assert err <= 1e-5, (eq, err)
    print("gradient vs float64: %d points, %d excluded as ill-conditioned, worst %.2e on %r" % (total, excluded, worst[0], worst[1]))
    assert excluded < total // 2


def test_value_part_is_bit_identical_to_the_interpreter(mcb):
    """On every triple from the special values (+-0, subnormals, +-inf, NaN, huge) and random points, including negative
    bases of ^: the value mcb_interp_grad_scalar returns has the bits of mcb_interp_scalar."""
    a, b, c = np.meshgrid(SPECIAL, SPECIAL, SPECIAL[::3], indexing="ij")
    pts = np.stack([a.ravel(), b.ravel(), c.ravel()], axis=1)
    pts = np.concatenate([pts, np.random.default_rng(3).uniform(-2, 2, (2000, 3)).astype(np.float32)])
    eqs = FUNCTION_EQUATIONS + CSG_EQUATIONS + ["x^y+z", "x^2.5-y^3+z^0.5", "(x-1)^y", "x/y-z", "min(x,y)*max(z,x)",
                                                "abs(x)-sqrt(y)+1/z"] + random_csg_equations(mcb, 5, 30)
    for eq in eqs:
        v, p, _, _ = host_eval(eq, pts)
        assert same_bits(v, p), eq


def test_plane_and_sphere_are_exact():
    rng = np.random.default_rng(2)
    pts = rng.uniform(-1, 1, (3000, 3)).astype(np.float32)
    sx, sy, sz = np.float32(1.1), np.float32(0.7), np.float32(1.3)
    _, _, g, n = host_eval("x+2y-3z+0.1", pts, (sx, sy, sz))
    want = np.array([sx, np.float32(2) * sy, -(np.float32(3) * sz)], np.float32)
    assert same_bits(g, np.tile(want, (len(pts), 1)))
    assert same_bits(n, np.tile(normalise32(want), (len(pts), 1)))
    _, _, g, n = host_eval("x^2+y^2+z^2-0.5", pts, (sx, sy, sz))
    X = pts * np.array([sx, sy, sz], np.float32)
    want = (np.float32(2) * X) * np.array([sx, sy, sz], np.float32)
    assert same_bits(g, want) and same_bits(n, normalise32(want))


def test_normalisation_matches_its_numpy_restatement():
    rng = np.random.default_rng(4)
    g = np.concatenate([rng.normal(size=(5000, 3)).astype(np.float32) * np.float32(10.0) ** rng.integers(-40, 38, (5000, 1)).astype(np.float32),
                        np.array(np.meshgrid(SPECIAL, SPECIAL, SPECIAL)).reshape(3, -1).T.astype(np.float32)])
    n = host_normalise(g)
    assert same_bits(n, normalise32(g))
    big = host_normalise(np.array([[3e38, 3e38, 0]], np.float32))[0]  # no overflow: a direction, not (0,0,0)
    assert big[0] == big[1] > 0.7 and big[2] == 0


def test_kink_conventions():
    def nrm(eq, p):
        return host_eval(eq, np.array([p], np.float32))[3][0]
    assert tuple(nrm("abs(x)", (0.0, 0.2, 0.3))) == (1.0, 0.0, 0.0)
    assert tuple(nrm("abs(x)", (-0.0, 0.2, 0.3))) == (-1.0, 0.0, 0.0)
    r = np.float32(1) / np.sqrt(np.float32(2))
    assert same_bits(nrm("min(x,y)", (0.25, 0.25, 0.0)), np.array([r, r, 0], np.float32))
    assert same_bits(nrm("max(x,-y)", (0.5, -0.5, 0.0)), np.array([r, -r, 0], np.float32))
    assert same_bits(nrm("min(x,y)", (0.0, -0.0, 0.0)), np.array([0, 1, 0], np.float32))  # -0 < +0: min returns y
    for eq, p in (("sqrt(x^2+y^2+z^2)", (0, 0, 0)), ("x^0.5", (0, 0.3, 0.1)), ("1/x", (0, 0.3, 0.1)), ("sqrt(x)", (0, 1, 1))):
        assert tuple(nrm(eq, p)) == (0.0, 0.0, 0.0), eq


# ---- emulated device pipeline --------------------------------------------------------------------------------------------
EMULATED = {"sphere": ("x^2+y^2+z^2-0.49", 0), "torus_sdf": (FUNCTION_EQUATIONS[1], F), "union": (CSG_EQUATIONS[0], F),
            "box": (CSG_BOX_SDF, F), "mixed": (FUNCTION_EQUATIONS[5], F)}


@pytest.mark.parametrize("name", sorted(EMULATED))
@pytest.mark.parametrize("mode", ["dense", "blocks"])
def test_emulated_pipeline_mode3(mcb_emu, name, mode):
    """The device code executed on the host at step 2/32 (33^3 cubes): mode 3's positions, tri_list and counts equal mode
    0's byte for byte, every soup and welded normal is the host build's normal at its position, bit for bit, and soup and
    welded normals agree where the positions do."""
    eq, grammar = EMULATED[name]
    scale = (1.1, 1.1, 1.1)
    fm = mcb_emu.FIELD_DENSE if mode == "dense" else mcb_emu.FIELD_AUTO
    m3 = run_mesh(mcb_emu, eq, 2.0 / 32, scale, NORMALS_ANALYTIC, field_mode=fm, grammar=grammar)
    m0 = run_mesh(mcb_emu, eq, 2.0 / 32, scale, 0, field_mode=fm, grammar=grammar)
    assert m3["counts"].triangles > 200
    assert counts_tuple(m3["counts"]) == counts_tuple(m0["counts"])
    assert same_bits(m3["pos"], m0["pos"]) and same_bits(m3["vl"], m0["vl"]) and np.array_equal(m3["tl"], m0["tl"])
    p = m3["pos"][:, :, :3].reshape(-1, 3)
    assert same_bits(m3["nrm"][:, :, :3].reshape(-1, 3), host_eval(eq, p, scale, grammar)[3])
    assert not m3["nrm"][:, :, 3].any()
    assert same_bits(m3["vn"], host_eval(eq, m3["vl"], scale, grammar)[3])
    a, b, k = soup_matches_welded(m3)
    assert k > len(p) // 2 and same_bits(a, b)


def test_emulated_box_faces_are_flat(mcb_emu):
    """CSG_BOX_SDF, scale 1, step 0.05: every welded vertex strictly inside a face region has a normal of exactly +-1 on the
    face's axis and 0 elsewhere.  Mode 1 (central differences) rounds the normals next to the box's edges; its largest
    deviation there is printed."""
    m3 = run_mesh(mcb_emu, CSG_BOX_SDF, 0.05, normals=NORMALS_ANALYTIC)
    m1 = run_mesh(mcb_emu, CSG_BOX_SDF, 0.05, normals=1)
    assert same_bits(m3["vl"], m1["vl"])
    flat, dev1 = _check_box_faces(m3["vl"], m3["vn"], m1["vn"])
    print("box SDF: %d vertices inside face regions, mode 1's largest deviation there %.3g" % (flat, dev1))
    assert flat > 200 and dev1 > 1e-3


def _check_box_faces(vl, vn3, vn1):
    half = np.array([0.5, 0.4, 0.3], np.float32)
    inside = np.abs(vl) < half  # per axis: strictly within the box's extent
    flat = 0
    dev1 = 0.0
    for ax in range(3):
        o = [i for i in range(3) if i != ax]
        sel = inside[:, o[0]] & inside[:, o[1]] & (np.abs(vl[:, ax]) > half[ax])
        want = np.zeros((int(sel.sum()), 3), np.float32)
        want[:, ax] = np.where(vl[sel, ax] > 0, 1.0, -1.0)
        assert same_bits(vn3[sel], want), ax
        flat += int(sel.sum())
        dev1 = max(dev1, float(np.abs(vn1[sel] - want).max()))
    return flat, dev1
