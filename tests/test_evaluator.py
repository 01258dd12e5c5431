"""The operator table (csrc/mcb_bytecode.h): every operation of the grammar is written once, for float values and for the
dual numbers of the analytic normals.  One small equation per operation, at inputs that include the kinks of abs, min and
max and sqrt(0):
  - CPU: together the equations reach every postfix opcode; the dual evaluation's value part equals the plain value bit for
    bit; the gradients at the kinks are the conventions include/mcb.h states.
  - GPU: device values (mcb_eval_points) and device gradients (mcb_eval_gradients) equal the host build's bit for bit, and
    the meshes of a fixed set of equations (soup and welded positions, analytic normals, refined positions) are
    byte-identical to the ones the build before the operator table produced (tests/golden/evaluator_mesh_hashes.json,
    written by tests/golden/make_evaluator_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

from .csg_common import CSG_BOX_SDF, CSG_LENS, CSG_SPHERE_MINUS_CYLINDER, CSG_UNION2
from .functions_common import GRAMMAR_FUNCTIONS, GYROID, OCTAHEDRON, TORUS_SDF
from .helpers import same_bits
from .normals_common import host_eval

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = GRAMMAR_FUNCTIONS
OPERATORS = {"ADD": "x+y", "SUB": "x-y", "RSUB": "z-x*y", "MUL": "x*y", "DIV": "x/y", "RDIV": "z/(x*y)", "POW": "x^y",
             "RPOW": "z^(x*y)", "POW2": "x^2", "NEG": "-x+2.5", "SIN": "sin(x)", "COS": "cos(x)", "SQRT": "sqrt(x)",
             "ABS": "abs(x)", "MIN": "min(x,y)", "MAX": "max(x,y)"}
KINKS = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, 1.0, -1.0, 0.5, 2.0, -2.5, 3.4e38, np.inf, -np.inf, np.nan, 0.37],
                 np.float32)
MESH_CASES = {  # name: (equation, grammar, step)
    "sphere": ("x^2+y^2+z^2-0.49", 0, 0.0625), "pow_div": ("2^x*y-z/(1.5+x)-0.3", 0, 0.0625),
    "gyroid": (GYROID, F, 0.0625), "torus_sdf": (TORUS_SDF, F, 0.0625), "octahedron": (OCTAHEDRON, F, 0.0625),
    "box_sdf": (CSG_BOX_SDF, F, 0.0625), "union2": (CSG_UNION2, F, 0.0625), "lens": (CSG_LENS, F, 0.0625),
    "sphere_minus_cylinder": (CSG_SPHERE_MINUS_CYLINDER, F, 0.0625)}
MESH_SCALE = (1.1, 0.9, 1.3)
HASHES = os.path.join(ROOT, "tests", "golden", "evaluator_mesh_hashes.json")


def kink_points():
    """every (x, y) pair of KINKS, with z = 0.37 and z = -0.0"""
    x, y, z = np.meshgrid(KINKS, KINKS, np.array([0.37, -0.0], np.float32), indexing="ij")
    return np.stack([x.ravel(), y.ravel(), z.ravel()], axis=1)


def mesh_digests(mcb, name):
    """sha256 per refinement setting of the counts and the bytes of soup positions and normals, welded vertices, indices
    and normals, with analytic normals (mode 3)"""
    from .refine_common import counts_tuple, run_refined
    eq, grammar, step = MESH_CASES[name]
    out = {}
    for refine in (False, True):
        m = run_refined(mcb, eq, step, MESH_SCALE, refine, normals=3, grammar=grammar)
        h = hashlib.sha256(repr(counts_tuple(m["counts"])).encode())
        for k in ("pos", "nrm", "vl", "tl", "vn"):
            h.update(np.ascontiguousarray(m[k]).tobytes())
        out["refined" if refine else "linear"] = h.hexdigest()
    return out


def test_the_equations_reach_every_opcode(mcb):
    ops = set()
    for eq in OPERATORS.values():
        ops |= set(mcb.disassemble(eq, 0, grammar=F).split())
    assert {k for k in OPERATORS if k != "POW2"} <= ops, ops


@pytest.mark.parametrize("op", sorted(OPERATORS))
def test_dual_value_part_is_the_plain_value(op):
    value, plain, _, _ = host_eval(OPERATORS[op], kink_points())
    assert same_bits(value, plain), op


def test_gradients_at_the_kinks():
    """abs takes the sign bit of its operand, min / max the operand whose bits the result has and the mean on a tie,
    sqrt(0) divides by 0 + 0"""
    f32 = np.float32
    p = np.array([[0.0, 0, 0], [-0.0, 0, 0], [1, 1, 0], [0.0, -0.0, 0], [-0.0, 0.0, 0]], f32)
    _, _, g, _ = host_eval("abs(x)", p[:2])
    assert same_bits(g, np.array([[1, 0, 0], [-1, -0.0, -0.0]], f32))
    _, _, g, _ = host_eval("min(x,y)", p[2:])
    assert same_bits(g, np.array([[0.5, 0.5, 0], [0, 1, 0], [1, 0, 0]], f32))  # min(+0,-0) = -0, y's bits
    _, _, g, _ = host_eval("max(x,y)", p[2:])
    assert same_bits(g, np.array([[0.5, 0.5, 0], [1, 0, 0], [0, 1, 0]], f32))  # max(+0,-0) = +0
    with np.errstate(all="ignore"):
        _, _, g, _ = host_eval("sqrt(x)", p[:2])
        assert same_bits(g, np.array([[1, 0, 0], [1, 0, 0]], f32) / np.array([[0.0], [-0.0]], f32))  # sqrt(-0) = -0


@pytest.mark.gpu
def test_device_values_and_gradients_equal_the_host(mcb):
    pts = kink_points()
    c = mcb.Context(0)
    try:
        c.set_grammar(F)
        c.set_scaling(*MESH_SCALE)
        for op, eq in sorted(OPERATORS.items()):
            assert c.set_equation(eq) == 0, eq
            for scale in ((1.0, 1.0, 1.0), MESH_SCALE):
                value, plain, grad, _ = host_eval(eq, pts, scale)
                applied = scale != (1.0, 1.0, 1.0)
                assert same_bits(c.eval_points(pts, apply_scale=applied), plain), (op, scale)
                assert same_bits(c.eval_gradients(pts, apply_scale=applied), grad), (op, scale)
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MESH_CASES))
def test_meshes_equal_the_build_before_the_operator_table(mcb, name):
    assert mesh_digests(mcb, name) == json.load(open(HASHES))[name]
