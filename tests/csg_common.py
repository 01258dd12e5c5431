"""Shared material of the min( / max( tests (test_csg_host.py, test_gpu_csg.py): combined shapes, a random generator of
equations that combine sub-expressions with min / max, and oracle/mc_oracle_csg.c, the oracle's restatement of the whole
function grammar including min and max."""
import ctypes as C
import os

import numpy as np

from oracle import oraclebind

from .functions_common import GRAMMAR_FUNCTIONS, ORACLE, _build, _headers, random_function_equation

# ---- min( max( of the function grammar: unions, intersections and differences of shapes (test_csg_host.py, test_gpu_csg.py)
def _ball(cx, cy, cz, r2):
    """(x-cx)^2+(y-cy)^2+(z-cz)^2-r2 with the signs written out: every term is an axis table of the grid program"""
    t = lambda v, c: v if c == 0 else "(%s%s%s)" % (v, "-" if c > 0 else "+", ("%g" % abs(c)).lstrip("0"))
    return "%s^2+%s^2+%s^2-%s" % (t("x", cx), t("y", cy), t("z", cz), ("%g" % r2).lstrip("0"))


CSG_UNION2 = "min(sqrt(x^2+y^2+z^2)-0.5,sqrt((x-0.45)^2+y^2+z^2)-0.35)"
CSG_LENS = "max(sqrt((x-0.3)^2+y^2+z^2)-0.6,sqrt((x+0.3)^2+y^2+z^2)-0.6)"
CSG_SPHERE_MINUS_CYLINDER = "max(sqrt(x^2+y^2+z^2)-0.7,-(sqrt(x^2+y^2)-0.3))"
CSG_BOX_SDF = "sqrt(max(abs(x)-0.5,0)^2+max(abs(y)-0.4,0)^2+max(abs(z)-0.3,0)^2)-0.1"
_CORNERS = [_ball(0.4 * sx, 0.4 * sy, 0.4 * sz, 0.09) for sz in (-1, 1) for sy in (-1, 1) for sx in (-1, 1)]
CSG_UNION8 = "min(min(min(%s,%s),min(%s,%s)),min(min(%s,%s),min(%s,%s)))" % tuple(_CORNERS)
CSG_EQUATIONS = [CSG_UNION2, CSG_LENS, CSG_SPHERE_MINUS_CYLINDER, CSG_BOX_SDF, CSG_UNION8]


def random_csg_equation(rng, depth):
    """A random string over the function grammar with min( max(: the forms of random_function_equation wrapped in nested
    min / max, with constant-only and single-variable arguments among them (those fold or become axis tables)."""
    r = rng.random()
    if depth <= 0 or r < 0.3:
        return random_function_equation(rng, int(rng.integers(0, 3)))
    if r < 0.75:
        f = ("min", "max")[rng.integers(0, 2)]
        pre = ("", "", "", "2", "-", "x", "0.5")[rng.integers(0, 7)]
        args = [random_csg_equation(rng, depth - 1), random_csg_equation(rng, depth - 1)]
        k = int(rng.integers(0, 2))
        q = rng.random()
        if q < 0.15:  # constant-only
            args[k] = ("%d.%d" % (rng.integers(0, 4), rng.integers(0, 100)), "sqrt(2)-1", "-3", "min(2,0.5)")[rng.integers(0, 4)]
        elif q < 0.35:  # one variable
            v = "xyz"[rng.integers(0, 3)]
            args[k] = ("abs(%s)-0.%d" % (v, rng.integers(1, 10)), "%d.%d%s" % (rng.integers(1, 9), rng.integers(0, 100), v),
                       "max(%s,-%s)" % (v, v), "sqrt(%s)" % v)[rng.integers(0, 4)]
        return pre + f + "(" + args[0] + "," + args[1] + ")"
    if r < 0.85:
        return random_csg_equation(rng, depth - 1) + "+-*/^"[rng.integers(0, 5)] + random_csg_equation(rng, depth - 1)
    if r < 0.93:
        return "(" + random_csg_equation(rng, depth - 1) + ")"
    return ("sin(", "sqrt(", "abs(")[rng.integers(0, 3)] + random_csg_equation(rng, depth - 1) + ")"


def random_csg_equations(mcb, seed, n, max_len=140, min_depth=1, max_depth=4):
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        eq = random_csg_equation(rng, int(rng.integers(min_depth, max_depth + 1)))
        if len(eq) <= max_len and ("min(" in eq or "max(" in eq) and mcb.parse_ok(eq, grammar=GRAMMAR_FUNCTIONS):
            out.append(eq)
    return out


_csg_oracle = None


def csg_oracle_lib():
    """oracle/mc_oracle_csg.c: the plain-C oracle with its own restatement of the function grammar and of min / max"""
    global _csg_oracle
    if _csg_oracle is None:
        so = _build("libmcoracle_csg.so", [os.path.join(ORACLE, "mc_oracle_csg.c")],
                    _headers() + [os.path.join(ORACLE, "mc_oracle.c"), os.path.join(ORACLE, "mc_oracle.h")],
                    ["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-pthread"], shared=True)
        L = C.CDLL(so)
        vp, cp, i, f, l = C.c_void_p, C.c_char_p, C.c_int, C.c_float, C.c_long
        L.mco_create.restype = vp
        L.mco_destroy.argtypes = [vp]
        L.mco_set_pow_mode.argtypes = [vp, i]
        L.mcoc_parse_ok.argtypes = [cp]
        L.mcoc_set_equation.argtypes = [vp, i, cp]
        L.mcoc_min.argtypes = [f, f]
        L.mcoc_min.restype = f
        L.mcoc_max.argtypes = [f, f]
        L.mcoc_max.restype = f
        L.mco_eval_points.argtypes = [vp, i, vp, vp, l, i]
        L.mco_set_step.argtypes = [vp, f]
        L.mco_set_scale.argtypes = [vp, f, f, f]
        L.mco_set_iso.argtypes = [vp, f]
        L.mco_set_constraint.argtypes = [vp, i, i, f, i]
        L.mco_grid.argtypes = [vp, vp, i]
        L.mco_sweep.argtypes = [vp, i, i, i, vp, vp, vp, vp, vp, l, vp, vp, vp]
        L.mco_sweep.restype = l
        L.mco_recalculate.argtypes = [vp, i]
        L.mco_recalculate.restype = l
        L.mco_num_vertices.argtypes = [vp]
        L.mco_num_vertices.restype = l
        L.mco_num_triangles.argtypes = [vp]
        L.mco_num_triangles.restype = l
        L.mco_copy_mesh.argtypes = [vp, vp, vp]
        _csg_oracle = L
    return _csg_oracle


def csg_parse_ok(eq):
    return bool(csg_oracle_lib().mcoc_parse_ok(eq.encode()))


def csg_oracle_minmax():
    """mcoc_min / mcoc_max: the oracle's own restatement of minimumNumber / maximumNumber"""
    L = csg_oracle_lib()
    return L.mcoc_min, L.mcoc_max


class CsgOracle(oraclebind.Oracle):
    """The oracle's reference pipeline (oracle/oraclebind.py's methods) on equations of the function grammar with min and
    max: surface and constraint left-hand sides parse with mc_oracle_csg.c's tokenizer."""

    def __init__(self, eq, step=None, scale=(1.0, 1.0, 1.0), iso=0.0, pow_mode=1, cons=()):
        self.L = csg_oracle_lib()
        self.h = C.c_void_p(self.L.mco_create())
        self.L.mco_set_pow_mode(self.h, pow_mode)
        if not self.L.mcoc_set_equation(self.h, 0, eq.encode()):
            raise ValueError("oracle rejected %r" % eq)
        if step is not None:
            self.M = self.L.mco_set_step(self.h, step)
        self.L.mco_set_scale(self.h, *scale)
        self.L.mco_set_iso(self.h, iso)
        for k, (lhs, op, rhs) in enumerate(cons):
            assert self.L.mcoc_set_equation(self.h, k + 1, lhs.encode()), lhs
            assert self.L.mco_set_constraint(self.h, k, {">": 0, "<": 1, ">=": 2, "<=": 3}[op], rhs, 1)

    def set_equation(self, slot, eq):
        return bool(self.L.mcoc_set_equation(self.h, slot, eq.encode()))
