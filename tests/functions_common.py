"""Shared material of the function-grammar tests (test_functions_host.py, test_gpu_functions.py)."""
import numpy as np

GRAMMAR_FUNCTIONS = 1

# a literal gyroid (4 pi = 12.566371: two periods over [-1, 1]) and signed-distance shapes
GYROID = "sin(12.566371x)cos(12.566371y)+sin(12.566371y)cos(12.566371z)+sin(12.566371z)cos(12.566371x)"
TORUS_SDF = "sqrt((sqrt(x^2+y^2)-0.5)^2+z^2)-0.2"
NONHOIST = "sin(6(x^2+y^2+z^2))"
OCTAHEDRON = "abs(x)+abs(y)+abs(z)-0.7"
SCHWARZ_P = "cos(9.424778x)+cos(9.424778y)+cos(9.424778z)"
MIXED = "sqrt(abs(x*y)+z^2)-0.4+0.1sin(7x+5y)cos(3z-x)"

FUNCTION_EQUATIONS = [GYROID, TORUS_SDF, NONHOIST, OCTAHEDRON, SCHWARZ_P, MIXED]

# 8 pi = 25.132741: at step 1/8 the product of cosines is +-1 and changes sign at every grid vertex, so every cube is
# active with 12 crossing edges and a 64-cube chunk of the soup emitter needs 768 edge slots, more than its 512: the
# chunk is emitted in several runs.  The small polynomial keeps the gradient away from zero, so the normals mean something
# (the cosines' central differences are 0 at every vertex).  Not +0.1(x+y^2+z^3): there the reference's vertex set keeps
# 10 duplicate vertices, the documented deviation of the weld (DESIGN.md §5, K4).
CHECKER = "cos(25.132741x)cos(25.132741y)cos(25.132741z)+0.1(x^3+0.6y+0.3z^2)"


def random_function_equation(rng, depth):
    """A random string over the function grammar: the reference's forms (variables, numbers, + - * / ^, brackets,
    unary minus, implicit multiplication) plus sin( cos( sqrt( abs( around sub-expressions, including constant-only
    and single-variable arguments, and with implicit multiplication before a function."""
    r = rng.random()
    if depth <= 0 or r < 0.22:
        k = rng.integers(0, 6)
        if k < 3:
            return "xyz"[k]
        if k == 3:
            return str(int(rng.integers(0, 10)))
        if k == 4:
            return "%d.%d" % (rng.integers(0, 4), rng.integers(0, 100))
        return "XYZ"[rng.integers(0, 3)]
    if r < 0.50:
        f = ("sin", "cos", "sqrt", "abs")[rng.integers(0, 4)]
        pre = ("", "", "2", "-", "x", "0.5")[rng.integers(0, 6)]
        inner = random_function_equation(rng, depth - 1)
        if rng.random() < 0.3:  # a single-variable argument with a scale: hoisted into an axis table
            inner = "%d.%d%s" % (rng.integers(1, 20), rng.integers(0, 100), "xyz"[rng.integers(0, 3)])
        return pre + f + "(" + inner + ")"
    if r < 0.58:
        return "(" + random_function_equation(rng, depth - 1) + ")"
    if r < 0.63:
        return "-" + random_function_equation(rng, depth - 1)
    if r < 0.68:
        return random_function_equation(rng, depth - 1) + "(" + random_function_equation(rng, depth - 1) + ")"
    return random_function_equation(rng, depth - 1) + "+-*/^"[rng.integers(0, 5)] + random_function_equation(rng, depth - 1)


def random_function_equations(mcb, seed, n, max_len=110, min_depth=1, max_depth=5):
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        eq = random_function_equation(rng, int(rng.integers(min_depth, max_depth + 1)))
        if len(eq) <= max_len and ("sin" in eq or "cos" in eq or "sqrt" in eq or "abs" in eq) and \
                mcb.parse_ok(eq, grammar=GRAMMAR_FUNCTIONS):
            out.append(eq)
    return out


# ---- test-only native helpers, compiled on first use into a temporary directory (the tree may be read-only) ----------
import ctypes as C  # noqa: E402
import hashlib  # noqa: E402
import os  # noqa: E402
import subprocess  # noqa: E402
import tempfile  # noqa: E402

from oracle import oraclebind  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "csrc")
ORACLE = os.path.join(ROOT, "oracle")


def _build(name, sources, deps, cmd_head, shared):
    """Compile `sources` (+ `deps` in the hash) once per content into $TMPDIR/mcb_functions_<hash>/<name>."""
    h = hashlib.sha256()
    for p in sorted(set(sources + deps)):
        h.update(p.encode() + open(p, "rb").read())
    h.update(" ".join(cmd_head).encode())
    out_dir = os.path.join(tempfile.gettempdir(), "mcb_functions_" + h.hexdigest()[:16])
    out = os.path.join(out_dir, name)
    if not os.path.exists(out):
        os.makedirs(out_dir, exist_ok=True)
        tmp = out + ".%d" % os.getpid()
        cmd = cmd_head + (["-shared", "-fPIC"] if shared else []) + ["-o", tmp] + sources + ["-lm"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("building %s failed:\n%s" % (name, r.stdout + r.stderr))
        os.replace(tmp, out)
    return out


def _headers():
    return [os.path.join(CSRC, f) for f in ("mcb_pow.h", "mcb_trig.h", "mcb_bytecode.h", "mcb_interval.h", "mcb_lower.h", "mcb_tables.h")] + \
        [os.path.join(ROOT, "include", "mcb.h")]


def trig_exhaustive_exe():
    """oracle/trig_exhaustive: csrc/mcb_trig.h against libm sinf / cosf."""
    return _build("trig_exhaustive", [os.path.join(ORACLE, "trig_exhaustive.c")], _headers(),
                  ["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-pthread"], shared=False)


def host_fn_lib():
    """oracle/host_interp_fn.cpp: the product's lowering and host interpreters (host_interp.cpp) under a chosen grammar."""
    so = _build("libmcoracle_host_fn.so", [os.path.join(ORACLE, "host_interp_fn.cpp"), os.path.join(CSRC, "mcb_lower.cpp")],
                _headers() + [os.path.join(ORACLE, "host_interp.cpp")], ["g++", "-std=c++17", "-O2", "-ffp-contract=off"], shared=True)
    H = C.CDLL(so)
    vp = C.c_void_p
    H.mcoh_set_grammar.argtypes = [C.c_int]
    H.mcoh_set_grammar(GRAMMAR_FUNCTIONS)
    H.mcoh_eval_points.argtypes = [C.c_char_p, vp, vp, C.c_long]
    H.mcoh_eval_grid.argtypes = [C.c_char_p, vp, C.c_int, vp, C.c_int, vp, C.c_int, vp]
    H.mcoh_tables.argtypes = [C.c_char_p, vp, vp, vp, C.c_int, vp, C.c_int, vp]
    H.mcoh_interval_check.argtypes = [C.c_char_p, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp]
    return H


_fn_oracle = None


def fn_oracle_lib():
    """oracle/mc_oracle_fn.c: the plain-C oracle with its own restatement of the function grammar (libm sinf/cosf/...)."""
    global _fn_oracle
    if _fn_oracle is None:
        so = _build("libmcoracle_fn.so", [os.path.join(ORACLE, "mc_oracle_fn.c")],
                    _headers() + [os.path.join(ORACLE, "mc_oracle.c"), os.path.join(ORACLE, "mc_oracle.h")],
                    ["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-pthread"], shared=True)
        L = C.CDLL(so)
        vp, cp, i, f, l = C.c_void_p, C.c_char_p, C.c_int, C.c_float, C.c_long
        L.mco_create.restype = vp
        L.mco_destroy.argtypes = [vp]
        L.mco_set_pow_mode.argtypes = [vp, i]
        L.mcof_parse_ok.argtypes = [cp]
        L.mcof_set_equation.argtypes = [vp, i, cp]
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
        _fn_oracle = L
    return _fn_oracle


def fn_parse_ok(eq):
    return bool(fn_oracle_lib().mcof_parse_ok(eq.encode()))


class FnOracle(oraclebind.Oracle):
    """The oracle's reference pipeline (oracle/oraclebind.py's methods) on function-grammar equations: surface and
    constraint left-hand sides parse with mc_oracle_fn.c's tokenizer."""

    def __init__(self, eq, step=None, scale=(1.0, 1.0, 1.0), iso=0.0, pow_mode=1, cons=()):
        self.L = fn_oracle_lib()
        self.h = C.c_void_p(self.L.mco_create())
        self.L.mco_set_pow_mode(self.h, pow_mode)
        if not self.L.mcof_set_equation(self.h, 0, eq.encode()):
            raise ValueError("oracle rejected %r" % eq)
        if step is not None:
            self.M = self.L.mco_set_step(self.h, step)
        self.L.mco_set_scale(self.h, *scale)
        self.L.mco_set_iso(self.h, iso)
        for k, (lhs, op, rhs) in enumerate(cons):
            assert self.L.mcof_set_equation(self.h, k + 1, lhs.encode()), lhs
            assert self.L.mco_set_constraint(self.h, k, {">": 0, "<": 1, ">=": 2, "<=": 3}[op], rhs, 1)

    def set_equation(self, slot, eq):
        return bool(self.L.mcof_set_equation(self.h, slot, eq.encode()))
