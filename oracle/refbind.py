"""TEST INFRASTRUCTURE ONLY — ctypes binding of oracle/_ref/libmcref.so (the unmodified reference
compiled by oracle/Makefile behind oracle/ref_harness.cpp).

May be imported only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs.  The product package never imports this module.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libmcref.so")

# The reference's example_files/equation_{1..8}.txt contents (one line each, no newline) — inputs only.
EXAMPLE_EQUATIONS = {
    1: "x+y",
    2: "x^2*y^2+x^2*z^2+z^2*y^2+x*y*z",
    3: "(x^2+y^2+z^2+(1/3)^2-(1/5)^2)^2-4*((1/2)*x-(2.36/6)*(1/5))^2-4*(1/3)^2*y^2",
    4: "(x^2+y^2+z^2+(1/3)^2-(5/12)^2)^2-4*((1/2)*x-(2.36/6)*(5/12))^2-4*(1/3)^2*y^2",
    5: "(x^2+y^2+z^2+(1/3)^2-(3/4)^2)^2-4*((1/2)*x-(2.36/6)*(3/4))^2-4*(1/3)^2*y^2",
    6: "(x+0.5)*(x^2+y^2+z^2-0.5^2*0.5^2*0.25)+0.5*z^2",
    7: "(x+1.5)*(x^2+y^2+z^2-((3/2)^2*(1/2)^2*0.25))+0.5*z^2",
    8: "(x^2+y^2-(1/16))^2+(y^2+z^2-(1/16))^2+(z^2+x^2-(1/16))^2-8*(x^2+y^2+z^2-(1/4))^2",
}
SPHERE = "x^2+y^2+z^2-0.49"
TORUS = "(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)"
GYR34 = ("((x*(-3+4*x^2))*(1+y^2*(-8+8*y^2)))+((y*(-3+4*y^2))*(1+z^2*(-8+8*z^2)))"
         "+((z*(-3+4*z^2))*(1+x^2*(-8+8*x^2)))")
GYR78 = ("((x*(-7+x^2*(56+x^2*(-112+64*x^2))))*(1+y^2*(-32+y^2*(160+y^2*(-256+128*y^2)))))"
         "+((y*(-7+y^2*(56+y^2*(-112+64*y^2))))*(1+z^2*(-32+z^2*(160+z^2*(-256+128*z^2)))))"
         "+((z*(-7+z^2*(56+z^2*(-112+64*z^2))))*(1+x^2*(-32+x^2*(160+x^2*(-256+128*x^2)))))")


def available():
    return os.path.exists(REF_SO)


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(REF_SO)
        L.mcref_create.restype = C.c_void_p
        L.mcref_destroy.argtypes = [C.c_void_p]
        L.mcref_parse_ok.argtypes = [C.c_char_p]
        L.mcref_set_equation.argtypes = [C.c_void_p, C.c_char_p]
        L.mcref_evaluate.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float]
        L.mcref_evaluate.restype = C.c_float
        L.mcref_eval_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long]
        L.mcref_march_eval_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long]
        L.mcref_set_step.argtypes = [C.c_void_p, C.c_float]
        L.mcref_force_step.argtypes = [C.c_void_p, C.c_float]
        L.mcref_get_step.argtypes = [C.c_void_p]
        L.mcref_get_step.restype = C.c_float
        L.mcref_set_scale.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float]
        L.mcref_set_iso.argtypes = [C.c_void_p, C.c_float]
        L.mcref_set_constraint.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_float, C.c_int]
        L.mcref_recalculate.argtypes = [C.c_void_p]
        L.mcref_set_repeat.argtypes = [C.c_void_p, C.c_int, C.c_float]
        L.mcref_seed_recalculate.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float]
        L.mcref_step_all.argtypes = [C.c_void_p, C.c_long]
        L.mcref_step_all.restype = C.c_long
        L.mcref_num_vertices.argtypes = [C.c_void_p]
        L.mcref_num_vertices.restype = C.c_long
        L.mcref_num_triangles.argtypes = [C.c_void_p]
        L.mcref_num_triangles.restype = C.c_long
        L.mcref_copy_mesh.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mcref_normals.argtypes = [C.c_void_p, C.c_void_p]
        L.mcref_grid_coords.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.mcref_sweep.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_long, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mcref_sweep.restype = C.c_long
        L.mcref_timed_rows_mt.argtypes = [C.c_char_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                          C.c_long, C.c_long, C.c_int, C.c_void_p, C.c_void_p]
        L.mcref_timed_rows_mt.restype = C.c_double
        L.mcref_timed_recalculate.argtypes = [C.c_void_p]
        L.mcref_timed_recalculate.restype = C.c_double
        L.mcref_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def parse_ok(eq):
    """Evaluator::tokenize's verdict on `eq`."""
    return bool(lib().mcref_parse_ok(eq.encode()))


def fnv1a64(b: bytes) -> str:
    h = 0xCBF29CE484222325
    for x in b:
        h ^= x
        h = (h * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return "%016x" % h


class Ref:
    """One reference Evaluator + Marching pair."""

    def __init__(self, eq=None, step=None, scale=(1.0, 1.0, 1.0), iso=0.0, force_step=False):
        self.L = lib()
        self.h = C.c_void_p(self.L.mcref_create())
        if eq is not None:
            if not self.set_equation(eq):
                raise ValueError("reference rejected equation %r" % eq)
        if step is not None:
            if force_step:
                self.L.mcref_force_step(self.h, step)
            elif not self.L.mcref_set_step(self.h, step):
                raise ValueError("reference rejected step %r" % step)
        self.L.mcref_set_scale(self.h, *scale)
        self.L.mcref_set_iso(self.h, iso)

    def __del__(self):
        try:
            self.L.mcref_destroy(self.h)
        except Exception:
            pass

    def set_equation(self, eq):
        return bool(self.L.mcref_set_equation(self.h, eq.encode()))

    def evaluate(self, x, y, z):
        return float(self.L.mcref_evaluate(self.h, x, y, z))

    def eval_points(self, xyz, scaled=False):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        out = np.empty(len(xyz), dtype=np.float32)
        f = self.L.mcref_march_eval_points if scaled else self.L.mcref_eval_points
        f(self.h, _p(xyz), _p(out), len(xyz))
        return out

    def set_constraint(self, i, lhs, op, rhs, in_use=True):
        opi = {">": 0, "<": 1, ">=": 2, "<=": 3}[op]
        return bool(self.L.mcref_set_constraint(self.h, i, lhs.encode(), opi, rhs, int(in_use)))

    def coords(self):
        M = self.L.mcref_grid_coords(self.h, None, 0)
        c = np.empty(M + 1, dtype=np.float32)
        self.L.mcref_grid_coords(self.h, _p(c), M + 1)
        return M, c

    def set_repeat(self, on, distance=0.0):
        """Repeating-surface mode via set_surface_repeat_step_distance + repeating_surface_mode."""
        return bool(self.L.mcref_set_repeat(self.h, int(bool(on)), distance))

    def recalculate(self):
        """Unmodified Marching::recalculate(); returns (vertex_list[n,3], tri_list[t,3])."""
        self.L.mcref_recalculate(self.h)
        return self.mesh()

    def step_all(self, max_calls=10 ** 7):
        """Step-by-step mode run to completion (one cube per recalculate(), marching.cpp:386-428).
        Returns (calls, vertex_list, tri_list)."""
        n = self.L.mcref_step_all(self.h, max_calls)
        v, t = self.mesh()
        return n, v, t

    def seed_recalculate(self, sx, sy, sz):
        """Seed mode: only the cubes face-connected (through crossing faces) to the cube containing the seed, in BFS
        order (marching.cpp:310-331).  Returns (vertex_list, tri_list) or None when the seed is rejected."""
        if not self.L.mcref_seed_recalculate(self.h, sx, sy, sz):
            return None
        return self.mesh()

    def mesh(self):
        nv, nt = self.L.mcref_num_vertices(self.h), self.L.mcref_num_triangles(self.h)
        v = np.empty((nv, 3), dtype=np.float32)
        t = np.empty((nt, 3), dtype=np.uint32)
        self.L.mcref_copy_mesh(self.h, _p(v), _p(t))
        return v, t

    def normals(self):
        nv = self.L.mcref_num_vertices(self.h)
        n = np.empty((nv, 3), dtype=np.float32)
        self.L.mcref_normals(self.h, _p(n))
        return n

    def sweep(self, k0=0, k1=None, corners=False, soup=True, weld=False):
        M, _ = self.coords()
        if k1 is None:
            k1 = M
        n = (k1 - k0) * M * M
        code = np.zeros(n, np.uint8)
        tidx = np.zeros(n, np.uint8)
        ntri = np.zeros(n, np.uint8)
        cv = np.zeros((n, 8), np.float32) if corners else None
        na, nb, nr = C.c_long(0), C.c_long(0), C.c_long(0)
        T = self.L.mcref_sweep(self.h, k0, k1, _p(code), _p(tidx), _p(ntri), _p(cv), None, 0, 0,
                               C.byref(na), C.byref(nb), C.byref(nr))
        out = dict(M=M, code=code, table_idx=tidx, ntri=ntri, T=int(T), active=na.value, ambiguous=nb.value,
                   redirected=nr.value)
        if corners:
            out["corner_values"] = cv
        if soup or weld:
            s = np.zeros((max(T, 1), 3, 3), np.float32)
            self.L.mcref_sweep(self.h, k0, k1, None, None, None, None, _p(s), T, int(weld), None, None, None)
            out["soup"] = s[:T]
        return out


def sweep_rows_mt(eq, step, row0, row1, nthreads=None, scale=(1.0, 1.0, 1.0), iso=0.0, force_step=True):
    """Per-cube code / table_idx / ntri and the triangle soup of cube rows [row0, row1) (row = k*M + j) from the UNMODIFIED
    reference, the rows spread over `nthreads` threads with one Evaluator + Marching pair each (they share no state; the
    calls release the GIL).  Order of the outputs = the reference's loop order."""
    import threading
    nthreads = nthreads or min(32, os.cpu_count() or 1)
    L = lib()
    L.mcref_sweep_rows.restype = C.c_long
    L.mcref_sweep_rows.argtypes = [C.c_void_p, C.c_long, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    refs = [Ref(eq, step, scale, iso, force_step=force_step) for _ in range(nthreads)]
    M, _ = refs[0].coords()
    cuts = [row0 + (row1 - row0) * t // nthreads for t in range(nthreads + 1)]
    parts = [None] * nthreads

    def work(t):
        a, b = cuts[t], cuts[t + 1]
        n = (b - a) * M
        code, tidx, ntri = np.zeros(n, np.uint8), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        na, nb, nr = C.c_long(0), C.c_long(0), C.c_long(0)
        T = L.mcref_sweep_rows(refs[t].h, a, b, _p(code), _p(tidx), _p(ntri), None, None, 0, 0, C.byref(na), C.byref(nb), C.byref(nr))
        soup = np.zeros((max(T, 1), 3, 3), np.float32)
        L.mcref_sweep_rows(refs[t].h, a, b, None, None, None, None, _p(soup), T, 0, None, None, None)
        parts[t] = (code, tidx, ntri, soup[:T], int(T), na.value, nb.value, nr.value)
    th = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    return dict(M=M, code=np.concatenate([p[0] for p in parts]), table_idx=np.concatenate([p[1] for p in parts]),
                ntri=np.concatenate([p[2] for p in parts]), soup=np.concatenate([p[3] for p in parts]), T=sum(p[4] for p in parts),
                active=sum(p[5] for p in parts), ambiguous=sum(p[6] for p in parts), redirected=sum(p[7] for p in parts))


def timed_rows_mt(eq, step, scale=(1.0, 1.0, 1.0), iso=0.0, row0=0, nrows=1 << 40, nthreads=1):
    """Reference CPU baseline over cube rows [row0,row0+nrows) (row = k*M+j); returns (seconds, cubes, triangles)."""
    cubes, tris = C.c_long(0), C.c_long(0)
    sec = lib().mcref_timed_rows_mt(eq.encode(), step, scale[0], scale[1], scale[2], iso, row0, nrows, nthreads,
                                    C.byref(cubes), C.byref(tris))
    return sec, cubes.value, tris.value


def tables():
    tri = np.zeros((256, 16), np.int32)
    amb = np.zeros((256, 5), np.int32)
    edge = np.zeros((12, 2), np.int32)
    lib().mcref_tables(_p(tri), _p(amb), _p(edge))
    return tri, amb, edge
