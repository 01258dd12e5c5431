"""TEST INFRASTRUCTURE ONLY — ctypes binding of oracle/libmcoracle.so (the plain-C restatement, oracle/mc_oracle.c).
May be imported only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libmcoracle.so")
_lib = None


def available():
    return os.path.exists(SO)


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(SO)
        vp, cp, i, f, l = C.c_void_p, C.c_char_p, C.c_int, C.c_float, C.c_long
        L.mco_create.restype = vp
        L.mco_destroy.argtypes = [vp]
        L.mco_set_pow_mode.argtypes = [vp, i]
        L.mco_parse_ok.argtypes = [cp]
        L.mco_tokenize_ok.argtypes = [cp]
        L.mco_set_equation.argtypes = [vp, i, cp]
        L.mco_evaluate.argtypes = [vp, i, f, f, f]
        L.mco_evaluate.restype = f
        L.mco_eval_points.argtypes = [vp, i, vp, vp, l, i]
        L.mco_set_step.argtypes = [vp, f]
        L.mco_set_scale.argtypes = [vp, f, f, f]
        L.mco_set_iso.argtypes = [vp, f]
        L.mco_set_repeat.argtypes = [vp, i, f]
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
        L.mco_normals.argtypes = [vp, vp]
        L.mco_timed_rows.argtypes = [vp, l, l, i, vp, vp]
        L.mco_timed_rows.restype = C.c_double
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Oracle:
    def __init__(self, eq=None, step=None, scale=(1.0, 1.0, 1.0), iso=0.0, pow_mode=0, cons=(), repeat=0.0):
        self.L = lib()
        self.h = C.c_void_p(self.L.mco_create())
        self.L.mco_set_pow_mode(self.h, pow_mode)
        if eq is not None and not self.L.mco_set_equation(self.h, 0, eq.encode()):
            raise ValueError("oracle rejected %r" % eq)
        if step is not None:
            self.M = self.L.mco_set_step(self.h, step)
        self.L.mco_set_scale(self.h, *scale)
        self.L.mco_set_iso(self.h, iso)
        if repeat:
            assert self.L.mco_set_repeat(self.h, 1, repeat)
        for i, (lhs, op, rhs) in enumerate(cons):
            assert self.L.mco_set_equation(self.h, i + 1, lhs.encode())
            assert self.L.mco_set_constraint(self.h, i, {">": 0, "<": 1, ">=": 2, "<=": 3}[op], rhs, 1)

    def __del__(self):
        try:
            self.L.mco_destroy(self.h)
        except Exception:
            pass

    def eval_points(self, xyz, scaled=False, slot=0):
        xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
        out = np.empty(len(xyz), np.float32)
        self.L.mco_eval_points(self.h, slot, _p(xyz), _p(out), len(xyz), int(scaled))
        return out

    def coords(self):
        M = self.L.mco_grid(self.h, None, 0)
        c = np.empty(M + 1, np.float32)
        self.L.mco_grid(self.h, _p(c), M + 1)
        return M, c

    def sweep(self, k0=0, k1=None, nthreads=None, soup=True, grad_normals=False):
        M = self.L.mco_grid(self.h, None, 0)
        k1 = M if k1 is None else k1
        nthreads = nthreads or (os.cpu_count() or 1)
        n = (k1 - k0) * M * M
        code, tidx, ntri = np.zeros(n, np.uint8), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        na, nb, nr = C.c_long(0), C.c_long(0), C.c_long(0)
        T = self.L.mco_sweep(self.h, k0, k1, nthreads, _p(code), _p(tidx), _p(ntri), None, None, 0, C.byref(na), C.byref(nb), C.byref(nr))
        out = dict(M=M, code=code, table_idx=tidx, ntri=ntri, T=int(T), active=na.value, ambiguous=nb.value, redirected=nr.value)
        if soup or grad_normals:
            s = np.zeros((max(T, 1), 3, 3), np.float32) if soup else None
            g = np.zeros((max(T, 1), 3, 3), np.float32) if grad_normals else None
            self.L.mco_sweep(self.h, k0, k1, nthreads, None, None, None, _p(s), _p(g), T, None, None, None)
            if soup:
                out["soup"] = s[:T]
            if grad_normals:
                out["grad_normals"] = g[:T]
        return out

    def recalculate(self, nthreads=None):
        self.L.mco_recalculate(self.h, nthreads or (os.cpu_count() or 1))
        nv, nt = self.L.mco_num_vertices(self.h), self.L.mco_num_triangles(self.h)
        v, t = np.empty((nv, 3), np.float32), np.empty((nt, 3), np.uint32)
        self.L.mco_copy_mesh(self.h, _p(v), _p(t))
        return v, t

    def normals(self):
        n = np.empty((self.L.mco_num_vertices(self.h), 3), np.float32)
        self.L.mco_normals(self.h, _p(n))
        return n

    def timed_rows(self, row0, nrows, nthreads):
        cubes, tris = C.c_long(0), C.c_long(0)
        sec = self.L.mco_timed_rows(self.h, row0, nrows, nthreads, C.byref(cubes), C.byref(tris))
        return sec, cubes.value, tris.value
