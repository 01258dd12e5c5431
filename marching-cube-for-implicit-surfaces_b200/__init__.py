"""marching-cube-for-implicit-surfaces_b200 — Python face of libmcb200.so (the C ABI in include/mcb.h).

This module is a thin ctypes mirror of the reference's two entry-point classes for the hot path:

    Evaluator  (Source/evaluator.h:24-86)   set_equation / evaluate
    Marching   (Source/marching.h:72-157)   set_evaluator / set_grid_step_size / set_scaling_* /
                                            set_surface_constant / set_constraint* / use_constraint* / recalculate /
                                            get_poly_data

with the same names, argument meaning and bool-return error convention, so that parity tests read like calls into
the reference.  All computation happens in CUDA kernels behind the C ABI; there is no Python or CPU implementation
of the path here, and importing the module fails loudly if the native library has not been built.

The directory name contains hyphens, so import it with
    importlib.import_module("marching-cube-for-implicit-surfaces_b200")
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmcb200.so")

MESH_SOUP, MESH_INDEXED = 1, 2
MESH_DC = 4  # dual contouring, used alone: one vertex per active cube on sharp edges and corners (include/mcb.h, DESIGN.md §14)
FIELD_DENSE, FIELD_SPARSE, FIELD_AUTO = 0, 1, 2
JIT_OFF, JIT_ON, JIT_AUTO = 0, 1, 2
GRAMMAR_REFERENCE, GRAMMAR_FUNCTIONS = 0, 1  # the reference's equation language / the same plus sin( cos( sqrt( abs( min( max(
NORMALS_ANALYTIC = 3  # set_normals mode: the equation's own gradient at every output vertex (include/mcb.h, DESIGN.md §12)
MCB_OK, MCB_E_PARSE, MCB_E_ARG, MCB_E_CUDA, MCB_E_NOMEM, MCB_E_STATE, MCB_E_CAPACITY, MCB_E_NODEVICE = 0, -1, -2, -3, -4, -5, -6, -7


class McbError(RuntimeError):
    def __init__(self, status, msg=""):
        self.status = status
        super().__init__("mcb status %d (%s) %s" % (status, status_string(status), msg))


class Counts(C.Structure):
    _fields_ = [("cubes", C.c_uint64), ("active", C.c_uint64), ("triangles", C.c_uint64), ("ambiguous", C.c_uint64),
                ("redirected", C.c_uint64), ("M", C.c_int32), ("k_begin", C.c_int32), ("k_end", C.c_int32),
                ("ms_tables", C.c_float), ("ms_eval", C.c_float), ("ms_classify", C.c_float), ("ms_emit", C.c_float),
                ("ms_total", C.c_float), ("launches", C.c_uint32), ("reruns", C.c_uint32), ("ms_weld", C.c_float),
                ("mesh_mode", C.c_uint32), ("vertices", C.c_uint64), ("ms_fill", C.c_float), ("field_mode", C.c_uint32),
                ("field_blocks", C.c_uint64), ("jit", C.c_uint32), ("ms_compile", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class StepData(C.Structure):
    """mcb_step_data: Step_Data (marching.h:15-23) of one cube, as Marching::calculate_step fills it."""
    _fields_ = [("corner_coords", C.c_float * 24), ("corner_values", C.c_float * 8), ("intersect_coord", C.c_float * 36),
                ("edge_list", C.c_int32 * 12), ("tri_vlist", C.c_int32 * 15), ("n_edges", C.c_int32), ("n_tri_idx", C.c_int32),
                ("cube_code", C.c_int32), ("table_idx", C.c_int32), ("skipped", C.c_int32), ("surf_constant", C.c_float)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError("libmcb200.so is not built: run `python __graft_entry__.py` (or build.py) first — "
                          "there is no fallback implementation")
    L = C.CDLL(LIB_PATH)
    vp, cp, i, f, u64, sz = C.c_void_p, C.c_char_p, C.c_int, C.c_float, C.c_uint64, C.c_size_t
    sigs = {
        "mcb_abi_version": ([], i),
        "mcb_build_stamp": ([], cp),
        "mcb_struct_size": ([i], i),
        "mcb_status_string": ([i], cp),
        "mcb_parse": ([cp], i),
        "mcb_tokens": ([cp, cp, sz], i),
        "mcb_postfix": ([cp, cp, sz], i),
        "mcb_disassemble": ([cp, i, cp, sz], i),
        "mcb_grammar_text": ([cp, i, i, cp, sz], i),
        "mcb_grid_axis": ([f, vp, i], i),
        "mcb_tri_row": ([i], u64),
        "mcb_slab_range": ([i, i, i, C.POINTER(i), C.POINTER(i)], i),
        "mcb_create": ([i, C.POINTER(vp)], i),
        "mcb_destroy": ([vp], None),
        "mcb_last_error": ([vp], cp),
        "mcb_set_stream": ([vp, vp], i),
        "mcb_set_equation": ([vp, i, cp], i),
        "mcb_set_grammar": ([vp, i], i),
        "mcb_eval_points": ([vp, i, vp, vp, sz, i], i),
        "mcb_eval_gradients": ([vp, i, vp, vp, sz, i], i),
        "mcb_set_grid_step": ([vp, f], i),
        "mcb_set_slab": ([vp, i, i], i),
        "mcb_set_surface_constant": ([vp, f], i),
        "mcb_set_scaling": ([vp, f, f, f], i),
        "mcb_set_constraint": ([vp, i, i, f, i], i),
        "mcb_set_normals": ([vp, i], i),
        "mcb_set_refine_vertices": ([vp, i], i),
        "mcb_set_seed": ([vp, i, f, f, f], i),
        "mcb_set_repeat": ([vp, i, f], i),
        "mcb_inspect_cube": ([vp, f, f, f, C.POINTER(StepData)], i),
        "mcb_polygonise": ([vp, C.POINTER(Counts)], i),
        "mcb_get_mesh": ([vp, vp, vp, u64], i),
        "mcb_get_mesh_device": ([vp, C.POINTER(vp), C.POINTER(vp)], i),
        "mcb_counts_device": ([vp, C.POINTER(vp)], i),
        "mcb_set_mesh_mode": ([vp, i], i),
        "mcb_set_field_mode": ([vp, i], i),
        "mcb_set_stage_timing": ([vp, i], i),
        "mcb_set_index_base": ([vp, C.c_uint32], i),
        "mcb_set_jit": ([vp, i], i),
        "mcb_jit_wait": ([vp], i),
        "mcb_jit_check": ([cp, cp, sz], i),
        "mcb_jit_check_grammar": ([cp, i, cp, sz], i),
        "mcb_get_indexed_mesh": ([vp, vp, vp, vp, u64, u64], i),
        "mcb_get_indexed_mesh_device": ([vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)], i),
        "mcb_set_host_output": ([vp, vp, vp, vp, u64, u64], i),
        "mcb_host_output_filled": ([vp], i),
        "mcb_get_cases": ([vp, vp, vp], i),
        "mcb_get_field": ([vp, vp], i),
        "mcb_get_active": ([vp, vp, vp, u64], i),
        "mcb_layer_triangles": ([vp, vp], i),
        "mcb_balance_slabs": ([i, i, vp, C.c_double, vp], i),
        "mcb_comm_unique_id": ([vp], i),
        "mcb_comm_init": ([vp, vp, i, i], i),
        "mcb_comm_exchange": ([vp], i),
        "mcb_comm_set_auto": ([vp, i], i),
        "mcb_comm_offsets": ([vp, C.POINTER(u64), C.POINTER(u64), vp], i),
        "mcb_rebalance_slabs": ([i, i, C.c_void_p, C.c_void_p, C.c_void_p], i),
        "mcb_comm_balance": ([vp, C.c_double, C.POINTER(i), C.POINTER(i)], i),
        "mcb_comm_rebalance": ([vp, C.c_double, C.POINTER(i), C.POINTER(i)], i),
        "mcb_comm_finalize": ([vp], i),
        "mcb_host_register": ([vp, sz], i),
        "mcb_host_unregister": ([vp], i),
    }
    for name, (args, res) in sigs.items():
        fn = getattr(L, name)  # AttributeError here = the library does not export what include/mcb.h declares
        fn.argtypes = args
        fn.restype = res
    return L, sorted(sigs)


lib, EXPORTS = _load()
if lib.mcb_struct_size(0) != C.sizeof(Counts) or lib.mcb_struct_size(1) != C.sizeof(StepData):
    raise ImportError("libmcb200.so and this ctypes mirror disagree on a struct layout: rebuild the library")


def status_string(s):
    return lib.mcb_status_string(int(s)).decode()


def _text(fn, *args, cap=1 << 16):
    buf = C.create_string_buffer(cap)
    rc = fn(*args, buf, cap)
    if rc != MCB_OK:
        raise McbError(rc)
    return buf.value.decode()


def parse_ok(eq, *, grammar=GRAMMAR_REFERENCE):
    """Evaluator::tokenize accept/reject (evaluator.cpp:139-237), or that of the function grammar; host-only."""
    if grammar == GRAMMAR_REFERENCE:
        return lib.mcb_parse(eq.encode()) == MCB_OK
    return lib.mcb_grammar_text(eq.encode(), grammar, -1, None, 0) == MCB_OK


def tokens(eq, *, grammar=GRAMMAR_REFERENCE):
    if grammar == GRAMMAR_REFERENCE:
        return _text(lib.mcb_tokens, eq.encode())
    return _text(lib.mcb_grammar_text, eq.encode(), grammar, 0)


def postfix(eq, *, grammar=GRAMMAR_REFERENCE):
    """Operation order of the reference's two-stack evaluator as postfix text; host-only."""
    if grammar == GRAMMAR_REFERENCE:
        return _text(lib.mcb_postfix, eq.encode())
    return _text(lib.mcb_grammar_text, eq.encode(), grammar, 1)


def disassemble(eq, which=1, *, grammar=GRAMMAR_REFERENCE):
    if grammar == GRAMMAR_REFERENCE:
        return _text(lib.mcb_disassemble, eq.encode(), which)
    return _text(lib.mcb_grammar_text, eq.encode(), grammar, 2 + which)


def jit_check(eq, cap=1 << 18, *, grammar=GRAMMAR_REFERENCE):
    """Host-only: (cubin bytes, generated CUDA source) of the run-time specialised evaluator for `eq`; raises with the log."""
    buf = C.create_string_buffer(cap)
    rc = lib.mcb_jit_check(eq.encode(), buf, cap) if grammar == GRAMMAR_REFERENCE else \
        lib.mcb_jit_check_grammar(eq.encode(), grammar, buf, cap)
    if rc <= 0:
        raise McbError(rc, buf.value.decode(errors="replace"))
    return rc, buf.value.decode(errors="replace")


def grid_axis(step):
    """(M, c[0..M]) of the reference grid loop (marching.cpp:372-377); host-only."""
    M = lib.mcb_grid_axis(step, None, 0)
    if M < 0:
        raise McbError(M)
    c = np.empty(M + 1, np.float32)
    lib.mcb_grid_axis(step, c.ctypes.data_as(C.c_void_p), M + 1)
    return M, c


def slab_range(M, rank, nranks):
    a, b = C.c_int(0), C.c_int(0)
    rc = lib.mcb_slab_range(M, rank, nranks, C.byref(a), C.byref(b))
    if rc != MCB_OK:
        raise McbError(rc)
    return a.value, b.value


def balance_slabs(triangles_per_layer, nranks, fixed_cost_per_layer=-1.0):
    """Host-only: cut points [nranks+1] of contiguous z-slabs of (nearly) equal cost (mcb_balance_slabs)."""
    t = np.ascontiguousarray(triangles_per_layer, np.uint32)
    cuts = np.zeros(nranks + 1, np.int32)
    rc = lib.mcb_balance_slabs(len(t), nranks, t.ctypes.data_as(C.c_void_p), float(fixed_cost_per_layer), cuts.ctypes.data_as(C.c_void_p))
    if rc != MCB_OK:
        raise McbError(rc)
    return [int(x) for x in cuts]


def rebalance_slabs(cost_per_layer, cuts, ms_per_rank):
    """Host-only: one refinement of a cut by measured time (mcb_rebalance_slabs).  Returns (new cost per layer, new cuts)."""
    cost = np.array(cost_per_layer, np.float64)
    c = np.array(cuts, np.int32)
    ms = np.ascontiguousarray(ms_per_rank, np.float64)
    rc = lib.mcb_rebalance_slabs(len(cost), len(ms), cost.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p), ms.ctypes.data_as(C.c_void_p))
    if rc != MCB_OK:
        raise McbError(rc)
    return cost, [int(x) for x in c]


def comm_unique_id():
    """128 bytes of ncclGetUniqueId: made on one rank, handed to the others out of band."""
    buf = C.create_string_buffer(128)
    rc = lib.mcb_comm_unique_id(buf)
    if rc != MCB_OK:
        raise McbError(rc, "mcb_comm_unique_id (is libnccl.so.2 there?)")
    return buf.raw


class Context:
    """One mcb_ctx: the device state of one Marching object / one z-slab on one GPU."""

    def __init__(self, device=0):
        h = C.c_void_p()
        rc = lib.mcb_create(device, C.byref(h))
        if rc != MCB_OK:
            raise McbError(rc, "mcb_create")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            lib.mcb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise McbError(rc, lib.mcb_last_error(self.h).decode())
        return rc

    def set_stream(self, stream_ptr):
        self._ck(lib.mcb_set_stream(self.h, C.c_void_p(stream_ptr)))

    def set_equation(self, eq, slot=0):
        return lib.mcb_set_equation(self.h, slot, eq.encode())

    def set_grammar(self, grammar):
        """GRAMMAR_REFERENCE (default) or GRAMMAR_FUNCTIONS for the set_equation calls that follow, in every slot.
        GRAMMAR_FUNCTIONS adds sin( cos( sqrt( abs( and the two-argument min(a,b) max(a,b) (include/mcb.h)."""
        self._ck(lib.mcb_set_grammar(self.h, grammar))

    def eval_points(self, xyz, slot=0, apply_scale=False):
        xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
        out = np.empty(len(xyz), np.float32)
        self._ck(lib.mcb_eval_points(self.h, slot, xyz.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                     len(xyz), int(apply_scale)))
        return out

    def eval_gradients(self, xyz, slot=0, apply_scale=False):
        """The gradient (df/dx, df/dy, df/dz) of the slot's equation at n points, unnormalised: [n,3] f32.  Forward-mode
        differentiation of the same program eval_points runs (include/mcb.h, mcb_eval_gradients)."""
        xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
        out = np.empty((len(xyz), 3), np.float32)
        self._ck(lib.mcb_eval_gradients(self.h, slot, xyz.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                        len(xyz), int(apply_scale)))
        return out

    def set_grid_step(self, step):
        return lib.mcb_set_grid_step(self.h, step)

    def set_slab(self, k0, k1):
        self._ck(lib.mcb_set_slab(self.h, k0, k1))

    def set_surface_constant(self, iso):
        self._ck(lib.mcb_set_surface_constant(self.h, iso))

    def set_scaling(self, sx, sy, sz):
        self._ck(lib.mcb_set_scaling(self.h, sx, sy, sz))

    def set_constraint(self, i, op, rhs, in_use=True):
        opi = {">": 0, "<": 1, ">=": 2, "<=": 3}[op] if isinstance(op, str) else int(op)
        return lib.mcb_set_constraint(self.h, i, opi, rhs, int(in_use))

    def set_normals(self, mode):
        self._ck(lib.mcb_set_normals(self.h, int(mode)))

    def set_refine_vertices(self, enabled):
        """Refined vertices (include/mcb.h, DESIGN.md §13): every soup and welded vertex moved along its grid edge to where
        the equation reaches the surface constant; indices and counts unchanged.  Off by default."""
        self._ck(lib.mcb_set_refine_vertices(self.h, int(bool(enabled))))

    def inspect_cube(self, x0, y0, z0):
        """Marching::calculate_step(x0, y0, z0) for one cube, on the GPU."""
        sd = StepData()
        self._ck(lib.mcb_inspect_cube(self.h, x0, y0, z0, C.byref(sd)))
        return sd

    def set_repeat(self, enabled, distance=0.0):
        """Repeating-surface mode (marching.cpp:481-494): per-cube iso = highest level iso + n*distance <= the cube's largest corner value."""
        return lib.mcb_set_repeat(self.h, int(bool(enabled)), float(distance))

    def set_seed(self, enabled, x=0.0, y=0.0, z=0.0):
        """Seed mode: keep only the component of the cube containing (x,y,z). Returns the status (MCB_E_ARG outside [-1,1]^3)."""
        return lib.mcb_set_seed(self.h, int(bool(enabled)), x, y, z)

    def counts_device_ptr(self):
        """Device address of the live counters (5 x uint64: active, triangles, ambiguous, redirected, vertices)."""
        p = C.c_void_p()
        self._ck(lib.mcb_counts_device(self.h, C.byref(p)))
        return p.value

    def set_jit(self, mode):
        """JIT_AUTO (default) / JIT_ON / JIT_OFF: evaluate the field with a kernel NVRTC compiles for the equation
        (bit-identical to the interpreter; compiled on first use, cached per equation)."""
        self._ck(lib.mcb_set_jit(self.h, int(mode)))

    def set_index_base(self, base):
        """added on the device to every index get_indexed_mesh delivers (slab r of a mesh assembled from several slabs)"""
        self._ck(lib.mcb_set_index_base(self.h, int(base)))

    def jit_wait(self):
        """block until the background compile of the current equation is over; True when the compiled kernels will run"""
        rc = lib.mcb_jit_wait(self.h)
        if rc < 0:
            self._ck(rc)
        return rc == 1

    def set_field_mode(self, mode):
        """FIELD_DENSE (whole field in device memory) or FIELD_SPARSE (signs everywhere, values only around the surface)."""
        self._ck(lib.mcb_set_field_mode(self.h, int(mode)))

    def set_stage_timing(self, enabled):
        """CUDA events around the stages (Counts.ms_*): on by default; off shortens the gaps between the short kernels."""
        self._ck(lib.mcb_set_stage_timing(self.h, int(bool(enabled))))

    def set_mesh_mode(self, mode):
        """MESH_SOUP (float4 triangle soup), MESH_INDEXED (welded Poly_Data layout), both (3), or MESH_DC alone (the
        dual-contoured mesh in the indexed layout, read with get_indexed_mesh)."""
        self._ck(lib.mcb_set_mesh_mode(self.h, int(mode)))

    def get_indexed_mesh(self, normals=False):
        """(vertex_list[V,3] f32, tri_list[T,3] u32[, normals[V,3] f32]) as Marching::recalculate leaves them in Poly_Data."""
        V, T = int(self.counts.vertices), int(self.counts.triangles)
        vl = np.empty((V, 3), np.float32)
        tl = np.empty((T, 3), np.uint32)
        vn = np.empty((V, 3), np.float32) if normals else None
        self._ck(lib.mcb_get_indexed_mesh(self.h, vl.ctypes.data_as(C.c_void_p), tl.ctypes.data_as(C.c_void_p),
                                          vn.ctypes.data_as(C.c_void_p) if normals else None, V, T))
        return (vl, tl, vn) if normals else (vl, tl)

    def set_host_output(self, v_ptr, t_ptr, n_ptr, cap_v, cap_t):
        """Register (pinned) host buffers: polygonise() in MESH_INDEXED mode then streams the mesh into them."""
        self._ck(lib.mcb_set_host_output(self.h, C.c_void_p(v_ptr) if v_ptr else None, C.c_void_p(t_ptr) if t_ptr else None,
                                         C.c_void_p(n_ptr) if n_ptr else None, cap_v, cap_t))

    def host_output_filled(self):
        return bool(lib.mcb_host_output_filled(self.h))

    def get_indexed_mesh_into(self, v_ptr, t_ptr, n_ptr, cap_v, cap_t):
        """Raw-pointer variant (pinned host buffers owned by the caller)."""
        self._ck(lib.mcb_get_indexed_mesh(self.h, C.c_void_p(v_ptr) if v_ptr else None, C.c_void_p(t_ptr) if t_ptr else None,
                                          C.c_void_p(n_ptr) if n_ptr else None, cap_v, cap_t))

    def polygonise(self):
        c = Counts()
        self._ck(lib.mcb_polygonise(self.h, C.byref(c)))
        self.counts = c
        return c

    def get_mesh(self, normals=True, out_pos=None, out_nrm=None):
        """Triangle soup on the host: pos[T,3,4] (x,y,z,1) and nrm[T,3,4] (nx,ny,nz,0)."""
        T = int(self.counts.triangles)
        pos = out_pos if out_pos is not None else np.empty((T, 3, 4), np.float32)
        nrm = (out_nrm if out_nrm is not None else np.empty((T, 3, 4), np.float32)) if normals else None
        self._ck(lib.mcb_get_mesh(self.h, pos.ctypes.data_as(C.c_void_p),
                                  nrm.ctypes.data_as(C.c_void_p) if nrm is not None else None, pos.shape[0]))
        return pos[:T], (nrm[:T] if nrm is not None else None)

    def get_mesh_into(self, pos_ptr, nrm_ptr, cap_tris):
        """Raw-pointer variant (pinned host buffers owned by the caller)."""
        self._ck(lib.mcb_get_mesh(self.h, C.c_void_p(pos_ptr), C.c_void_p(nrm_ptr) if nrm_ptr else None, cap_tris))

    def get_cases(self):
        n = int(self.counts.cubes)
        code = np.empty(n, np.uint8)
        tidx = np.empty(n, np.uint8)
        self._ck(lib.mcb_get_cases(self.h, code.ctypes.data_as(C.c_void_p), tidx.ctypes.data_as(C.c_void_p)))
        return code, tidx

    def get_field(self):
        c = self.counts
        n1 = c.M + 1
        out = np.empty((c.k_end - c.k_begin + 1, n1, n1), np.float32)
        self._ck(lib.mcb_get_field(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def layer_triangles(self):
        """Triangles per cube layer of this slab in the last polygonisation (uint32[k_end - k_begin])."""
        c = self.counts
        out = np.zeros(c.k_end - c.k_begin, np.uint32)
        self._ck(lib.mcb_layer_triangles(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    # ---- z-slabs over several GPUs: the NCCL exchange behind the C ABI (mcb_comm_*) ----
    def comm_init(self, id128, rank, nranks):
        self._ck(lib.mcb_comm_init(self.h, C.c_char_p(id128), rank, nranks))

    def comm_exchange(self):
        self._ck(lib.mcb_comm_exchange(self.h))

    def comm_set_auto(self, enabled):
        """polygonise() enqueues the all-gather itself as soon as the slab's triangle count is final"""
        self._ck(lib.mcb_comm_set_auto(self.h, int(bool(enabled))))

    def comm_offsets(self, nranks):
        off, tot = C.c_uint64(0), C.c_uint64(0)
        per = np.zeros(nranks, np.uint64)
        self._ck(lib.mcb_comm_offsets(self.h, C.byref(off), C.byref(tot), per.ctypes.data_as(C.c_void_p)))
        return int(off.value), int(tot.value), [int(x) for x in per]

    def comm_balance(self, fixed_cost_per_layer=-1.0):
        a, b = C.c_int(0), C.c_int(0)
        self._ck(lib.mcb_comm_balance(self.h, float(fixed_cost_per_layer), C.byref(a), C.byref(b)))
        return a.value, b.value

    def comm_rebalance(self, ms_measured):
        """refine the balanced cut with the time this rank's slab was measured to take (collective)"""
        a, b = C.c_int(0), C.c_int(0)
        self._ck(lib.mcb_comm_rebalance(self.h, float(ms_measured), C.byref(a), C.byref(b)))
        return a.value, b.value

    def get_active(self):
        A = int(self.counts.active)
        rec = np.empty(A, np.uint64)
        off = np.empty(A, np.uint32)
        self._ck(lib.mcb_get_active(self.h, rec.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), A))
        return rec, off


class Evaluator:
    """Mirror of the reference's class Evaluator (evaluator.h:55-64).  Evaluation runs on the GPU."""

    def __init__(self, equation=None, device=0):
        self._ctx = Context(device)  # a fresh context already holds the default "x+y" (evaluator.cpp:6-8)
        self.equation = "x+y"
        self.function_grammar = False
        if equation is not None and not self.set_equation(equation):
            raise ValueError("parse error")  # Evaluator(string) throws on a parse error (evaluator.cpp:10-13)

    def set_function_grammar(self, on):
        """Extension: accept sin( cos( sqrt( abs( min( max( in later set_equation calls (GRAMMAR_FUNCTIONS); off by default."""
        self.function_grammar = bool(on)
        self._ctx.set_grammar(GRAMMAR_FUNCTIONS if on else GRAMMAR_REFERENCE)

    def set_equation(self, s):
        ok = self._ctx.set_equation(s) == MCB_OK
        if ok:
            self.equation = s.replace(" ", "")
        return ok

    def evaluate(self, x, y, z):
        return float(self._ctx.eval_points(np.array([[x, y, z]], np.float32))[0])


class PolyData:
    """Poly_Data (marching.h:26-30): vertex_list (xyz per welded vertex) and tri_list (3 indices per triangle), as
    Marching::recalculate() leaves them — welded and numbered on the GPU like add_step_to_poly_data (marching.cpp:599-654).
    vertex_normals = gradient normal per welded vertex (None when normals are off)."""

    def __init__(self, vertex_list, tri_list, vertex_normals=None):
        self._v, self._t, self.vertex_normals = vertex_list, tri_list, vertex_normals

    @property
    def vertex_list(self):
        return self._v.reshape(-1)

    @property
    def tri_list(self):
        return self._t.reshape(-1)


class Marching:
    """Mirror of the reference's class Marching (marching.h:75-122) for the full-grid path."""

    def __init__(self, device=0):
        self._ctx = Context(device)
        self._step = 0.25
        self._eval = None
        self._poly = PolyData(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32))
        self._normals = True
        self._ctx.set_mesh_mode(MESH_INDEXED)
        self._ctx.set_field_mode(FIELD_AUTO)  # like include/marching.h: this class never reads the field back
        self.counts = None

    def set_evaluator(self, e):
        if e is None:
            return False
        self._eval = e
        return True

    def set_grid_step_size(self, v):
        if not (np.float32(v) >= np.float32(0.001) and v <= 0.5):  # marching.cpp:227
            return False
        self._step = float(v)
        return self._ctx.set_grid_step(v) > 0

    def set_grid_resolution(self, n):
        """Extension (SURVEY.md D4): step 2/n, also below the reference's 0.001 floor (2048^3)."""
        self._step = 2.0 / n
        return self._ctx.set_grid_step(self._step) > 0

    def get_grid_size(self):
        return self._step

    def set_surface_constant(self, c):
        self._ctx.set_surface_constant(c)

    def set_scaling_x(self, s):
        self._scale = getattr(self, "_scale", [1.0, 1.0, 1.0]); self._scale[0] = s; self._ctx.set_scaling(*self._scale)

    def set_scaling_y(self, s):
        self._scale = getattr(self, "_scale", [1.0, 1.0, 1.0]); self._scale[1] = s; self._ctx.set_scaling(*self._scale)

    def set_scaling_z(self, s):
        self._scale = getattr(self, "_scale", [1.0, 1.0, 1.0]); self._scale[2] = s; self._ctx.set_scaling(*self._scale)

    def set_constraint(self, i, lhs, op, rhs):
        if i < 0 or i > 2 or op not in (">", "<", ">=", "<="):
            return False
        # the left-hand side parses in the grammar of the evaluator set at this time (as include/marching.h)
        self._ctx.set_grammar(GRAMMAR_FUNCTIONS if getattr(self._eval, "function_grammar", False) else GRAMMAR_REFERENCE)
        if self._ctx.set_equation(lhs, slot=i + 1) != MCB_OK:
            return False
        self._cons = getattr(self, "_cons", {})
        self._cons[i] = (op, rhs, self._cons.get(i, (None, None, False))[2])
        return self._ctx.set_constraint(i, op, rhs, self._cons[i][2]) == MCB_OK

    def use_constraint(self, i, use):
        c = getattr(self, "_cons", {}).get(i)
        if c is None:
            return False
        self._cons[i] = (c[0], c[1], bool(use))
        return self._ctx.set_constraint(i, c[0], c[1], bool(use)) == MCB_OK and bool(use)

    def set_slab(self, k0, k1):
        self._ctx.set_slab(k0, k1)

    def set_surface_repeat_step_distance(self, l):  # marching.cpp:156-162
        if l <= 0:
            return False
        self._repeat_step = float(l)
        return self._ctx.set_repeat(getattr(self, "_repeat_on", False), self._repeat_step) == MCB_OK

    def repeating_surface_mode(self, b):  # marching.cpp:164-170; a positive distance must have been set (the reference's 0 draws nothing)
        self._repeat_on = bool(b)
        return self._ctx.set_repeat(self._repeat_on and getattr(self, "_repeat_step", 0.0) > 0, getattr(self, "_repeat_step", 0.0)) == MCB_OK

    def seed_mode(self, b):
        self._seed_on = bool(b)
        s = getattr(self, "_seed", (0.0, 0.0, 0.0))
        self._ctx.set_seed(self._seed_on, *s)

    def set_seed(self, x, y, z):
        if not (-1 <= x <= 1 and -1 <= y <= 1 and -1 <= z <= 1):  # marching.cpp:128-137
            return False
        self._seed = (x, y, z)
        self._ctx.set_seed(getattr(self, "_seed_on", False), x, y, z)
        return True

    def set_normals(self, mode):
        self._normals = bool(mode)
        self._ctx.set_normals(mode)

    def set_refined_vertices(self, b):
        """Extension: include/marching.h Marching::set_refined_vertices (Context.set_refine_vertices)."""
        self._ctx.set_refine_vertices(b)

    def set_dual_contouring(self, b):
        """Extension: include/marching.h Marching::set_dual_contouring — Poly_Data holds the dual-contoured mesh (MESH_DC)."""
        self._ctx.set_mesh_mode(MESH_DC if b else MESH_INDEXED)

    def recalculate(self, fetch=True):
        if self._eval is None:
            return False  # the reference evaluates to 0 everywhere without an evaluator: an empty mesh
        self._ctx.set_grammar(GRAMMAR_FUNCTIONS if getattr(self._eval, "function_grammar", False) else GRAMMAR_REFERENCE)
        if self._ctx.set_equation(self._eval.equation) != MCB_OK:
            return False
        self.counts = self._ctx.polygonise()
        if fetch:
            self._poly = PolyData(*self._ctx.get_indexed_mesh(normals=self._normals))
        return True

    def get_poly_data(self):
        return self._poly
