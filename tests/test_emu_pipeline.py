"""-m "not gpu": the product's DEVICE CODE executed on the host (tests/emu: csrc/mcb_api.cu + mcb_kernels.cuh compiled by g++
against an emulated CUDA runtime, every CUDA thread a fiber) through the same C ABI and ctypes mirror the GPU tests use.

This is test infrastructure for the build container, which has no GPU: kernel logic (tiling, scans, ballots, the block
skipping of the block-field mode, the ambiguity list, the weld) is checked here against the golden vectors of the
unmodified reference at small sizes; the -m gpu tier repeats it, and everything at size, on the real device through
libmcb200.so.  The product never loads the emulated library."""
import numpy as np
import pytest

from .helpers import configure, load_meta, same_bits

CASES = ["eq1_gui", "eq8_ctor", "sphere_17", "gyr78_17", "constraint_2", "quirk_div", "saddle_17", "torus_33", "sphere_33_iso", "nonuniform_scale"]


@pytest.fixture(scope="module")
def ctx(mcb_emu):
    c = mcb_emu.Context(0)
    c.set_mesh_mode(mcb_emu.MESH_SOUP | mcb_emu.MESH_INDEXED)
    yield c
    c.close()


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("mode", ["dense", "blocks"])
def test_golden_cases_through_the_emulated_kernels(mcb_emu, ctx, golden, name, mode):
    case = load_meta(golden)[name]
    configure(ctx, case)
    ctx.set_field_mode(mcb_emu.FIELD_DENSE if mode == "dense" else mcb_emu.FIELD_AUTO)
    ctx.set_normals(2)
    cnt = ctx.polygonise()
    assert cnt.field_mode == (mcb_emu.FIELD_DENSE if mode == "dense" else mcb_emu.FIELD_SPARSE)
    code, tidx = ctx.get_cases()
    pos, _ = ctx.get_mesh(normals=False)
    vl, tl, vn = ctx.get_indexed_mesh(normals=True)
    assert np.array_equal(code, golden[name + "/code"]) and np.array_equal(tidx, golden[name + "/table_idx"])
    assert cnt.triangles == case["T"]
    assert same_bits(pos[:, :, :3], golden[name + "/soup"])
    assert same_bits(vl, golden[name + "/vertex_list"].reshape(-1, 3)) and np.array_equal(tl, golden[name + "/tri_list"].reshape(-1, 3))
    assert same_bits(vn, golden[name + "/normals"].reshape(-1, 3))


GYR78 = ("((x*(-7+x^2*(56+x^2*(-112+64*x^2))))*(1+y^2*(-32+y^2*(160+y^2*(-256+128*y^2)))))"
         "+((y*(-7+y^2*(56+y^2*(-112+64*y^2))))*(1+z^2*(-32+z^2*(160+z^2*(-256+128*z^2)))))"
         "+((z*(-7+z^2*(56+z^2*(-112+64*z^2))))*(1+x^2*(-32+x^2*(160+x^2*(-256+128*x^2)))))")


@pytest.mark.parametrize("eq,n,expect", [("x^2+y^2+z^2-0.49", 64, None), (GYR78, 64, (155478, 338, 163))])
def test_block_mode_skips_space_and_equals_dense_at_65_cubed(mcb_emu, ctx, eq, n, expect):
    """large enough for whole 32 x 4 x 4 blocks to be proven empty and skipped; slab with a halo on both sides too.
    gyr78 at M = 65: triangle / ambiguous / redirected counts of the unmodified reference (SURVEY.md §8d cfg 4)."""
    res = {}
    for mode in (mcb_emu.FIELD_DENSE, mcb_emu.FIELD_AUTO):
        for slab in (None, (7, 22)):
            assert ctx.set_equation(eq) == 0
            M = ctx.set_grid_step(2.0 / n)
            ctx.set_scaling(1, 1, 1); ctx.set_surface_constant(0.0)
            for i in range(3):
                ctx.set_constraint(i, ">", 0.0, False)
            if slab:
                ctx.set_slab(*slab)
            ctx.set_field_mode(mode)
            ctx.set_normals(1)
            cnt = ctx.polygonise()
            res[(mode, slab)] = (cnt, ctx.get_active(), ctx.get_mesh(normals=True), ctx.get_indexed_mesh(normals=True))
    for slab in (None, (7, 22)):
        (cd, rd, md, idd), (cb, rb, mb, ib) = res[(mcb_emu.FIELD_DENSE, slab)], res[(mcb_emu.FIELD_AUTO, slab)]
        assert (cd.active, cd.triangles, cd.ambiguous, cd.redirected, cd.vertices) == (cb.active, cb.triangles, cb.ambiguous, cb.redirected, cb.vertices)
        assert np.array_equal(rd[0], rb[0]) and np.array_equal(rd[1], rb[1])
        assert same_bits(md[0], mb[0]) and same_bits(md[1], mb[1])
        assert same_bits(idd[0], ib[0]) and np.array_equal(idd[1], ib[1]) and same_bits(idd[2], ib[2])
    full = res[(mcb_emu.FIELD_AUTO, None)][0]
    nblocks = ((full.M + 3 + 31) // 32) * ((full.M + 3 + 3) // 4) ** 2
    assert 0 < full.field_blocks <= nblocks
    if expect is None:
        assert full.field_blocks < 0.5 * nblocks   # the sphere leaves most blocks decided, i.e. skipped
    if expect:
        assert (full.triangles, full.ambiguous, full.redirected) == expect


def test_cpp_dropin_class_over_the_emulated_library(golden, tmp_path, mcb_emu):
    """include/marching.h + include/evaluator.h (the reference-facing classes) linked against the emulated library: one
    Marching object polygonises the golden cases one after the other — growing, shrinking and repeated meshes, i.e. both
    the streamed path into the page-locked Poly_Data vectors and the plain copy — and Poly_Data equals the unmodified
    reference's byte for byte (FNV-1a-64 of vertex_list / tri_list)."""
    import os
    import subprocess
    from .test_cpp_dropin import ROOT, fnv1a64
    from . import emu
    lib_dir = os.path.join(ROOT, "tests", "emu", "_build")
    exe = str(tmp_path / "dropin_emu")
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "dropin_main.cpp"), "-o", exe, "-L", lib_dir, "-lmcb200_emu",
                           "-Wl,-rpath," + lib_dir, "-pthread"])
    meta = load_meta(golden)
    names = ["sphere_17", "eq1_gui", "gyr78_17", "gyr78_17", "eq8_ctor", "torus_33", "sphere_17", "sphere_33_iso", "sphere_33_iso"]
    args = []
    for n in names:
        c = meta[n]
        args += [n, c["eq"], repr(c["step"]), repr(c["scale"][0]), repr(c["scale"][1]), repr(c["scale"][2]), repr(c["iso"])]
    out = subprocess.check_output([exe] + args, text=True)
    got = [l.split() for l in out.strip().splitlines()]
    for n, line in zip(names, got):
        v, t = golden[n + "/vertex_list"], golden[n + "/tri_list"]
        assert line[0] == n and line[1:3] == [str(len(v)), str(len(t))], (n, line)
        assert line[3] == fnv1a64(v.tobytes()) and line[4] == fnv1a64(t.tobytes()), n


def test_layer_histogram_and_balanced_cut(mcb_emu, ctx, golden):
    """mcb_layer_triangles (layer_hist_kernel) against the reference's per-cube triangle counts, whole grid and a slab; the
    cut mcb_balance_slabs makes from it gives every rank nearly the same number of triangles"""
    case = load_meta(golden)["sphere_33_iso"]
    configure(ctx, case)
    ctx.set_field_mode(mcb_emu.FIELD_AUTO)
    ctx.set_normals(1)
    M = case["M"]
    want = golden["sphere_33_iso/ntri"].reshape(M, M, M).astype(np.int64).sum(axis=(1, 2))
    ctx.polygonise()
    assert np.array_equal(ctx.layer_triangles().astype(np.int64), want)
    ctx.set_slab(9, 21)
    ctx.polygonise()
    assert np.array_equal(ctx.layer_triangles().astype(np.int64), want[9:21])
    cuts = mcb_emu.balance_slabs(want.astype(np.uint32), 4, 1.0)
    per = [int(want[a:b].sum()) for a, b in zip(cuts, cuts[1:])]
    assert sum(per) == case["T"] and max(per) - min(per) <= 2 * int(want.max())
    uniform = [int(want[(M * r) // 4:(M * (r + 1)) // 4].sum()) for r in range(4)]
    assert max(per) < max(uniform)


@pytest.mark.parametrize("name", ["sphere_17", "gyr78_17", "quirk_div", "nonuniform_scale"])
def test_index_base_shifts_the_tri_list_through_the_emulated_kernels(mcb_emu, golden, name):
    """mcb_set_index_base: the tri_list of the whole grid and of a slab shifted on the device (add_index_base_kernel) and
    shifted back, the vertices untouched."""
    case = load_meta(golden)[name]
    c = mcb_emu.Context(0)
    c.set_mesh_mode(mcb_emu.MESH_SOUP | mcb_emu.MESH_INDEXED)
    configure(c, case)
    for i in range(3):
        c.set_constraint(i, ">", 0.0, False)
    c.set_normals(1)
    for slab in (None, (case["M"] // 3, 2 * case["M"] // 3 + 1)):
        if slab:
            c.set_slab(*slab)
        assert c.polygonise().triangles > 0
        v0, t0 = c.get_indexed_mesh()
        c.set_index_base(123456)
        v1, t1 = c.get_indexed_mesh()
        assert np.array_equal(t1.astype(np.int64), t0.astype(np.int64) + 123456) and same_bits(v0, v1)
        c.set_index_base(0)
        v2, t2 = c.get_indexed_mesh()
        assert np.array_equal(t2, t0) and same_bits(v0, v2)
    c.close()
