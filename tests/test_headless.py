"""mcb_headless — the reference's main.cpp wiring without the GUI (tools/headless_main.cpp, built on the C++ drop-in
headers): equation file in, counts out, mesh dumped as the reference's ASCII PLY and as a lossless binary."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from .helpers import load_meta, load_repeat_golden, same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "mcb_headless")


def test_headless_is_built_and_fails_loudly_without_a_device(mcb):
    assert os.path.exists(EXE)
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([EXE, "--eq", "x+y"], capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stderr
    assert subprocess.run([EXE, "--eq", "(x(y)"], capture_output=True, text=True).returncode == 1  # parse errors need no GPU


@pytest.mark.gpu
def test_headless_config0_default_resolution_mesh_dump(mcb, golden, tmp_path):
    """BASELINE.json configs[0]: example_files/equation_N.txt at the reference's default grid (0.2, scale 1.1), headless,
    mesh dumped for diff — here diffed against the unmodified reference's Poly_Data."""
    meta = load_meta(golden)
    for n in (1, 3, 8):
        case = meta["eq%d_gui" % n]
        eqf = tmp_path / ("equation_%d.txt" % n)
        eqf.write_text(case["eq"])  # one line, the format of example_files/ (evaluator.cpp:285-300)
        ply, dump = tmp_path / "m.ply", tmp_path / "m.bin"
        out = subprocess.check_output([EXE, "--eq-file", str(eqf), "--ply", str(ply), "--dump", str(dump)], text=True)
        info = json.loads(out.strip().splitlines()[-1])
        vref = golden["eq%d_gui/vertex_list" % n].reshape(-1, 3)
        tref = golden["eq%d_gui/tri_list" % n].reshape(-1, 3)
        assert (info["M"], info["vertices"], info["triangles"]) == (11, len(vref), len(tref))
        raw = dump.read_bytes()
        nv, nt = struct.unpack("<QQ", raw[:16])
        v = np.frombuffer(raw, np.float32, nv * 3, 16).reshape(-1, 3)
        t = np.frombuffer(raw, np.uint32, nt * 3, 16 + nv * 12).reshape(-1, 3)
        assert same_bits(v, vref) and np.array_equal(t, tref)
        # the ASCII PLY of marching.cpp:821-850: "element face %d " keeps its trailing blank, coordinates are %f
        lines = ply.read_text().splitlines()
        assert lines[:3] == ["ply", "format ascii 1.0", "element vertex %d" % nv] and lines[6] == "element face %d " % nt
        body = lines[lines.index("end_header") + 1:]
        pv = np.array([[float(x) for x in l.split()] for l in body[:nv]])
        pt = np.array([[int(x) for x in l.split()] for l in body[nv:nv + nt]])
        assert np.allclose(pv, v, atol=5.1e-7) and np.array_equal(pt[:, 1:], t) and np.all(pt[:, 0] == 3)


@pytest.mark.gpu
def test_headless_finer_than_the_reference_allows(mcb, tmp_path):
    r = subprocess.run([EXE, "--eq", "x^2+y^2+z^2-0.49", "--step", "0.0005"], capture_output=True, text=True)
    assert r.returncode == 1  # set_grid_step_size rejects < 0.001 (marching.cpp:227)
    out = subprocess.check_output([EXE, "--eq", "x^2+y^2+z^2-0.49", "--res", "256", "--scale", "1", "1", "1"], text=True)
    info = json.loads(out.strip().splitlines()[-1])
    assert (info["M"], info["vertices"], info["triangles"]) == (257, 151398, 302792)


@pytest.mark.gpu
def test_headless_repeating_surface_mode(mcb, tmp_path):
    """The drop-in class in repeating-surface mode (set_surface_repeat_step_distance + repeating_surface_mode, the setting of
    the reference's own test drawer, marching_test_drawer.h:238) against the unmodified reference's Poly_Data."""
    rep = load_repeat_golden(os.path.join(ROOT, "tests", "golden", "repeat_cases.npz"))
    case = json.loads(bytes(rep["meta_json"]).decode())["rep_testdrawer"]
    dump = tmp_path / "m.bin"
    out = subprocess.check_output([EXE, "--eq", case["eq"], "--step", str(case["step"]), "--scale", "1", "1", "1", "--levels", str(case["dist"]),
                                   "--dump", str(dump)], text=True)
    info = json.loads(out.strip().splitlines()[-1])
    assert (info["M"], info["vertices"], info["triangles"]) == (case["M"], case["V"], case["T"])
    raw = dump.read_bytes()
    nv, nt = struct.unpack("<QQ", raw[:16])
    v = np.frombuffer(raw, np.float32, nv * 3, 16).reshape(-1, 3)
    t = np.frombuffer(raw, np.uint32, nt * 3, 16 + nv * 12).reshape(-1, 3)
    assert same_bits(v, rep["rep_testdrawer/vertex_list"]) and np.array_equal(t, rep["rep_testdrawer/tri_list"])
    assert subprocess.run([EXE, "--levels", "0"], capture_output=True).returncode == 1


@pytest.mark.gpu
def test_headless_repeated_recalculate_switches_to_the_sparse_field_and_keeps_the_mesh(mcb, tmp_path):
    """The drop-in class uses MCB_FIELD_AUTO: the first recalculate() of a configuration writes the whole field, the
    following ones only its signs (sphere at 640^3: 0.36 % active cubes).  The Poly_Data must not notice."""
    dumps = []
    for rep in (1, 3):
        dump = tmp_path / ("m%d.bin" % rep)
        out = subprocess.check_output([EXE, "--eq", "x^2+y^2+z^2-0.49", "--res", "640", "--scale", "1", "1", "1", "--repeat", str(rep),
                                       "--dump", str(dump)], text=True)
        info = json.loads(out.strip().splitlines()[-1])
        assert info["M"] == 641 and info["triangles"] > 1000000
        dumps.append(dump.read_bytes())
    assert dumps[0] == dumps[1]
