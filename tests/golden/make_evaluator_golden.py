"""Writes tests/golden/evaluator_mesh_hashes.json: the digests of tests/test_evaluator.py's meshes (mesh_digests) as a given
build of the package computes them.  The committed file was written on a B200 by the build of the commit before the
operator table (csrc/mcb_bytecode.h), so that test_meshes_equal_the_build_before_the_operator_table pins every later
build to that one's bytes.

    python tests/golden/make_evaluator_golden.py [repository root whose package to load; default this one]"""
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.test_evaluator import HASHES, MESH_CASES, mesh_digests  # noqa: E402

src = sys.argv[1] if len(sys.argv) > 1 else ROOT
pkg = os.path.join(src, "marching-cube-for-implicit-surfaces_b200", "__init__.py")
spec = importlib.util.spec_from_file_location("mcb_golden_build", pkg)
mcb = importlib.util.module_from_spec(spec)
spec.loader.exec_module(mcb)
out = {name: mesh_digests(mcb, name) for name in sorted(MESH_CASES)}
with open(HASHES, "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
print(json.dumps(out, indent=1, sort_keys=True))
