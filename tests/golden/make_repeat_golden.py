"""Generates tests/golden/repeat_cases.npz from the UNMODIFIED reference in repeating-surface mode
(Marching::set_surface_repeat_step_distance + repeating_surface_mode(true) + recalculate(), marching.cpp:156-170,
481-494) through oracle/_ref.  Run in the build container only.
Per case: Poly_Data (vertex_list, tri_list) of recalculate(), normal.h normals, and the per-cube sweep through the
private calculate_step (cube_code against the cube's own surf_constant, tri_table row, triangle count, soup)."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refbind as R  # noqa: E402
from tests.helpers import save_repeat_golden  # noqa: E402

CASES = {
    # marching_test_drawer.h:238 uses distance 1.5; smaller distances give several nested shells
    "rep_sphere_20": dict(eq=R.SPHERE, step=2.0 / 20, scale=1.0, iso=0.0, dist=0.25),
    "rep_sphere_iso": dict(eq=R.SPHERE, step=2.0 / 18, scale=1.1, iso=0.07, dist=0.3),
    "rep_eq1_ctor": dict(eq=R.EXAMPLE_EQUATIONS[1], step=0.25, scale=1.0, iso=0.0, dist=0.5),      # planes through grid corners
    "rep_eq1_gui": dict(eq=R.EXAMPLE_EQUATIONS[1], step=0.2, scale=1.1, iso=0.0, dist=0.37),
    "rep_torus_24": dict(eq=R.TORUS, step=2.0 / 24, scale=1.0, iso=0.0, dist=0.08),
    "rep_eq8_gui": dict(eq=R.EXAMPLE_EQUATIONS[8], step=0.2, scale=1.1, iso=0.0, dist=0.02),
    "rep_gyr78_17": dict(eq=R.GYR78, step=2.0 / 17, scale=1.0, iso=0.0, dist=0.4),                  # ambiguous cubes, non-dyadic step
    "rep_quirk_div": dict(eq="x/y-z", step=2.0 / 16, scale=1.0, iso=0.0, dist=0.75),               # inf / NaN corner values
    "rep_testdrawer": dict(eq=R.SPHERE, step=0.25, scale=1.0, iso=0.0, dist=1.5),                    # the test drawer's own setting
    "rep_cons": dict(eq=R.SPHERE, step=2.0 / 18, scale=1.0, iso=0.0, dist=0.2, cons=[("x+y", "<", 0.3)]),
}
out, meta = {}, {}
for name, c in CASES.items():
    r = R.Ref(c["eq"], c["step"], scale=(c["scale"],) * 3, iso=c["iso"])
    for i, (lhs, op, rhs) in enumerate(c.get("cons", [])):
        assert r.set_constraint(i, lhs, op, rhs, True)
    assert r.set_repeat(True, c["dist"])
    v, t = r.recalculate()
    n = r.normals()
    sw = r.sweep(soup=True)
    assert sw["T"] == len(t), (name, sw["T"], len(t))
    out[name + "/vertex_list"] = v
    out[name + "/tri_list"] = t
    out[name + "/normals"] = n
    out[name + "/code"] = sw["code"]
    out[name + "/table_idx"] = sw["table_idx"]
    out[name + "/ntri"] = sw["ntri"]
    out[name + "/soup"] = sw["soup"]
    meta[name] = dict(eq=c["eq"], step=c["step"], scale=[c["scale"]] * 3, iso=c["iso"], dist=c["dist"], cons=c.get("cons", []),
                      M=int(sw["M"]), T=int(len(t)), V=int(len(v)), active=int(sw["active"]), ambiguous=int(sw["ambiguous"]),
                      redirected=int(sw["redirected"]))
    print(name, meta[name]["M"], "M", meta[name]["V"], "vertices", meta[name]["T"], "triangles", meta[name]["active"], "active",
          meta[name]["ambiguous"], "ambiguous")
out["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
save_repeat_golden(os.path.join(ROOT, "tests", "golden", "repeat_cases.npz"), out)
