"""Combined shapes at 1024^3 (min( max( of MCB_GRAMMAR_FUNCTIONS): a union of 8 spheres (nested min), a lens (max), a sphere
minus a cylinder (max(a,-b)), a box SDF whose max terms are all axis tables, and the plain sphere beside them.  One JSON
line: per workload the counts, the per-stage device times (mean over the timed calls), field_blocks and jit, plus the
device name and power limit read in the same run.

    python tools/bench_csg.py [--res 1024] [--steps 20] [--warmup 3] [--field auto|dense] [--jit auto|off]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# the shapes of tests/csg_common.py (CSG_*); spheres of radius 0.3 at the corners (+-0.4, +-0.4, +-0.4)
UNION8 = ("min(min(min((x+.4)^2+(y+.4)^2+(z+.4)^2-.09,(x-.4)^2+(y+.4)^2+(z+.4)^2-.09),"
          "min((x+.4)^2+(y-.4)^2+(z+.4)^2-.09,(x-.4)^2+(y-.4)^2+(z+.4)^2-.09)),"
          "min(min((x+.4)^2+(y+.4)^2+(z-.4)^2-.09,(x-.4)^2+(y+.4)^2+(z-.4)^2-.09),"
          "min((x+.4)^2+(y-.4)^2+(z-.4)^2-.09,(x-.4)^2+(y-.4)^2+(z-.4)^2-.09)))")
WORKLOADS = [
    ("union8_spheres", 1, UNION8),
    ("lens", 1, "max(sqrt((x-0.3)^2+y^2+z^2)-0.6,sqrt((x+0.3)^2+y^2+z^2)-0.6)"),
    ("sphere_minus_cylinder", 1, "max(sqrt(x^2+y^2+z^2)-0.7,-(sqrt(x^2+y^2)-0.3))"),
    ("box_sdf", 1, "sqrt(max(abs(x)-0.5,0)^2+max(abs(y)-0.4,0)^2+max(abs(z)-0.3,0)^2)-0.1"),
    ("sphere", 0, "x^2+y^2+z^2-0.49"),
]
STAGES = ("ms_tables", "ms_eval", "ms_fill", "ms_classify", "ms_emit", "ms_weld", "ms_total")


def device_info(index=0):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return name, limit
    except Exception as e:  # the numbers are still reported; the line says what could not be read
        return None, "unavailable (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--field", choices=("auto", "dense"), default="auto")
    ap.add_argument("--jit", choices=("auto", "off"), default="auto")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_csg.py measures the GPU path: no CUDA device")
    mcb = importlib.import_module("marching-cube-for-implicit-surfaces_b200")
    name, limit = device_info(0)
    res = {"tool": "bench_csg", "res": a.res, "steps": a.steps, "warmup": a.warmup, "field": a.field, "jit_mode": a.jit,
           "device": name or torch.cuda.get_device_name(0), "power_limit": limit, "workloads": {}}
    for wname, grammar, eq in WORKLOADS:
        c = mcb.Context(0)
        try:
            c.set_mesh_mode(mcb.MESH_SOUP)
            c.set_normals(1)
            c.set_field_mode(mcb.FIELD_AUTO if a.field == "auto" else mcb.FIELD_DENSE)
            c.set_jit(mcb.JIT_AUTO if a.jit == "auto" else mcb.JIT_OFF)
            c.set_grammar(grammar)
            assert c.set_equation(eq) == 0, eq
            M = c.set_grid_step(2.0 / a.res)
            c.polygonise()
            if a.jit == "auto":
                c.jit_wait()
            for _ in range(a.warmup):
                c.polygonise()
            sums = dict.fromkeys(STAGES, 0.0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                cnt = c.polygonise()
                for k in STAGES:
                    sums[k] += getattr(cnt, k)
            wall = (time.perf_counter() - t0) * 1e3 / a.steps
            res["workloads"][wname] = dict(
                equation=eq, grammar=grammar, M=M, cubes=cnt.cubes, active=cnt.active, triangles=cnt.triangles,
                ambiguous=cnt.ambiguous, redirected=cnt.redirected, field_mode=cnt.field_mode, field_blocks=cnt.field_blocks,
                jit=cnt.jit, launches=cnt.launches, wall_ms_per_call=round(wall, 4),
                **{k: round(v / a.steps, 4) for k, v in sums.items()},
                gvoxels_per_s=round(cnt.cubes / (sums["ms_total"] / a.steps) / 1e6, 1) if sums["ms_total"] > 0 else None)
        finally:
            c.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
