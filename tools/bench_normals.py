"""Analytic normals (mcb_set_normals 3) against central-difference normals (mode 1) at 1024^3: a sphere, a torus SDF, a box
SDF and the literal gyroid, each in soup and in indexed mode.  Per workload and mode: counts, the mean per-stage device times
over the timed calls (the analytic pass is inside ms_emit for the soup, ms_weld for the indexed mesh, and ms_total), and the
analytic pass's own kernel time from torch.profiler in a separate, untimed run.  Mode 0 (positions only) is measured beside
them.  One JSON line, with the device name and power limit read in the same run.

    python tools/bench_normals.py [--res 1024] [--steps 10] [--warmup 3]
"""
import argparse
import importlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_csg import device_info  # noqa: E402

WORKLOADS = [
    ("sphere", 0, "x^2+y^2+z^2-0.49"),
    ("torus_sdf", 1, "sqrt((sqrt(x^2+y^2)-0.5)^2+z^2)-0.2"),
    ("box_sdf", 1, "sqrt(max(abs(x)-0.5,0)^2+max(abs(y)-0.4,0)^2+max(abs(z)-0.3,0)^2)-0.1"),
    ("gyroid", 1, "sin(12.566371x)cos(12.566371y)+sin(12.566371y)cos(12.566371z)+sin(12.566371z)cos(12.566371x)"),
]
STAGES = ("ms_eval", "ms_classify", "ms_emit", "ms_weld", "ms_total")


def pass_ms(torch, c, calls=3):
    """mean device time per call of grad_normals_kernel (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            c.polygonise()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "grad_normals_kernel" in e.key)
    return round(us / 1e3 / calls, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_normals.py measures the GPU path: no CUDA device")
    mcb = importlib.import_module("marching-cube-for-implicit-surfaces_b200")
    name, limit = device_info(0)
    res = {"tool": "bench_normals", "res": a.res, "steps": a.steps, "warmup": a.warmup,
           "device": name or torch.cuda.get_device_name(0), "power_limit": limit, "workloads": {}}
    for wname, grammar, eq in WORKLOADS:
        for mesh in ("soup", "indexed"):
            row = {}
            for normals in (0, 1, 3):
                c = mcb.Context(0)
                try:
                    c.set_mesh_mode(mcb.MESH_SOUP if mesh == "soup" else mcb.MESH_INDEXED)
                    c.set_normals(normals)
                    c.set_grammar(grammar)
                    assert c.set_equation(eq) == 0, eq
                    M = c.set_grid_step(2.0 / a.res)
                    c.polygonise()
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
                    r = dict(M=M, triangles=cnt.triangles, vertices=cnt.vertices, launches=cnt.launches, jit=cnt.jit,
                             wall_ms_per_call=round(wall, 4), **{k: round(v / a.steps, 4) for k, v in sums.items()})
                    if normals == 3:
                        r["ms_analytic_pass"] = pass_ms(torch, c)
                    row["mode%d" % normals] = r
                finally:
                    c.close()
            res["workloads"]["%s_%s" % (wname, mesh)] = dict(equation=eq, grammar=grammar, **row)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
