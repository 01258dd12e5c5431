"""Function-grammar workloads at 1024^3 (MCB_GRAMMAR_FUNCTIONS): literal gyroid, SDF torus, a trig field that cannot be
hoisted into axis tables, and the polynomial gyroid gyr78 of the reference grammar beside them.  One JSON line: per
workload the counts, the per-stage device times (mean over the timed calls), field_blocks and jit, plus the device name
and power limit read in the same run.

    python tools/bench_functions.py [--res 1024] [--steps 20] [--warmup 3] [--field auto|dense] [--jit auto|off]
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

GYR78 = ("((x*(-7+x^2*(56+x^2*(-112+64*x^2))))*(1+y^2*(-32+y^2*(160+y^2*(-256+128*y^2)))))"
         "+((y*(-7+y^2*(56+y^2*(-112+64*y^2))))*(1+z^2*(-32+z^2*(160+z^2*(-256+128*z^2)))))"
         "+((z*(-7+z^2*(56+z^2*(-112+64*z^2))))*(1+x^2*(-32+x^2*(160+x^2*(-256+128*x^2)))))")
WORKLOADS = [
    ("gyroid_literal", 1, "sin(12.566371x)cos(12.566371y)+sin(12.566371y)cos(12.566371z)+sin(12.566371z)cos(12.566371x)"),
    ("torus_sdf", 1, "sqrt((sqrt(x^2+y^2)-0.5)^2+z^2)-0.2"),
    ("trig_nonhoisted", 1, "sin(6(x^2+y^2+z^2))"),
    ("gyr78", 0, GYR78),
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
        raise SystemExit("bench_functions.py measures the GPU path: no CUDA device")
    mcb = importlib.import_module("marching-cube-for-implicit-surfaces_b200")
    name, limit = device_info(0)
    res = {"tool": "bench_functions", "res": a.res, "steps": a.steps, "warmup": a.warmup, "field": a.field, "jit_mode": a.jit,
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
