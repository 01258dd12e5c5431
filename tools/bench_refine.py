"""Refined vertices (mcb_set_refine_vertices) at 1024^3: a sphere, a torus SDF, a box SDF and the literal gyroid, each in soup
and in indexed mode, with refinement off and on.  Per workload and mode: counts, the mean per-stage device times over the
timed calls (the refinement pass is inside ms_emit for the soup, ms_weld for the indexed mesh, and ms_total), the pass's
own kernel time from torch.profiler in a separate, untimed run, and the evaluations of the equation per refined vertex
(mean and maximum, the host build of the rule run on a random sample of the unrefined vertices: the count is a function of
the position alone).  Then the accuracy table of DESIGN.md §13: the float64 |f| / |grad f| at the welded vertices, linear
against refined, at step 0.2 and 2/256.  One JSON line, with the device name and power limit read in the same run.

    python tools/bench_refine.py [--res 1024] [--steps 10] [--warmup 3] [--sample 200000]
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

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
    """mean device time per call of refine_vertices_kernel (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            c.polygonise()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "refine_vertices_kernel" in e.key)
    return round(us / 1e3 / calls, 4)


def context(mcb, eq, grammar, step, mesh_mode, refine):
    c = mcb.Context(0)
    c.set_mesh_mode(mesh_mode)
    c.set_normals(0)
    c.set_grammar(grammar)
    assert c.set_equation(eq) == 0, eq
    c.set_grid_step(step)
    c.set_refine_vertices(refine)
    return c


def accuracy(mcb, refine_common, postfix_program, grad64, eq, grammar, step):
    """float64 |f| / |grad f| at the welded vertices of the unrefined and the refined mesh: max and mean"""
    out = {}
    for refine in (False, True):
        c = context(mcb, eq, grammar, step, mcb.MESH_INDEXED, refine)
        try:
            c.polygonise()
            vl = c.get_indexed_mesh()[0]
        finally:
            c.close()
        v, g = grad64(postfix_program(mcb, eq, grammar), vl)
        with np.errstate(all="ignore"):
            d = np.abs(v) / np.linalg.norm(g, axis=1)
        d = d[np.isfinite(d)]
        out["refined" if refine else "linear"] = {"vertices": int(len(vl)), "max": float(d.max()), "mean": float(d.mean())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=200000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_refine.py measures the GPU path: no CUDA device")
    mcb = importlib.import_module("marching-cube-for-implicit-surfaces_b200")
    from tests import refine_common
    from tests.normals_common import grad64, postfix_program
    name, limit = device_info(0)
    res = {"tool": "bench_refine", "res": a.res, "steps": a.steps, "warmup": a.warmup, "eval_sample": a.sample,
           "device": name or torch.cuda.get_device_name(0), "power_limit": limit, "workloads": {}, "accuracy": {}}
    rng = np.random.default_rng(0)
    for wname, grammar, eq in WORKLOADS:
        for mesh in ("soup", "indexed"):
            row = {}
            for refine in (False, True):
                c = context(mcb, eq, grammar, 2.0 / a.res, mcb.MESH_SOUP if mesh == "soup" else mcb.MESH_INDEXED, refine)
                try:
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
                    r = dict(M=cnt.M, triangles=cnt.triangles, vertices=cnt.vertices, launches=cnt.launches, jit=cnt.jit,
                             wall_ms_per_call=round(wall, 4), **{k: round(v / a.steps, 4) for k, v in sums.items()})
                    if refine:
                        r["ms_refine_pass"] = pass_ms(torch, c)
                    else:  # evaluations per vertex: the host rule on a sample of the unrefined positions
                        p = c.get_mesh(normals=False)[0][:, :, :3].reshape(-1, 3) if mesh == "soup" else c.get_indexed_mesh()[0]
                        p = p[rng.choice(len(p), min(a.sample, len(p)), replace=False)]
                        _, ev, _ = refine_common.host_refine(eq, mcb.grid_axis(2.0 / a.res)[1], p, 0.0, (1.0, 1.0, 1.0), grammar)
                        moved = ev[ev > 0]
                        r["evals_per_refined_vertex"] = {"mean": round(float(moved.mean()), 3), "max": int(moved.max()),
                                                         "refined_share": round(len(moved) / len(ev), 4),
                                                         "same_sign": int((ev == refine_common.SAME_SIGN).sum())}
                    row["refine" if refine else "off"] = r
                finally:
                    c.close()
            res["workloads"]["%s_%s" % (wname, mesh)] = dict(equation=eq, grammar=grammar, **row)
    for wname, grammar, eq in WORKLOADS:
        for step in (0.2, 2.0 / 256):
            res["accuracy"]["%s_step_%g" % (wname, step)] = accuracy(mcb, refine_common, postfix_program, grad64, eq, grammar, step)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
