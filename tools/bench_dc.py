"""Dual contouring (MCB_MESH_DC, DESIGN.md §14) at 1024^3 against the closest existing quality path, the indexed mesh with
refined vertices and analytic normals, both in one run: a sphere, a torus SDF, the exact box, a union of two spheres and
the literal gyroid.  Per workload and path: counts, the mean per-stage device times over the timed calls (the DC stage or
the weld + refinement + normals is ms_weld), the wall time per call, and in a separate, untimed run the DC stage's kernel
times from torch.profiler.  For the DC mesh also the non-manifold edges (edges not used by exactly two triangles), and for
the box and the union the largest distance from points sampled on the true feature lines (the box's 12 edges, the seam
circle) to each mesh.  One JSON line (also written to --out), with the device name and power limit read in the same run.

    python tools/bench_dc.py [--res 1024] [--steps 10] [--warmup 3] [--out profiles/dc_bench_1024.json]
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

BOX = "max(max(abs(x)-0.5,abs(y)-0.4),abs(z)-0.3)"
UNION = "min(sqrt(x^2+y^2+z^2)-0.5,sqrt((x-0.45)^2+y^2+z^2)-0.35)"
WORKLOADS = [
    ("sphere", "x^2+y^2+z^2-0.49"),
    ("torus_sdf", "sqrt((sqrt(x^2+y^2)-0.5)^2+z^2)-0.2"),
    ("box", BOX),
    ("sphere_union", UNION),
    ("gyroid", "sin(12.566371x)cos(12.566371y)+sin(12.566371y)cos(12.566371z)+sin(12.566371z)cos(12.566371x)"),
]
STAGES = ("ms_eval", "ms_classify", "ms_fill", "ms_emit", "ms_weld", "ms_total")
DC_KERNELS = ("dc_edges_kernel", "dc_vertex_kernel", "dc_emit_kernel", "scan_block_sums_kernel", "scan_sums_kernel", "scan_apply_kernel")


def feature_points(name, n=4000):
    if name == "box":
        t = np.linspace(-1, 1, n)
        pts = []
        h = (0.5, 0.4, 0.3)
        for ax in range(3):
            for s1 in (-1, 1):
                for s2 in (-1, 1):
                    p = np.zeros((n, 3))
                    o = [a for a in range(3) if a != ax]
                    p[:, ax] = t * h[ax]
                    p[:, o[0]] = s1 * h[o[0]]
                    p[:, o[1]] = s2 * h[o[1]]
                    pts.append(p)
        return np.concatenate(pts)
    x0 = (0.25 - 0.1225 + 0.45 ** 2) / 0.9
    r0 = np.sqrt(0.25 - x0 ** 2)
    th = np.linspace(0, 2 * np.pi, n, endpoint=False)
    return np.stack([np.full_like(th, x0), r0 * np.cos(th), r0 * np.sin(th)], 1)


def point_triangle_distance(p, a, b, c):
    """exact distance from points p[n,3] to triangles (a, b, c)[n,3] (float64)"""
    ab, ac = b - a, c - a
    nrm = np.cross(ab, ac)
    nn = (nrm * nrm).sum(1)
    with np.errstate(all="ignore"):
        t = ((p - a) * nrm).sum(1) / nn
        q = p - t[:, None] * nrm
        # barycentric inside test of the projection
        v0, v1, v2 = ac, ab, q - a
        d00, d01, d02, d11, d12 = (v0 * v0).sum(1), (v0 * v1).sum(1), (v0 * v2).sum(1), (v1 * v1).sum(1), (v1 * v2).sum(1)
        den = d00 * d11 - d01 * d01
        u = (d11 * d02 - d01 * d12) / den
        v = (d00 * d12 - d01 * d02) / den
        inside = (u >= 0) & (v >= 0) & (u + v <= 1) & (nn > 0)
        dplane = np.abs(t) * np.sqrt(nn)

    def seg(x, y):
        d = y - x
        s = np.clip(((p - x) * d).sum(1) / np.maximum((d * d).sum(1), 1e-300), 0, 1)
        return np.linalg.norm(p - (x + s[:, None] * d), axis=1)
    dedge = np.minimum(np.minimum(seg(a, b), seg(b, c)), seg(c, a))
    return np.where(inside, np.minimum(dplane, dedge), dedge)


def feature_distance(name, vl, tl, k=24):
    """largest distance from the sampled feature points to the mesh (nearest of the k triangles with the closest centroids)"""
    from scipy.spatial import cKDTree
    p = feature_points(name)
    v = vl.astype(np.float64)
    cen = v[tl].mean(axis=1)
    tree = cKDTree(cen)
    _, idx = tree.query(p, k=k)
    best = np.full(len(p), np.inf)
    for j in range(k):
        t = tl[idx[:, j]]
        best = np.minimum(best, point_triangle_distance(p, v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]))
    return float(best.max())


def nonmanifold_edges(tl):
    e = np.sort(np.concatenate([tl[:, [0, 1]], tl[:, [1, 2]], tl[:, [2, 0]]]).astype(np.int64), axis=1)
    _, n = np.unique(e[:, 0] * (1 << 32) + e[:, 1], return_counts=True)
    return int(np.count_nonzero(n != 2))


def context(mcb, eq, step, dc):
    c = mcb.Context(0)
    c.set_mesh_mode(4 if dc else mcb.MESH_INDEXED)
    c.set_grammar(mcb.GRAMMAR_FUNCTIONS)
    assert c.set_equation(eq) == 0, eq
    c.set_grid_step(step)
    c.set_field_mode(mcb.FIELD_AUTO)
    c.set_normals(3)
    c.set_refine_vertices(not dc)
    return c


def stage_ms(torch, c, calls=3):
    """mean device time per call of the DC stage's kernels (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            c.polygonise()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for kname in DC_KERNELS:
            if kname in e.key:
                out[kname] = out.get(kname, 0.0) + e.device_time_total / 1e3 / calls
    out = {k: round(v, 4) for k, v in out.items()}
    out["stage"] = round(sum(out.values()), 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_dc.py measures the GPU path: no CUDA device")
    mcb = importlib.import_module("marching-cube-for-implicit-surfaces_b200")
    name, limit = device_info(0)
    res = {"tool": "bench_dc", "res": a.res, "steps": a.steps, "warmup": a.warmup, "device": name or torch.cuda.get_device_name(0),
           "power_limit": limit, "workloads": {}}
    for wname, eq in WORKLOADS:
        row = {"equation": eq}
        for path in ("indexed_refined_mode3", "dc"):
            dc = path == "dc"
            c = context(mcb, eq, 2.0 / a.res, dc)
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
                r = dict(M=cnt.M, active=cnt.active, triangles=cnt.triangles, vertices=cnt.vertices, launches=cnt.launches, jit=cnt.jit,
                         wall_ms_per_call=round(wall, 4), **{k: round(v / a.steps, 4) for k, v in sums.items()})
                vl, tl = c.get_indexed_mesh()
                if dc:
                    r["profiler_ms"] = stage_ms(torch, c)
                    r["nonmanifold_edges"] = nonmanifold_edges(tl)
                if wname in ("box", "sphere_union"):
                    r["feature_line_max_distance"] = feature_distance(wname, vl, tl)
                row[path] = r
            finally:
                c.close()
        row["total_ratio_dc_over_indexed"] = round(row["dc"]["ms_total"] / row["indexed_refined_mode3"]["ms_total"], 3)
        res["workloads"][wname] = row
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
