#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json: Gvoxels/s and Mtriangles/s at 1024^3 / 2048^3).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N ...            # the reference's own CPU implementation (oracle/_ref)

One "step" = one full polygonisation of the workload through the C ABI: axis tables -> interval classes of the vertex
blocks -> field + sign planes where undecided -> classify/scan/compact -> emit (positions + normals), inputs (bytecode,
coordinates) already resident in HBM, and the 48-byte counts read back.  Nothing is carried over from one step to the
next: a first or changed configuration runs the same path (`changed_param`, `first_call` in the line).
MCB_JIT_AUTO compiles a new equation's kernels on a background thread; the timed loops start after mcb_jit_wait (the steady
state), `first_call` shows the first mesh of a new equation (interpreter) and when the compiled kernels were in place.
For N>1 each rank owns a z-slab (SURVEY.md §8e), cut so that every rank carries the same cost (mcb_comm_balance, refined
twice by measured time: mcb_comm_rebalance; `strong_2048.per_rank` shows every rank's slab and kernel times), and every
step includes the all-gather of the per-slab triangle counts (NCCL, behind the C ABI, enqueued inside mcb_polygonise on a
side stream: mcb_comm_set_auto) that gives every slab its global output offset.

Workloads (BASELINE.json configs):
  headline   sphere x^2+y^2+z^2-0.49, configs[2]; N=1 -> 1024^3 (M=1025 cubes per axis in the reference's loop semantics);
             N ranks -> the grid with N times the voxels, step 2/n with n = round(1024*N^(1/3)) (N=8: 2048^3), weak scaling
  workloads  configs[3] the polynomial gyroid gyr78 (high triangle density, ambiguity redirect at scale) and the torus at
             1024^3, in the N=1 line under "workloads"
  strong_2048 configs[4]: the 2048^3 sphere on N GPUs (strong scaling) next to the same grid on rank 0 alone
"voxel" = one cube visited by the reference loop.
"""
import argparse
import importlib
import itertools
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "marching-cube-for-implicit-surfaces_b200"
_REAL_STDOUT = None


def emit_line(obj):
    """the one JSON line, on the process's original stdout"""
    data = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)

WORKLOADS = {
    "sphere": "x^2+y^2+z^2-0.49",
    "torus": "(x^2+y^2+z^2+0.25-0.0625)^2-(x^2+y^2)",
    "eq8": "(x^2+y^2-(1/16))^2+(y^2+z^2-(1/16))^2+(z^2+x^2-(1/16))^2-8*(x^2+y^2+z^2-(1/4))^2",
    # BASELINE.json configs[3]: a true gyroid is not expressible in the reference grammar (no sin/cos); this is the
    # polynomial gyroid of SURVEY.md Appendix B (Chebyshev T7/T8 in Horner form), the high-triangle-density stress field
    "gyr78": ("((x*(-7+x^2*(56+x^2*(-112+64*x^2))))*(1+y^2*(-32+y^2*(160+y^2*(-256+128*y^2)))))"
              "+((y*(-7+y^2*(56+y^2*(-112+64*y^2))))*(1+z^2*(-32+z^2*(160+z^2*(-256+128*z^2)))))"
              "+((z*(-7+z^2*(56+z^2*(-112+64*z^2))))*(1+x^2*(-32+x^2*(160+x^2*(-256+128*x^2)))))"),
}


DUMP_BYTES = 64_000_000


def dump_outputs(path, ctx, suffix=""):
    """Writes what the last timed step computed, as a caller of polygonise() + get_mesh() receives it: the triangle soup's
    positions and gradient normals (float32, [T,3,3]) and the step's counts (float64).  A soup larger than DUMP_BYTES is
    cut to a fixed, seeded sample of its triangles, kept in soup order, with their indices in the soup alongside."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    c = ctx.counts
    pos, nrm = ctx.get_mesh()
    T = pos.shape[0]
    keep = min(T, (DUMP_BYTES - 4096) // (2 * 36 + 8))  # positions + normals + index per triangle
    idx = np.arange(T) if keep == T else np.sort(np.random.default_rng(0).choice(T, keep, replace=False))
    arrays = {"soup_positions": pos[idx, :, :3], "soup_normals": nrm[idx, :, :3], "soup_triangle_index": idx.astype(np.float64),
              "counts": np.array([c.cubes, c.active, c.triangles, c.ambiguous, c.redirected, c.M, c.k_begin, c.k_end], np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + suffix + ".npy"), np.ascontiguousarray(a))


def resolution_for(ngpus, base):
    n = int(round(base * ngpus ** (1.0 / 3.0)))
    return n + (n & 1)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def count_since(self, t0):
        return sum(1 for (t, _) in self.rows if t >= t0)

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for (t, line) in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            inside = t0 - 0.05 <= t <= t1 + 0.05
            try:
                if inside:
                    sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            if inside:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: take the nearest samples
            for (t, line) in self.rows[-3:]:
                try:
                    sm.append(float(line.split(",")[0]))
                except ValueError:
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_rate(eq, step, seconds_target, threads):
    """Times the UNMODIFIED reference (oracle/_ref: calculate_step + add_step_to_poly_data per cube, marching.cpp:375-383)
    on a bounded sample: the middle cube layers of the same grid, split over `threads` independent Evaluator+Marching
    pairs.  Returns (Gvoxels/s, Mtriangles/s, sample description, seconds).  Only oracle/ is loaded here, never the
    product library."""
    from oracle import refbind
    if not refbind.available():
        raise RuntimeError("oracle/_ref/libmcref.so missing: run __graft_entry__.build() where /root/reference exists")
    M, _ = refbind.Ref(eq, step, force_step=True).coords()  # the reference's own grid loop (marching.cpp:372-377)
    # calibrate on a few rows through the middle of the grid, then size the sample for ~seconds_target of wall time
    mid_row = (M // 2) * M + M // 4
    t_probe, cubes_p, _ = refbind.timed_rows_mt(eq, step, row0=mid_row, nrows=threads * 2, nthreads=threads)
    rate = cubes_p / max(t_probe, 1e-6)
    nrows = int(max(threads * 2, min(M * M, round(seconds_target * rate / M))))
    # centre the sample on the middle layers so that it crosses the surface like the full grid does
    row0 = max(0, min(M * M - nrows, (M // 2) * M + M // 2 - nrows // 2))
    sec, cubes, tris = refbind.timed_rows_mt(eq, step, row0=row0, nrows=nrows, nthreads=threads)
    sample = "cube rows [%d,%d) (row=k*M+j, M=%d: %d cubes around the middle layers of the %d^3-cube grid), %d threads, unmodified Marching::calculate_step+add_step_to_poly_data" % (
        row0, row0 + nrows, M, cubes, M, threads)
    cpu_reference_rate.last_M = M
    return cubes / sec / 1e9, tris / sec / 1e6, sample, sec


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    eq = WORKLOADS[args.workload]
    n = resolution_for(args.gpus, args.base_res)
    step = 2.0 / n
    threads = os.cpu_count() or 1
    per_step = max(1.0, min(6.0, 120.0 / max(1, args.steps + args.warmup)))
    vals, tris, secs = [], [], []
    sample = ""
    t_all = time.time()
    for i in range(args.warmup + args.steps):
        gv, mt, sample, sec = cpu_reference_rate(eq, step, per_step, threads)
        if i >= args.warmup:
            vals.append(gv); tris.append(mt); secs.append(sec)
    v = statistics.mean(vals)
    M = cpu_reference_rate.last_M
    full_ms = float(M) ** 3 / (v * 1e9) * 1e3  # one pass over the whole grid at the measured per-cube rate
    out = {"impl": "reference", "metric": "Gvoxels/s", "value": v, "unit": "Gvoxels/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": full_ms, "ms_per_sample_step": statistics.mean(secs) * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "mtriangles_per_s": statistics.mean(tris),
           "config": {"workload": "%s %s at %d^3 (step 2/%d), CPU reference on a bounded sample" % (args.workload, eq, n, n),
                      "timing": "wall clock around the reference loop; ms_per_step = the whole %d^3-cube grid at the measured per-cube rate "
                                "(a full pass takes minutes), ms_per_sample_step = what one timed step really ran" % M},
           "cpu_baseline": {"value": v, "unit": "Gvoxels/s", "cores": threads, "kind": "reference", "sample": sample},
           "e2e": {"value": v, "unit": "Gvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "wall_s": time.time() - t_all}
    emit_line(out)
    return 0


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        # the driver's NCCL_DEBUG goes through; NCCL's own log is sent to stderr so that stdout stays the one JSON line
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    mcb = importlib.import_module(PKG)
    stream = torch.cuda.current_stream()
    launches_total = [0]
    comm_up = [False]
    auto_on = [False]

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_ranks(xs):
        """[rank][len(xs)] list of every rank's values"""
        t = torch.tensor([float(x) for x in xs], dtype=torch.float64, device="cuda")
        if world == 1:
            return [[float(x) for x in t.tolist()]]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [[float(x) for x in o.tolist()] for o in out]

    def sum_over_ranks(xs):
        t = torch.tensor([float(x) for x in xs], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    ctx = mcb.Context(local)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_field_mode(mcb.FIELD_AUTO)  # what the drop-in class uses
    if world > 1:  # the path's own communicator, behind the C ABI (libnccl dlopen'ed by libmcb200.so); the id travels by torch
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(mcb.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        comm_id = bytes(idt.cpu().numpy().tobytes())

    def configure(eq, n, mesh=mcb.MESH_SOUP, normals=1, balance=True):
        """equation + grid + this rank's slab; with several ranks the slabs are cut by measured cost (one profiling pass)"""
        assert ctx.set_equation(eq) == 0
        ctx.jit_wait()  # MCB_JIT_AUTO compiles in the background: the steady state is what is timed (first_call shows the rest)
        ctx.set_surface_constant(0.0)
        M = ctx.set_grid_step(2.0 / n)
        ctx.set_mesh_mode(mesh)
        ctx.set_normals(normals)
        ctx.set_host_output(0, 0, 0, 0, 0)
        k0, k1 = 0, M
        if world > 1:
            k0, k1 = mcb.slab_range(M, rank, world)
            if not comm_up[0]:
                ctx.comm_init(comm_id, rank, world)      # ncclCommInitRank + the uniform slab (mcb_slab_range)
                ctx.comm_set_auto(True)                  # the all-gather is enqueued inside polygonise(), behind the emission
                auto_on[0] = True
                comm_up[0] = True
            else:
                ctx.set_slab(k0, k1)
            if balance:
                ctx.set_stage_timing(True)
                ctx.polygonise()                         # profile: triangles per layer of the uniform slab
                k0, k1 = ctx.comm_balance()              # NCCL all-reduce of the layer histogram + the same cut on every rank
                for _ in range(2):                       # two refinements by measured device time (mcb_comm_rebalance)
                    ctx.polygonise()
                    ms = sum(ctx.polygonise().ms_total for _ in range(4)) / 4
                    k0, k1 = ctx.comm_rebalance(ms)
        return M, k0, k1

    def step_fn():
        c = ctx.polygonise()
        if world > 1:      # the path's only exchange: per-slab triangle counts -> global output offsets (NCCL all-gather
            ctx.comm_exchange()  # straight from the device counters, on a side stream)
        launches_total[0] += c.launches
        return c

    def timed(fn, steps, warm=3):
        """K steps between two CUDA events on the launching stream (stage events off: they sit between the short kernels);
        the per-stage device times come from a few extra, untimed steps with the stage events on."""
        ctx.set_stage_timing(False)
        for _ in range(warm):
            c = fn()
        if world > 1 and comm_up[0] and auto_on[0]:
            ctx.comm_offsets(world)  # the warm-up's exchanges (NCCL sets its channels up lazily) are over before the clock starts
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        launches_total[0] = 0  # kernels launched inside the timed region only
        e0.record(stream)
        for _ in range(steps):
            c = fn()
        if world > 1 and auto_on[0]:
            ctx.comm_offsets(world)  # the last exchange is inside the timed region
        e1.record(stream)
        sync_all()
        t1 = time.time()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        launches = launches_total[0]
        ctx.set_stage_timing(True)
        stage = {"ms_tables": 0.0, "ms_eval": 0.0, "ms_classify": 0.0, "ms_emit": 0.0, "ms_fill": 0.0, "ms_weld": 0.0}
        ns = max(1, min(steps, 8))
        for _ in range(ns):
            c = fn()
            for k in stage:
                stage[k] += getattr(c, k)
        sync_all()
        launches_total[0] = launches
        return ms, c, {k: v / ns for k, v in stage.items()}, (t0, t1)

    def e2e_times(eq, n, k0, k1, steps):
        """equation text in -> mesh on the HOST, host<->device copies inside the timed region, three output forms"""
        step = 2.0 / n

        def make(mode, normals):
            ctx.set_mesh_mode(mode)
            ctx.set_normals(normals)
            ctx.set_host_output(0, 0, 0, 0, 0)
            cc0 = ctx.polygonise()
            capT = int(cc0.triangles) + 1024
            if mode == mcb.MESH_INDEXED:
                capV = int(cc0.vertices) + 1024
                bufs = [torch.empty((capV, 3), dtype=torch.float32).pin_memory(), torch.empty((capT, 3), dtype=torch.int32).pin_memory(),
                        torch.empty((capV, 3), dtype=torch.float32).pin_memory()]
                ctx.set_host_output(bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr() if normals else 0, capV, capT)
            else:
                bufs = [torch.empty((capT, 3, 4), dtype=torch.float32).pin_memory(), torch.empty((capT, 3, 4), dtype=torch.float32).pin_memory()]

            def one():
                assert ctx.set_equation(eq) == 0          # tokenise + lower + upload bytecode (H2D) + fold constants
                ctx.set_grid_step(step)                   # host coordinate loop + upload (H2D)
                ctx.set_slab(k0, k1)
                cc = step_fn()                            # MESH_INDEXED: returns when Poly_Data is in the host buffers (D2H inside)
                if mode == mcb.MESH_INDEXED:
                    if not ctx.host_output_filled():      # first call after a buffer had to grow: plain copy
                        ctx.get_indexed_mesh_into(bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr() if normals else 0, capV, capT)
                else:
                    ctx.get_mesh_into(bufs[0].data_ptr(), bufs[1].data_ptr(), capT)  # D2H of positions + normals
                return cc
            return one, bufs

        out = {}
        for key, mode, normals in (("soup", mcb.MESH_SOUP, 1), ("poly_data_only", mcb.MESH_INDEXED, 0), ("indexed", mcb.MESH_INDEXED, 1)):
            one, bufs = make(mode, normals)
            for _ in range(2):
                one()
            sync_all()
            nst = max(1, min(steps, 10))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0 = time.perf_counter()
            e0.record(stream)
            for _ in range(nst):
                cc = one()
            e1.record(stream)
            sync_all()
            wall_ms = (time.perf_counter() - w0) * 1e3
            ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms) / nst)
            if key == "soup":
                d2h = int(cc.triangles) * 96 + 48
            elif key == "poly_data_only":
                d2h = int(cc.vertices) * 12 + int(cc.triangles) * 12 + 48
            else:
                d2h = int(cc.vertices) * 24 + int(cc.triangles) * 12 + 48
            out[key] = {"ms_per_step": ms, "d2h_bytes_per_step": int(sum_over_ranks([d2h])[0]), "steps": nst, "ms_weld": cc.ms_weld}
            del bufs
        ctx.set_host_output(0, 0, 0, 0, 0)
        ctx.set_mesh_mode(mcb.MESH_SOUP)
        ctx.set_normals(1)
        return out

    def kernels_of(per, c, M, layers):
        """per-stage device times with their algorithmic bytes (SURVEY.md §8(d) / DESIGN.md §roofline)"""
        V = (M + 1) * (M + 1) * (layers + 1)
        A_r, T_r = float(c.active), float(c.triangles)
        kern = {
            "eval_field": {"ms": per["ms_eval"], "bytes": 4.0 * V + V / 8.0, "written_bytes": 2112.0 * float(c.field_blocks),
                           "what": "SURVEY 8(d) accounting: 4 B field + 1 bit sign per grid vertex.  Block-field mode: interval classes of all 32x4x4 vertex "
                                   "blocks, field + signs written only in the undecided ones (written_bytes), so this algorithmic rate exceeds the HBM "
                                   "peak - as SURVEY 8(d) anticipates for a variant that never writes the field; variants.dense_field.eval_GBps is the "
                                   "kernel that really writes 4 B/vertex (%s)" % ("kernels NVRTC compiled for the equation" if c.jit else "bytecode interpreter")},
            "classify+compact": {"ms": per["ms_classify"], "bytes": V / 8.0 + 12.0 * A_r,
                                 "what": "1 bit per vertex read + 12 B per active cube written (our layout; SURVEY's 4V+C accounting is in classify_scan_emit_vs_survey_bytes)"},
            "emit": {"ms": per["ms_emit"], "bytes": 12.0 * A_r + 32.0 * A_r + 96.0 * T_r,
                     "what": "12 B record + 8 corner values per active cube read, 96 B per triangle written"},
            "apron_refill": {"ms": per["ms_fill"], "bytes": 8.0 * A_r, "what": "field blocks next to the surface that the interval test had decided: evaluated for the gradient stencil"},
        }
        return kern

    def finish(kern, hbm):
        for d in kern.values():
            d["GBps"] = d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else None
            d["frac_of_hbm_peak"] = d["GBps"] / hbm if d["GBps"] else None
        return kern

    # ================================ headline: sphere, weak scaling ================================================
    eq = WORKLOADS[args.workload]
    n = resolution_for(world, args.base_res)
    sampler = ClockSampler(local) if rank == 0 else None  # nvidia-smi takes ~0.1 s to start: it runs from the warm-up on
    M, k0, k1 = configure(eq, n)
    ms_per_step, c, per, (t0, t1) = timed(step_fn, args.steps, max(3, args.warmup))
    headline_launches = launches_total[0]  # kernels launched inside the timed region
    soak = 0
    if sampler and sampler.proc and world == 1:
        # a timed region shorter than the sampling period holds no sample: keep the same load running (untimed) until
        # one has been taken, so that the clocks reported are clocks under this load
        t_soak = time.time()
        while sampler.count_since(t0) < 2 and time.time() - t_soak < 1.0:
            step_fn()
            soak += 1
        torch.cuda.synchronize()
        t1 = time.time()
    clocks = sampler.stop(t0, t1) if sampler else None
    if clocks is not None:
        clocks["window"] = "timed region" if soak == 0 else "timed region + %d untimed steps of the same load after it" % soak
    # the untimed steps since the last timed one (timed()'s stage-timing steps, the soak) repeat it with the same inputs, so
    # the device still holds its outputs; dumping later keeps the clock sampler's window on the load
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ctx, "" if world == 1 else "_rank%d" % rank)
    cubes, tris, active = sum_over_ranks([c.cubes, c.triangles, c.active])
    value = cubes / (ms_per_step * 1e-3) / 1e9
    layers = k1 - k0
    slabs = [int(x) for x in sum_over_ranks([k0 if r == rank else 0 for r in range(world)])] + [M] if world > 1 else [0, M]

    # ---- every step a NEW configuration (another iso value): nothing learnt from the previous step can help --------
    isos = [1e-4 * (1 + (i % 9)) for i in range(args.steps)]
    it = itertools.cycle(isos)

    def changed_step():
        ctx.set_surface_constant(next(it))
        return step_fn()
    ch_ms, _, _, _ = timed(changed_step, args.steps, 3)
    ctx.set_surface_constant(0.0)
    changed = {"ms_per_step": ch_ms, "value": cubes / (ch_ms * 1e-3) / 1e9, "ratio_to_value": ms_per_step / ch_ms,
               "what": "same equation, a different surface constant in every timed step (a slider move): the same code path as `value`"}

    # ---- variants / first call / other workloads (N = 1 only: informational, outside the headline timing) ----------
    variants, first_call, workloads, strong = {}, None, {}, None
    if world == 1:
        nv = max(1, min(args.steps, 10))
        ctx.set_field_mode(mcb.FIELD_DENSE)
        dn_ms, cs_, dper, _ = timed(step_fn, nv, 3)
        V_ = (M + 1) * (M + 1) * (M + 1)
        variants["dense_field"] = {"value": float(cs_.cubes) / (dn_ms * 1e-3) / 1e9, "ms_per_step": dn_ms, "ms_eval": dper["ms_eval"], "steps": nv,
                                   "eval_GBps": (4.0 * V_ + V_ / 8.0) / (dper["ms_eval"] * 1e-3) / 1e9,
                                   "what": "mcb_set_field_mode(MCB_FIELD_DENSE): every vertex's value written to HBM (4 B/vertex); "
                                           "eval_GBps is that kernel's real write rate"}
        ctx.set_field_mode(mcb.FIELD_AUTO)
        ctx.set_jit(mcb.JIT_OFF)  # the bytecode interpreter instead of the kernels NVRTC compiled (same results bit for bit)
        in_ms, ci_, iper, _ = timed(step_fn, nv, 3)
        variants["interpreter"] = {"value": float(ci_.cubes) / (in_ms * 1e-3) / 1e9, "ms_per_step": in_ms, "ms_eval": iper["ms_eval"], "steps": nv,
                                   "what": "mcb_set_jit(MCB_JIT_OFF): eval_blocks_kernel interpreting the fused bytecode"}
        ctx.set_jit(mcb.JIT_AUTO)
        # a brand-new context and an equation nothing has compiled yet: wall time to the first mesh on the device
        w0 = time.perf_counter()
        c2 = mcb.Context(local)
        c2.set_field_mode(mcb.FIELD_AUTO)
        assert c2.set_equation("x^2+y^2+z^2-0.4899") == 0
        c2.set_grid_step(2.0 / n)
        c2.set_normals(1)
        cc2 = c2.polygonise()
        w1 = time.perf_counter()
        cc3 = c2.polygonise()
        w2 = time.perf_counter()
        c2.jit_wait()
        w3 = time.perf_counter()
        cc4 = c2.polygonise()
        w4 = time.perf_counter()
        first_call = {"ms_wall": (w1 - w0) * 1e3, "jit_first_call": int(cc2.jit), "ms_second_call_wall": (w2 - w1) * 1e3, "reruns": cc2.reruns,
                      "ms_until_compiled_wall": (w3 - w0) * 1e3, "ms_compile": cc4.ms_compile, "ms_call_after_compile_wall": (w4 - w3) * 1e3,
                      "what": "mcb_create + a new equation + buffer allocation + first polygonisation, wall clock (NVRTC compiles the "
                              "equation's kernels on a background thread meanwhile: that call and the next run the bytecode interpreter, "
                              "same results); then the wall time at which the compiled kernels were in place and the first call using them"}
        c2.close()

    # ---- e2e: through the reference-facing call with HOST buffers: equation text in, Poly_Data out ------------------
    e2e = e2e_times(eq, n, k0, k1, args.steps)
    idx_ms = e2e["indexed"]["ms_per_step"]
    h2d = 4 * (mcb.lib.mcb_grid_axis(2.0 / n, None, 0) + 3 + 64) * 2 + 2052 * 2 + 512

    if world == 1:
        # ---- BASELINE configs[3] (gyr78) and the torus at the same resolution -----------------------------------
        for name in ("gyr78", "torus"):
            Mw, a0, a1 = configure(WORKLOADS[name], n)
            st = max(3, min(args.steps, 20))
            w_ms, wc, wper, _ = timed(step_fn, st, 3)
            we = e2e_times(WORKLOADS[name], n, a0, a1, 5)
            workloads[name] = {"equation": WORKLOADS[name], "resolution": n, "M": Mw, "value": float(wc.cubes) / (w_ms * 1e-3) / 1e9, "ms_per_step": w_ms, "steps": st,
                               "mtriangles_per_s": float(wc.triangles) / (w_ms * 1e-3) / 1e6, "cubes": int(wc.cubes), "active_cubes": int(wc.active),
                               "triangles": int(wc.triangles), "ambiguous": int(wc.ambiguous), "redirected": int(wc.redirected),
                               "field_blocks_evaluated": int(wc.field_blocks), "kernels_ms": wper,
                               "e2e": {"value": float(wc.cubes) / (we["indexed"]["ms_per_step"] * 1e-3) / 1e9, **we["indexed"],
                                       "poly_data_only": we["poly_data_only"], "soup": we["soup"]}}
    # ---- BASELINE configs[4]: the 2048^3 sphere, strong scaling ---------------------------------------------------
    if not args.no_strong:
        ns = 2048
        Ms, s0, s1 = configure(WORKLOADS["sphere"], ns)
        st = max(3, min(args.steps, 20))
        s_ms, sc_, sper, _ = timed(step_fn, st, 3)
        s_cubes, s_tris = sum_over_ranks([sc_.cubes, sc_.triangles])
        per_rank = gather_ranks([s0, s1, sc_.triangles, sper["ms_eval"], sper["ms_classify"] + sper["ms_fill"], sper["ms_emit"],
                                 sper["ms_tables"] + sper["ms_eval"] + sper["ms_classify"] + sper["ms_fill"] + sper["ms_emit"]])
        strong = {"resolution": ns, "M": Ms, "ms_per_step": s_ms,
                  "per_rank": [{"slab": [int(r[0]), int(r[1])], "triangles": int(r[2]), "ms_eval": r[3], "ms_classify": r[4], "ms_emit": r[5],
                                "ms_kernels": r[6]} for r in per_rank], "value": s_cubes / (s_ms * 1e-3) / 1e9, "mtriangles_per_s": s_tris / (s_ms * 1e-3) / 1e6,
                  "steps": st, "triangles": s_tris, "rank0_slab": [s0, s1], "rank0_kernels_ms": sper, "scaling": "strong",
                  "slabs": "cut by measured cost (mcb_comm_balance)" if world > 1 else "one slab"}
        if world > 1:
            # the same grid on rank 0 alone, in the same run on the same box: the strong-scaling reference
            sync_all()
            ctx.comm_set_auto(False)  # rank 0 polygonises alone now: no collective may be enqueued
            auto_on[0] = False
            if rank == 0:
                ctx.set_slab(0, Ms)
                for _ in range(2):
                    ctx.polygonise()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(5):
                    ctx.polygonise()
                e1.record(stream)
                torch.cuda.synchronize()
                n1_ms = e0.elapsed_time(e1) / 5
                strong["n1_ms_per_step"] = n1_ms
                strong["efficiency_vs_n1_2048"] = n1_ms / (world * s_ms)
            sync_all()

    dropin = None
    if world == 1 and not args.no_dropin:
        # the reference-facing C++ class itself: include/marching.h Marching::recalculate() via tools/headless_main.cpp
        exe = os.path.join(ROOT, PKG, "mcb_headless")
        try:
            r = subprocess.run([exe, "--eq", eq, "--res", str(n), "--scale", "1", "1", "1", "--repeat", "14"], capture_output=True, text=True, timeout=300,
                               env=dict(os.environ, MCB_DEVICE=str(local)))
            d = json.loads(r.stdout.strip().splitlines()[-1])
            dropin = {"value": float(d["cubes"]) / (d["ms_recalculate_mean"] * 1e-3) / 1e9, "ms_per_step": d["ms_recalculate_mean"], "ms_best": d["ms_recalculate_wall"],
                      "ms_first_call": d["ms_recalculate_first"], "calls": d["calls"], "vertices": d["vertices"], "triangles": d["triangles"],
                      "what": "mcb_headless: Evaluator + Marching of include/*.h, wall clock around Marching::recalculate(), Poly_Data (std::vector) + vertex "
                              "normals filled on return; mean of the calls after the first three"}
        except Exception as ex:
            dropin = {"value": None, "error": str(ex)[:300]}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        hbm = float(peaks["hbm_gbs"])
        kern = finish(kernels_of(per, c, M, layers), hbm)
        dom = max((k for k in kern if k != "eval_field"), key=lambda k: kern[k]["ms"])
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # dram bytes per launch from the committed ncu --set full capture
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("%s@%d" % (args.workload, n), {}).get(dom)
            except Exception:
                traffic = None
        C_r, A_r, T_r = float(c.cubes), float(c.active), float(c.triangles)
        survey_bytes = 6.0 * C_r + 40.0 * A_r + 96.0 * T_r  # SURVEY.md §8(d) classify+scan+emit accounting
        pipe_ms = per["ms_classify"] + per["ms_emit"]
        out = {
            "metric": "Gvoxels/s", "value": value, "unit": "Gvoxels/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "mtriangles_per_s": tris / (ms_per_step * 1e-3) / 1e6,
            "config": {"workload": "%s %s at %d^3 (step 2/%d, M=%d cubes/axis), iso 0, scale 1, positions+gradient normals, field mode auto (block-field), z-slabs over %d GPU(s)" % (
                args.workload, eq, n, n, M, world), "cubes": cubes, "triangles": tris, "active_cubes": active,
                "field_mode": "block-field (interval proof per 32x4x4 vertex block, decided within the call)" if c.field_mode == mcb.FIELD_SPARSE else "dense",
                "slab_cuts": slabs,
                "l2": "nothing is read back between steps; every step re-derives classes, field blocks, records and writes the whole soup (%.2f GB per GPU, "
                      "larger than L2)" % (96.0 * T_r / 1e9),
                "timing": "CUDA events on the launching stream, max over ranks"},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["GBps"], "peak": hbm, "unit": "GB/s",
                         "frac": kern[dom]["frac_of_hbm_peak"], "traffic": traffic, "peak_source": peak_src,
                         "kernels": kern,
                         "field_write_kernel": ({"GBps": variants["dense_field"]["eval_GBps"], "frac": variants["dense_field"]["eval_GBps"] / hbm,
                                                 "ms": variants["dense_field"]["ms_eval"]} if "dense_field" in variants else None),
                         "classify_scan_emit_vs_survey_bytes": {"bytes": survey_bytes, "ms": pipe_ms,
                                                                "GBps": survey_bytes / (pipe_ms * 1e-3) / 1e9,
                                                                "frac": survey_bytes / (pipe_ms * 1e-3) / 1e9 / hbm}},
            "e2e": {"value": cubes / (idx_ms * 1e-3) / 1e9, "unit": "Gvoxels/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": e2e["indexed"]["d2h_bytes_per_step"], "ms_per_step": idx_ms, "steps": e2e["indexed"]["steps"],
                    "what": "equation text in -> Poly_Data on the host (welded vertex_list + tri_list + per-vertex normals), MCB_MESH_INDEXED, through the ctypes mirror of the C ABI",
                    "poly_data_only": {"value": cubes / (e2e["poly_data_only"]["ms_per_step"] * 1e-3) / 1e9, **e2e["poly_data_only"],
                                       "what": "same without the per-vertex normals: exactly the Poly_Data the reference's recalculate() leaves"},
                    "soup": {"value": cubes / (e2e["soup"]["ms_per_step"] * 1e-3) / 1e9, **e2e["soup"],
                             "what": "same, float4 triangle soup + float4 normals out (MCB_MESH_SOUP)"},
                    "dropin": dropin},
            "changed_param": changed, "first_call": first_call,
            "workloads": workloads, "strong_2048": strong,
            "variants": variants,
            "gpu_launches": int(sum_over_ranks([headline_launches])[0]) if world == 1 else None, "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                threads = os.cpu_count() or 1
                gv, mt, sample, sec = cpu_reference_rate(eq, 2.0 / n, args.cpu_seconds, threads)
                out["cpu_baseline"] = {"value": gv, "unit": "Gvoxels/s", "cores": threads, "kind": "reference", "sample": sample,
                                       "mtriangles_per_s": mt, "seconds": sec}
            except Exception as ex:  # the oracle is test infrastructure: its absence must not fail the product bench
                out["cpu_baseline"] = {"value": None, "unit": "Gvoxels/s", "cores": os.cpu_count(), "kind": "reference", "sample": "unavailable: %s" % ex}
    if world > 1:  # every rank takes part in the collectives above
        gl = sum_over_ranks([headline_launches])[0]
        if rank == 0:
            out["gpu_launches"] = int(gl)
    if rank == 0:
        emit_line(out)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    # stdout carries exactly one line, the JSON: whatever a library prints there (NCCL's version banner, a warning) is sent
    # to stderr instead, and the line is written to the saved descriptor at the end
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sphere", choices=sorted(WORKLOADS))
    ap.add_argument("--base-res", type=int, default=1024)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the 2048^3 strong-scaling block")
    ap.add_argument("--no-dropin", action="store_true", help="skip the C++ drop-in (mcb_headless) end-to-end number")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's last timed step (triangle soup, counts) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
