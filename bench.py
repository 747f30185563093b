#!/usr/bin/env python
"""Benchmark of the APAP hot path on B200 (BASELINE.json metric: moving-DLT cells/s and mesh-warp
Mpix/s vs roofline, beside the reference's CPU path timed on the same box).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic pair.  Two stages are timed, each for
exactly K steps after W warm-up steps (at least 3), on the device with CUDA events, with the L2 flushed (a
256 MiB write) before every step (the side measurements below -- global warp, spectral weighting, matcher,
c4 / c5 -- run K timed steps after W warm-up steps too):
  * moving DLT  = K1 (weights + Gram contraction) + K2 (9x9 Jacobi + de-normalise)  -> cells/s
    (the headline ``value``; ``ms_per_step`` is this stage)
  * mesh warp   = K3 (`local_warp`), plus K4 blend and the fused warp+blend          -> Mpix/s
    (reported under ``"warp"``)
N = 1 runs BASELINE config c2 (4K pair, 5k keypoints, 200x200 grid).  N > 1 (under torchrun, one
rank per GPU): every rank runs its own c2-shaped pair (independent pairs, no data-path collective,
"scaling": "weak"), and the c3 pass (8K, 20k keypoints, 400x400) is additionally run strong-scaled
-- cell rows and canvas row bands sharded, NCCL all-gather to assemble the panorama -- and
reported under ``"c3_sharded"``.  Times are max over ranks.  Prints ONE JSON line on rank 0.

``--dump-outputs DIR`` writes, after the timed steps, what each timed path of rank 0 computed in its last step as
``DIR/<name>.npy`` (see ``OutputDump``).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
sys.dont_write_bytecode = True          # the tree may be read-only: the bench writes nothing into it

METRIC = "apap_moving_dlt_cells_per_s"
UNIT = "cells/s"


def _peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def _ncu_traffic(name):
    """DRAM bytes (read + write) per launch of each kernel from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py); {} when there is none for this workload."""
    path = os.path.join(REPO, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(name, {})
    return {}


# ----------------------------------------------------------------------------- clock sampling
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed regions run."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.terminate)      # the sampler never outlives the bench, even one that fails
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for _, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        busy = [v for v in sm if mx and v > 0.5 * mx] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ CPU baselines
# The reference's own CPU implementation of the path on the box's host cores.  When ``oracle/_ref/pyviz`` holds the
# reference's scripts (oracle/make_ref.py, run by build() in the build container) the workers call the REAL
# ``APAP.local_homography`` / ``APAP.local_warp`` of pyviz/apap.py (kind "reference"); otherwise the oracle's
# restatement of the same per-cell loop (kind "port").  One persistent pool of worker processes, every worker builds
# its scene once; only the workers' compute loop is inside the timed wall.
_REF = {}


def _ref_init(name):
    """Pool initialiser: the scene, the reference module (or the port) and an H grid for the warp sample."""
    import contextlib
    import io
    from cvx_proj_b200 import synth
    from oracle import apap_oracle as orc
    from oracle import make_ref
    sc = synth.make_scene(name)
    with contextlib.redirect_stdout(io.StringIO()):
        ref = make_ref.load()
    _REF.update(sc=sc, ref=ref, orc=orc, img=None, h_rows=None)


def _ref_cells(rows):
    """``local_homography`` on the cell rows ``rows`` (a slice of the vertex grid): seconds of compute."""
    sc, ref, orc = _REF["sc"], _REF["ref"], _REF["orc"]
    verts = np.ascontiguousarray(sc.vertices[rows[0]:rows[1]])
    t0 = time.perf_counter()
    if ref is not None:
        st = ref.APAP(sc.gamma, sc.sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y])
        st.local_homography(sc.src, sc.dst, verts)
    else:
        orc.local_homography_svd(sc.src, sc.dst, verts, sc.gamma, sc.sigma)
    return time.perf_counter() - t0


def _ref_warp(n_rows):
    """``local_warp`` on the first ``n_rows`` canvas rows (the cell rows they touch): seconds of compute."""
    import contextlib
    import io
    sc, ref, orc = _REF["sc"], _REF["ref"], _REF["orc"]
    if _REF["img"] is None:
        _REF["img"] = sc.image(1)
        k = int(np.searchsorted(sc.mesh[1], n_rows, side="left")) + 1          # cell rows under the sampled canvas rows
        sub = np.ascontiguousarray(sc.vertices[:k, ::max(1, sc.mesh_cells // 8)])
        h_small = orc.local_homography_gram64(sc.src, sc.dst, sub, sc.gamma, sc.sigma)
        reps = -(-sc.mesh_cells // h_small.shape[1])
        _REF["h_rows"] = np.repeat(h_small, reps, 1)[:, :sc.mesh_cells].astype(np.float32).copy()
    img, h = _REF["img"], _REF["h_rows"].copy()
    t0 = time.perf_counter()
    if ref is not None:
        st = ref.APAP(sc.gamma, sc.sigma, [sc.final_w, n_rows], [sc.offset_x, sc.offset_y])
        with contextlib.redirect_stdout(io.StringIO()):
            st.local_warp(img, h, sc.mesh)
    else:
        orc.local_warp(img, orc.invert_grid(h), sc.mesh, (sc.final_w, n_rows), (sc.offset_x, sc.offset_y))
    return time.perf_counter() - t0


class ReferencePool:
    """``procs`` worker processes holding the workload's scene; ``dlt(rows_per_proc)`` / ``warp(n_rows)`` time one
    bounded sample each (wall clock around the pool call, the workers only compute)."""

    def __init__(self, name, procs):
        import multiprocessing as mp
        from cvx_proj_b200 import synth
        from oracle import make_ref
        self.name, self.procs = name, procs
        self.cfg = synth.CONFIGS[name]
        self.kind = "reference" if all(os.path.exists(os.path.join(make_ref.DST, f)) for f in make_ref.FILES) else "port"
        self.pool = mp.get_context("fork").Pool(procs, initializer=_ref_init, initargs=(name,))
        self.pool.map(_ref_cells, [(0, 0)] * procs)            # every worker is up and has its scene

    def close(self):
        self.pool.close()
        self.pool.join()

    def dlt(self, rows_per_proc):
        """Every worker solves ``rows_per_proc`` whole cell rows, the workers' rows spread evenly over the grid.
        Returns (cells, wall seconds)."""
        mesh = self.cfg["mesh"]
        rows_per_proc = max(1, min(rows_per_proc, mesh // self.procs))
        starts = np.linspace(0, mesh - rows_per_proc, self.procs).astype(int)
        t0 = time.perf_counter()
        self.pool.map(_ref_cells, [(int(a), int(a) + rows_per_proc) for a in starts])
        self.rows_used = rows_per_proc
        return self.procs * rows_per_proc * mesh, time.perf_counter() - t0

    def warp(self, seconds):
        """Every worker warps the first canvas rows (P identical samples, about ``seconds`` of wall at the reference's
        ~0.13 Mpix/s per process).  Returns (pixels, wall seconds)."""
        from cvx_proj_b200 import synth
        sc = synth.make_scene(self.name)
        n_rows = self.warp_rows = int(max(2, min(sc.final_h, seconds * 0.13e6 / sc.final_w)))
        t0 = time.perf_counter()
        self.pool.map(_ref_warp, [n_rows] * self.procs)
        return self.procs * n_rows * sc.final_w, time.perf_counter() - t0

    def describe(self):
        if self.kind == "reference":
            return ("the reference itself (oracle/_ref/pyviz/apap.py, unmodified): APAP.local_homography on disjoint "
                    f"cell-row slices in {self.procs} worker processes")
        return (f"oracle port of the reference's per-cell weighted-SVD loop (cv.SVDecomp float64) in {self.procs} "
                "worker processes (oracle/_ref absent)")


def _rows_for_seconds(pool, seconds):
    """Cell rows per worker for about ``seconds`` of wall per step, from one timed row per worker on this box."""
    _, wall = pool.dlt(1)
    return max(1, int(seconds / max(wall, 1e-3)))


def _config(name, world):
    """The ``config`` object of the bench line: the same for both arms."""
    return {"workload": _workload_desc(name), "per_rank": "one pair per GPU (independent pairs)" if world > 1 else "one pair",
            "l2": "GPU arm: flushed before every timed step (256 MiB write); CPU arm: n/a"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores, a bounded sample of the
    workload per step (persistent worker pool, scenes prebuilt: only the workers' loops are timed)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload or "c2"
    procs = os.cpu_count() or 1
    pool = ReferencePool(name, procs)
    rows = _rows_for_seconds(pool, 2.0)                           # ~2 s of wall per step
    walls, cells = [], 0
    for k in range(args.warmup + args.steps):
        cells, wall = pool.dlt(rows)
        if k >= args.warmup:
            walls.append(wall)
    wpx, wwall = pool.warp(1.0)
    pool.close()
    rows = pool.rows_used
    ms = 1e3 * float(np.mean(walls))
    value = cells / (ms * 1e-3)
    total = pool.cfg["mesh"] ** 2
    sample = f"{cells} of {total} cells of {name} per step ({rows} whole cell rows per worker, spread evenly); {pool.describe()}"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": _config(name, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": pool.kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "warp": {"metric": "apap_mesh_warp_mpix_per_s", "value": wpx / wwall / 1e6, "unit": "Mpix/s", "cores": procs,
                     "kind": pool.kind,
                     "sample": f"the first {pool.warp_rows} canvas rows of {name} in each of {procs} workers (APAP.local_warp's "
                               f"pixel loop and the per-cell inverses of the cell rows under them), {wwall:.1f} s wall"},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def _workload_desc(name):
    from cvx_proj_b200 import synth
    c = synth.CONFIGS[name]
    return (f"{name}: synthetic {c['width']}x{c['height']} pair, {c['n_kp']} matched keypoints, "
            f"APAP {c['mesh']}x{c['mesh']} grid, gamma=0.5 sigma=100")


# ----------------------------------------------------------------------------------- our arm
class Timer:
    def __init__(self, torch):
        self.torch = torch
        self.pairs = []

    def mark(self):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    @staticmethod
    def ms(a, b):
        return a.elapsed_time(b)


class Pass:
    """Device-resident state of one APAP pass (inputs already in HBM) + launch helpers."""

    def __init__(self, torch, device, name, seed=0, rows=None, gram_engine="tcgen05"):
        from cvx_proj_b200 import synth
        from cvx_proj_b200 import _runtime as rt
        from cvx_proj_b200.apap import APAP, cell_lookup_tables, scale_anchors, weight_scale
        self.torch, self.device, self.rt = torch, device, rt
        self.sc = sc = synth.make_scene(name, seed=seed)
        self.st = APAP(sc.gamma, sc.sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y], device=device,
                       gram_engine=gram_engine)
        self.lib = rt.load_library()
        m = sc.mesh_cells
        self.row0, self.row1 = rows if rows is not None else (0, m)          # owned cell rows
        verts = sc.vertices[self.row0:self.row1]
        self.cells = verts.shape[0] * verts.shape[1]
        cf1, cf2, tmats = self.st._condition(sc.src, sc.dst)                 # the O(N) host prologue of the public call
        self.engine = rt.GRAM_TCGEN05 if self.st.gram_engine == "tcgen05" else rt.GRAM_FFMA2
        points = np.ascontiguousarray(np.stack([cf1, cf2, sc.src])[:, None], dtype=np.float32)
        self.points = torch.from_numpy(points).to(device)                    # what the public call uploads
        self.rows = self.st.kp_rows_device(self.points)                      # keypoint row table, built on the device
        self.n_pad = self.rows.shape[1]
        self.table = self.st.kp_table_device(self.rows)[0]                   # the engine's table (blocks for tcgen05)
        self.anchors = torch.from_numpy(scale_anchors(verts, weight_scale(sc.sigma))).to(device)
        self.tmats = torch.from_numpy(tmats).to(device)
        self.t_bound = self.st.weight_bound_device(self.points[2], None, self.anchors[None])   # as the public call does
        self.k_splits, self.cells_padded, nbytes = rt.gram_plan(self.cells, self.n_pad, self.engine)
        self.partials = torch.empty(nbytes // 4, dtype=torch.float32, device=device)
        self.h_out = torch.empty((self.cells, 9), dtype=torch.float32, device=device)
        self.g2 = float(np.float32(float(sc.gamma) ** 2))
        self.col_cell, self.row_cell = cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, m, m)
        self.stream = rt.stream_ptr(torch, device)

    # -- moving DLT
    def gram(self):
        self.rt.check(self.lib.apap_gram_partials(self.table.data_ptr(), self.anchors.data_ptr(), 1, self.cells,
                                                  self.n_pad, self.g2, self.engine, self.t_bound.data_ptr(),
                                                  self.partials.data_ptr(), self.stream), "gram")

    def dlt(self, overlap=True):
        """K1 + K2 as the public call launches them (K2 a programmatic dependent of K1 when ``overlap``)."""
        self.st.local_homography_device(self.table[None], self.anchors[None], self.tmats[None], 1, self.cells,
                                        out_h=self.h_out[None] if self.h_out.dim() == 2 else self.h_out,
                                        partials=self.partials, overlap=overlap, t_bound=self.t_bound)

    def eig(self):
        self.rt.check(self.lib.apap_eig_denorm(self.partials.data_ptr(), self.tmats.data_ptr(), 1, self.cells,
                                               self.k_splits, self.rt.EIG_AUTO, self.h_out.data_ptr(), None, self.stream),
                      "eig")

    # -- warp
    def prepare_warp(self, px_rows=None):
        """Upload the image, the inverted grid rows and the lookup tables (outside the timed region)."""
        from cvx_proj_b200 import synth
        torch, sc = self.torch, self.sc
        self.torch.cuda.synchronize()
        m = sc.mesh_cells
        h = np.tile(np.eye(3, dtype=np.float32), (m, m, 1, 1))
        h[self.row0:self.row1] = self.h_out.cpu().numpy().reshape(-1, m, 3, 3)
        inv = np.linalg.inv(h).astype(np.float32)
        img = sc.image(1)
        centre = synth.make_image(sc.width, sc.height, seed=2)
        self.px_rows = px_rows if px_rows is not None else (0, sc.final_h)
        self.tables = self.st.warp_tables_device(inv, self.col_cell, self.row_cell, sc.width, sc.height, self.device,
                                                 self.px_rows[0], self.px_rows[1])
        self.flagged_cells = self.tables.exact_cells_frac()
        self.img = torch.from_numpy(img).to(self.device)
        self.centre = torch.from_numpy(centre).to(self.device)
        n = self.px_rows[1] - self.px_rows[0]
        self.canvas = torch.empty((n, sc.final_w, 3), dtype=torch.uint8, device=self.device)
        self.canvas2 = torch.empty_like(self.canvas)
        self.pasted = torch.zeros_like(self.canvas)
        self.host_img, self.host_centre = img, centre

    def warp(self, fused=False, legacy=False):
        self.st.warp_device(self.img, self.tables, self.sc.mesh_cells, centre_dev=self.centre if fused else None,
                            out=self.canvas, legacy=legacy)

    def blend(self):
        self.rt.blend_device(self.torch, self.canvas, self.pasted, out=self.canvas2)


class OutputDump:
    """``--dump-outputs DIR``: the arrays a caller of each timed path receives from its last timed step, written as
    ``DIR/<name>.npy`` in float32 (float32 results, uint8 images) or float64 (float64 and integer results).  An array
    larger than ``ARRAY_BYTES`` keeps a fixed seeded sample of its rows (first axis), the same rows in every run of
    the same shape, so that the 20 or so arrays stay under 64 MB in all.  ``path`` None: nothing is kept.
    Two runs of the same build give the same bits everywhere but in ``spectral_segment``: the power iteration sums
    its norm with float64 atomics, so its last bits vary from run to run (4e-16 apart in two runs on a B200)."""

    ARRAY_BYTES = 3 << 20
    TOTAL_BYTES = 64 * 10 ** 6

    def __init__(self, path):
        self.path, self.arrays = path, {}

    def add(self, name, value):
        if self.path is None:
            return
        a = value.cpu().numpy() if hasattr(value, "cpu") else np.asarray(value)
        dtype = np.float32 if a.dtype == np.float32 or a.dtype.itemsize <= 2 else np.float64
        keep = self.ARRAY_BYTES // (a[:1].size * np.dtype(dtype).itemsize)
        if a.shape[0] > keep:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        self.arrays[name] = a.astype(dtype)

    def write(self):
        if self.path is None:
            return
        total = sum(a.nbytes for a in self.arrays.values())
        if total > self.TOTAL_BYTES:
            raise RuntimeError(f"--dump-outputs: {total} bytes exceed {self.TOTAL_BYTES}")
        os.makedirs(self.path, exist_ok=True)
        for name, a in self.arrays.items():
            np.save(os.path.join(self.path, name + ".npy"), a)
        print(f"bench: {len(self.arrays)} outputs ({total / 1e6:.1f} MB) -> {self.path}", file=sys.stderr)


def timed_steps(torch, flush, warmup, steps, body, n_marks):
    """Run ``body(mark)`` warmup+steps times; ``body`` calls ``mark()`` n_marks times.  Returns the
    per-interval mean milliseconds over the timed steps (list of n_marks-1 floats)."""
    all_marks = []
    for k in range(warmup + steps):
        flush.add_(1)                       # 256 MiB write: evicts the 126 MB L2
        marks = []
        body(lambda: marks.append(_ev(torch)))
        if k >= warmup:
            all_marks.append(marks)
    torch.cuda.synchronize()
    sums = [0.0] * (n_marks - 1)
    for marks in all_marks:
        for i in range(n_marks - 1):
            sums[i] += marks[i].elapsed_time(marks[i + 1])
    return [s / steps for s in sums]


def _ev(torch):
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from cvx_proj_b200 import _runtime as rt
    from cvx_proj_b200 import sharding, synth

    peaks, peak_src = _peaks()
    name = args.workload or "c2"
    K, W = args.steps, max(args.warmup, 3)
    flush = torch.zeros(256 << 20, dtype=torch.uint8, device=device)
    launches = 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    fp32_peak = rt.fp32_peak_tflops(device)
    mufu_peak = rt.pipe_peak(rt.PROBE_MUFU, device) / 1e12                    # Tlane-op/s
    p = Pass(torch, device, name, seed=rank, gram_engine=args.gram_engine)
    sc = p.sc
    dump = OutputDump(args.dump_outputs if rank == 0 else None)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- stage 1: moving DLT (K1 + K2) ---------------------------------------------------------
    def dlt_body(mark):
        mark(); p.gram(); mark(); p.eig(); mark()
    barrier()
    t_gram, t_eig = timed_steps(torch, flush, W, K, dlt_body, 3)        # K1, K2 timed one by one (roofline attribution)
    barrier()
    (t_dlt,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.dlt(), mark()), 2)   # the stage as the public call launches it
    dump.add("h", p.h_out.reshape(-1, sc.mesh_cells, 3, 3))
    barrier()
    launches += 4 * K
    ms_dlt = max_over_ranks(t_dlt)
    ms_gram = max_over_ranks(t_gram)
    ms_eig = max_over_ranks(t_eig)
    cells_total = p.cells * world
    value = cells_total / (ms_dlt * 1e-3)

    # ---- stage 2: mesh warp (K3), blend (K4), fused K3+K4 -------------------------------------
    p.prepare_warp()
    barrier()
    (t_warp,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.warp(False), mark()), 2)
    dump.add("warp", p.canvas)
    (t_strip,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.warp(False, legacy=True), mark()), 2)
    dump.add("warp_strip", p.canvas)
    (t_fused,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.warp(True), mark()), 2)
    dump.add("warp_blend", p.canvas)
    (t_blend,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.blend(), mark()), 2)
    dump.add("blend", p.canvas2)
    barrier()
    launches += 4 * K
    ms_warp, ms_fused, ms_blend, ms_strip = (max_over_ranks(t) for t in (t_warp, t_fused, t_blend, t_strip))
    canvas_px = sc.canvas_px
    src_px = sc.width * sc.height
    warp_bytes = 3 * canvas_px + 3 * src_px                       # SURVEY.md 8d: write canvas once + read source once
    fused_bytes = 3 * canvas_px + 3 * src_px + 3 * src_px
    blend_bytes = 9 * canvas_px
    hbm = peaks["hbm_gbs"]

    # ---- global-homography warp (SURVEY 8f row N4: utils.image_warping = cv.warpPerspective + paste / mean blend)
    from cvx_proj_b200 import utils as putils
    g_cw, g_ch, g_tx, g_ty, g_m = putils.warping_canvas(p.host_img.shape, p.host_img.shape, sc.h_gt)
    g_out = torch.empty((g_ch, g_cw, 3), dtype=torch.uint8, device=device)
    g_times = {}
    for g_name, g_mode in (("warp_only", 0), ("paste", 1), ("mean_blend", 2)):
        (g_t,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), putils.warp_perspective(
            p.img, g_m, (g_cw, g_ch), base=p.centre, offset=(g_tx, g_ty), mode=g_mode, out=g_out), mark()), 2)
        dump.add("global_" + g_name, g_out)
        g_times[g_name] = max_over_ranks(g_t)
    launches += 3 * K
    barrier()

    # ---- spectral match weighting (SURVEY 8f row N4: calculate_M = N x N affinity matrix + leading singular vector)
    from cvx_proj_b200 import spectral_method as psm
    sp_n = 2500
    sp_rng = np.random.default_rng(7)
    sp_o, sp_c, _ = synth.make_keypoints(1024, 768, sp_n, seed=11)
    sp_c = sp_c.copy()
    sp_bad = sp_rng.random(sp_n) < 0.3
    sp_c[sp_bad] += sp_rng.normal(0, 60, (int(sp_bad.sum()), 2)).astype(np.float32)
    sp_diag = 0.9 + 0.1 * sp_rng.random(sp_n)
    sp_times = []
    for k in range(W + K):
        torch.cuda.synchronize()
        sp_t0 = time.perf_counter()
        sp_seg, sp_info = psm.spectral_segment_device(sp_c, sp_o, sp_diag, 30.0, device=device, return_info=True)
        torch.cuda.synchronize()
        if k >= W:
            sp_times.append((time.perf_counter() - sp_t0) * 1e3)
    sp_ms = float(np.mean(sp_times))
    dump.add("spectral_segment", sp_seg)
    launches += (W + K) * (1 + sp_info["iterations"] + sp_info["iterations"] // 16)   # k_affinity, k_power_step per step, k_power_diff per 16

    # ---- e2e through the public API: pinned host buffers in, host arrays out -------------------
    src_pin = rt.pinned_empty(sc.src.shape, np.float32); src_pin[...] = sc.src
    dst_pin = rt.pinned_empty(sc.dst.shape, np.float32); dst_pin[...] = sc.dst
    img_pin = rt.pinned_empty(p.host_img.shape, np.uint8); img_pin[...] = p.host_img
    vert_pin = rt.pinned_empty(sc.vertices.shape, np.float64); vert_pin[...] = sc.vertices
    st = p.st
    e2e_dlt, e2e_warp = [], []
    h_host = None
    for k in range(W + K):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h_host, _ = st.local_homography(src_pin, dst_pin, vert_pin)
        t1 = time.perf_counter()
        warped = st.local_warp(img_pin, h_host, sc.mesh)
        t2 = time.perf_counter()
        if k >= W:
            e2e_dlt.append(t1 - t0)
            e2e_warp.append(t2 - t1)
    dump.add("e2e_h_inverted", h_host)                # local_warp leaves the per-cell inverses in the caller's grid
    dump.add("e2e_warp", warped)
    # k_scale_anchors, k_condition, k_condition_mats, k_kp_rows, k_weight_bound, k_kp_blocks, k_gram_tc, k_eig;
    # k_inv_grid, k_warp_prep, k_tile_prep, k_warp_tile
    launches += 12 * K
    e2e_dlt_s = max_over_ranks(float(np.mean(e2e_dlt)))
    e2e_warp_s = max_over_ranks(float(np.mean(e2e_warp)))
    h2d_dlt = 2 * sc.src.shape[0] * 8 + p.cells * 16              # raw source and target points (float32), anchor points (float64)
    d2h_dlt = p.cells * 36
    h2d_warp = 3 * src_px + p.cells * 36 + 8 * sc.final_w + 8 * p.tables.n_blocks + 16 * sc.mesh_cells   # image, grid (inverted on the device), LUTs
    d2h_warp = 3 * canvas_px + p.cells * 37                      # canvas + the inverted grid and its flags

    # ---- c3 strong-scaled across ranks (cell rows + row bands, one all-gather) -----------------
    c3 = None
    if args.c3 and (world > 1 or args.c3 == "always"):
        c3 = run_c3_sharded(torch, dist, device, rank, world, flush, W, K, max_over_ranks, barrier, dump, args.gram_engine)
        launches += c3.pop("_launches")

    extras = None
    if world == 1 and not args.no_extras:
        extras = run_c4_c5(torch, device, flush, mufu_peak * 1e12, W, K, dump)
        launches += extras.pop("_launches")
        extras["matcher"] = run_matcher(torch, device, flush, fp32_peak, W, K, dump)
        launches += extras["matcher"].pop("_launches")

    clocks = sampler.stop() if rank == 0 else None
    dump.write()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline (rank 0, N = 1 only): bounded samples of the same workload ---------------
    cpu = None
    if world == 1 and not args.no_cpu:
        procs = os.cpu_count() or 1
        pool = ReferencePool(name, procs)
        rows = _rows_for_seconds(pool, 2.0)                         # the reference arm's step, five times: ~10 s of CPU work
        n_cells, wall = 0, 0.0
        for _ in range(5):
            c, w = pool.dlt(rows)
            n_cells, wall = n_cells + c, wall + w
        wpx, wwall = pool.warp(3.0)
        pool.close()
        rows = pool.rows_used
        cpu = {"value": n_cells / wall, "unit": UNIT, "cores": procs, "kind": pool.kind,
               "sample": (f"5 x {n_cells // 5} of {sc.n_cells} cells of {name} ({rows} whole cell rows per worker, spread evenly), "
                          f"{pool.describe()}, {wall:.1f} s wall"),
               "warp": {"value": wpx / wwall / 1e6, "unit": "Mpix/s", "cores": procs, "kind": pool.kind,
                        "sample": f"the first {pool.warp_rows} canvas rows of {name} in each of {procs} workers (APAP.local_warp), "
                                  f"{wwall:.1f} s wall"}}

    pairs = float(p.n_pad) * p.cells                                          # (cell, keypoint) pairs per launch
    gram_flops = 2.0 * 24 * pairs
    gram_s = ms_gram * 1e-3
    fp32_equiv = {"achieved": gram_flops / gram_s / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                  "frac": gram_flops / gram_s / 1e12 / fp32_peak,
                  "what": "2*24*n_kp_padded*cells flop of the 24-term contraction against the FP32 FFMA probe"}
    traffic = _ncu_traffic(name)
    if args.gram_engine == "tcgen05":
        tf32_peak = peaks["bf16_tflops"] / 2.0                                  # dense TF32 = half the bf16 rate
        mma_flops = 2.0 * 128 * 8 * (64 + 32) * (p.n_pad / 8) * math.ceil(p.cells / 128)   # N=64 + N=32 MMAs per block
        roof = {"kernel": "k_gram_tc", "bound": "xu",
                "achieved": 2.0 * pairs / gram_s / 1e12, "peak": mufu_peak, "unit": "Tlane-op/s",
                "frac": 2.0 * pairs / gram_s / 1e12 / mufu_peak, "traffic": next((v for k, v in traffic.items() if k.startswith("k_gram_tc")), None),
                "peak_source": "MUFU.EX2 probe kernel timed in this run (MEASURED_PEAKS.json has no XU figure); it equals the "
                               "nominal 148 SM x 16 lanes x SM clock",
                "algorithmic": "2 transcendental evaluations (sqrt, exp2) per (cell, keypoint) pair, the XU pipe's work in "
                               "the plain kernel; the contraction itself runs on the tensor pipe",
                "executed_mufu_per_pair": 1.5 if sc.gamma >= 0.5 else 2.0,
                "executed_note": "for gamma >= 0.5 half of the exp2 are evaluated by a degree-7 polynomial on the FMA "
                                 "pipe, so the XU pipe itself is busy achieved * 0.75 / peak",
                "tensor": {"achieved": mma_flops / gram_s / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                           "frac": mma_flops / gram_s / 1e12 / tf32_peak,
                           "what": "executed TF32 MMA flop (3xTF32, N padded to 32) against bf16_tflops / 2 "
                                   "of MEASURED_PEAKS.json"},
                "fp32_equivalent": fp32_equiv, "ms": ms_gram, "eig_ms": ms_eig,
                "fractions": {"xu_algorithmic": 2.0 * pairs / gram_s / 1e12 / mufu_peak,
                              "xu_executed": (1.5 if sc.gamma >= 0.5 else 2.0) * pairs / gram_s / 1e12 / mufu_peak,
                              "tensor_executed_tf32": mma_flops / gram_s / 1e12 / tf32_peak,
                              "tensor_algorithmic_24_terms": gram_flops / gram_s / 1e12 / tf32_peak,
                              "fp32_equivalent": fp32_equiv["frac"]},
                "stage_note": "ms / eig_ms: K1 and K2 launched and timed one by one; the stage (ms_per_step, value) is the "
                              "public call's launch, K2 a programmatic dependent of K1 that starts on finished cell tiles"}
    else:
        roof = {"kernel": "k_gram", "bound": "fp32_fma", "achieved": fp32_equiv["achieved"], "peak": fp32_peak,
                "unit": "TFLOP/s", "frac": fp32_equiv["frac"], "traffic": traffic.get("k_gram"),
                "peak_source": "FP32 FFMA probe kernel timed in this run (not in MEASURED_PEAKS.json)",
                "algorithmic": "2*24*n_kp_padded*cells flop per launch (24 executed terms)",
                "ms": ms_gram, "eig_ms": ms_eig}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_dlt, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32x3+f32" if args.gram_engine == "tcgen05" else "f32", "data": "synthetic",
        "config": _config(name, world),
        "setup": {"cells": p.cells, "n_kp_padded": p.n_pad, "k_splits": p.k_splits, "canvas": [sc.final_w, sc.final_h],
                  "gram_engine": args.gram_engine},
        "roofline": roof,
        "e2e": {"value": cells_total / e2e_dlt_s, "unit": UNIT, "h2d_bytes_per_step": h2d_dlt,
                "d2h_bytes_per_step": d2h_dlt, "ms_per_step": e2e_dlt_s * 1e3,
                "call": "APAP.local_homography(src, dst, vertices) with pinned numpy inputs (points float32, vertices float64), numpy H out; one library call enqueues the whole chain"},
        "warp": {
            "metric": "apap_mesh_warp_mpix_per_s", "value": world * canvas_px / (ms_warp * 1e-3) / 1e6, "unit": "Mpix/s",
            "ms_per_step": ms_warp, "dtype": "u8",
            "roofline": {"kernel": "k_warp_tile", "bound": "hbm", "achieved": warp_bytes / (ms_warp * 1e-3) / 1e9,
                         "peak": hbm, "unit": "GB/s", "frac": warp_bytes / (ms_warp * 1e-3) / 1e9 / hbm,
                         "traffic": next((v for k, v in traffic.items() if k.startswith("k_warp_tile")), None),
                         "peak_source": peak_src, "algorithmic": "3*canvas_px + 3*src_px bytes per launch",
                         "strip_kernel_ms": ms_strip,
                         "note": "tile engine (tensor-map TMA source boxes in shared memory, LDS gathers, TMA row stores); "
                                 "strip_kernel_ms = round 1's kernel on the same tables in the same run"},
            "fused_warp_blend": {"ms_per_step": ms_fused, "mpix_per_s": canvas_px / (ms_fused * 1e-3) / 1e6,
                                 "hbm_frac": fused_bytes / (ms_fused * 1e-3) / 1e9 / hbm},
            "blend": {"ms_per_step": ms_blend, "mpix_per_s": canvas_px / (ms_blend * 1e-3) / 1e6,
                      "hbm_frac": blend_bytes / (ms_blend * 1e-3) / 1e9 / hbm},
            "e2e": {"value": world * canvas_px / e2e_warp_s / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": h2d_warp,
                    "d2h_bytes_per_step": d2h_warp, "ms_per_step": e2e_warp_s * 1e3,
                    "call": "APAP.local_warp(img, H, mesh) with a pinned numpy image, numpy canvas out "
                            "(includes the in-place per-cell inverse of pyviz/apap.py:201-203: certified GPU inverse kept on the device for the warp and copied back into the caller's array, numpy for the cells it flags)"},
            "exact_path_cells_frac": p.flagged_cells,
        },
        "global_warp": {
            "what": "utils.image_warping of the reference's README pipeline (SURVEY 8f N4): bilinear cv.warpPerspective "
                    "semantics (bit-exact with OpenCV's 8-bit fixed-point path) fused with the paste / mean blend",
            "canvas": [g_cw, g_ch],
            "ms_per_step": g_times,
            "mpix_per_s": {k: world * g_cw * g_ch / (v * 1e-3) / 1e6 for k, v in g_times.items()},
            "hbm_frac_warp_only": (3 * g_cw * g_ch + 3 * src_px) / (g_times["warp_only"] * 1e-3) / 1e9 / hbm,
        },
        "spectral": {
            "what": "calculate_M of the reference's README pipeline (SURVEY 8f N4): affinity matrix over the matches "
                    "(bit-identical to the reference's) + float64 power iteration for |U[:, 0]| of its SVD",
            "matches": sp_n, "ms_host_to_host": sp_ms, "power_steps": sp_info["iterations"],
            "note": "np.linalg.svd of the same 2500 x 2500 matrix takes ~4 s on the build container's CPU",
        },
        "cpu_baseline": cpu,
        "clocks": clocks,
        "gpu_launches": launches,
    }
    if c3 is not None:
        line["c3_sharded"] = c3
    if extras is not None:
        line["c4_batch"] = extras["c4"]
        line["c5_sweep"] = extras["c5"]
        line["matcher"] = extras["matcher"]
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_c3_sharded(torch, dist, device, rank, world, flush, W, K, max_over_ranks, barrier, dump, gram_engine="tcgen05"):
    """BASELINE config c3 split over the ranks: cell rows [m0, m1) and the canvas rows they own per
    rank, keypoints and source image replicated, one NCCL all-gather of the row bands."""
    from cvx_proj_b200 import sharding
    from cvx_proj_b200.apap import cell_lookup_tables
    from cvx_proj_b200 import synth
    cfg = synth.CONFIGS["c3"]
    sc0 = synth.make_scene("c3")
    col, row = cell_lookup_tables(sc0.mesh, sc0.final_w, sc0.final_h, cfg["mesh"], cfg["mesh"])
    shards = sharding.plan_shards(row, cfg["mesh"], world)
    me = shards[rank]
    p = Pass(torch, device, "c3", seed=0, rows=(me.cell_row0, me.cell_row1), gram_engine=gram_engine)

    def dlt_body(mark):
        mark(); p.gram(); mark(); p.eig(); mark()
    barrier()
    t_gram, t_eig = timed_steps(torch, flush, W, K, dlt_body, 3)
    barrier()
    (t_dlt,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.dlt(), mark()), 2)
    dump.add("c3_h", p.h_out.reshape(-1, cfg["mesh"], 3, 3))
    barrier()
    p.prepare_warp(px_rows=(me.px_row0, me.px_row1))
    barrier()
    (t_warp,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), p.warp(False), mark()), 2)
    dump.add("c3_warp", p.canvas)
    barrier()
    t_gather = 0.0
    if world > 1:
        def gather_body(mark):
            mark(); sharding.gather_bands(p.canvas, shards, sc0.final_w); mark()
        (t_gather,) = timed_steps(torch, flush, W, K, gather_body, 2)
        barrier()
    # the panorama assembled by the warp kernel itself: row band stored into every GPU through the NVLS multicast mapping
    ms_fused, assembled_ok, assemble_variants = None, None, None
    if world > 1:
        try:
            sym = sharding.SymmetricPanorama(sc0.final_h, sc0.final_w, device)
        except Exception as exc:                     # no symmetric-memory support in this torch / on this box
            sym = None
            if rank == 0:
                print(f"bench: symmetric-memory panorama unavailable ({type(exc).__name__}: {exc})", file=sys.stderr)
        if sym is not None and sym.supported:
            own = sym.local[me.px_row0:me.px_row1]

            def fused_body(mark):
                mark()
                p.st.warp_device(p.img, p.tables, p.sc.mesh_cells, out=own)     # the band, straight into the panorama
                sym.broadcast_band(me.px_row0, me.px_row1)                      # ... and into everyone else's
                sym.barrier()
                mark()
            (t_fused,) = timed_steps(torch, flush, W, K, fused_body, 2)
            barrier()
            ms_bcast = max_over_ranks(t_fused)

            def direct_body(mark):
                mark()
                # ONE kernel: the tile engine stores its tiles' 384-byte rows straight into the multicast mapping
                p.st.warp_device(p.img, p.tables, p.sc.mesh_cells, multicast_ptr=sym.band_ptr(me.px_row0))
                sym.barrier()
                mark()
            sym.barrier()
            (t_direct,) = timed_steps(torch, flush, W, K, direct_body, 2)
            barrier()
            ms_direct = max_over_ranks(t_direct)
            ms_fused = min(ms_bcast, ms_direct)
            assemble_variants = {"warp_then_broadcast_kernel_ms": ms_bcast, "warp_kernel_multicast_stores_ms": ms_direct}
            # every band of this rank's panorama must be the band its owner warped (checksums travel over NCCL)
            def checksum(t):
                v = t.reshape(-1).to(torch.int64)
                return (v * (torch.arange(v.numel(), device=device, dtype=torch.int64) % 8191 + 1)).sum()
            sums = [torch.zeros((), dtype=torch.int64, device=device) for _ in range(world)]
            dist.all_gather(sums, checksum(p.canvas))
            same = all(bool(checksum(sym.local[s.px_row0:s.px_row1]) == sums[s.rank]) for s in shards)
            everyone = torch.tensor([int(same)], device=device)
            dist.all_reduce(everyone, op=dist.ReduceOp.MIN)
            assembled_ok = bool(everyone.item())
    ms_dlt = max_over_ranks(t_dlt)
    ms_warp = max_over_ranks(t_warp)
    ms_gather = max_over_ranks(t_gather)
    # the same pass on ONE GPU of this box in this run (every rank times the whole grid / canvas on its own GPU)
    one = {"dlt_ms": ms_dlt, "warp_ms": ms_warp}
    if world > 1:
        del p
        torch.cuda.empty_cache()
        pf = Pass(torch, device, "c3", seed=0, gram_engine=gram_engine)
        (t1_dlt,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), pf.dlt(), mark()), 2)
        pf.prepare_warp()
        (t1_warp,) = timed_steps(torch, flush, W, K, lambda mark: (mark(), pf.warp(False), mark()), 2)
        barrier()
        one = {"dlt_ms": max_over_ranks(t1_dlt), "warp_ms": max_over_ranks(t1_warp)}
    eff = {"dlt": one["dlt_ms"] / (world * ms_dlt), "warp": one["warp_ms"] / (world * ms_warp)}
    if ms_fused:
        eff["warp_and_assemble"] = one["warp_ms"] / (world * ms_fused)
    return {"workload": _workload_desc("c3"), "scaling": "strong", "n_gpus": world,
            "one_gpu_same_run": one, "efficiency_vs_1gpu": eff,
            "limiter": ("DLT: K1 is XU-bound and shards without exchange; the sharded grid has fewer cell tiles per SM wave. "
                        "Warp: the band kernel is a few tens of microseconds, launch latency and the fixed prologue do not shrink "
                        "with N. Assembly: every GPU receives (N-1)/N of the 124 MB panorama over NVLink whatever the method "
                        "(>= 150 us at the ~750 GB/s a B200 takes in)"),
            "cells_per_s": sc0.n_cells / (ms_dlt * 1e-3), "dlt_ms": ms_dlt, "gram_ms": max_over_ranks(t_gram),
            "warp_mpix_per_s": sc0.canvas_px / (ms_warp * 1e-3) / 1e6, "warp_ms": ms_warp,
            "allgather_ms": ms_gather, "allgather_bytes": 3 * sc0.canvas_px,
            "warp_and_assemble_ms": ms_fused, "warp_and_assemble_variants": assemble_variants,
            "assembled_panorama_verified_on_every_rank": assembled_ok,
            "warp_and_assemble_note": "warp into the rank's panorama (symmetric memory) + broadcast of the band into every "
                                      "other GPU's panorama (NVLS multimem.st kernel; a peer copy at 2 GPUs) + group barrier: "
                                      "replaces warp_ms + allgather_ms; null without NVSwitch multicast. Every GPU receives "
                                      "(N-1)/N of the panorama over NVLink either way",
            "shard": "cell rows + canvas row bands per rank; keypoints and source image replicated",
            "_launches": 5 * K + (3 * K if world > 1 else 0)}


def run_matcher(torch, device, flush, fp32_peak, W, K, dump):
    """SURVEY 8f row N3, matcher step: exact 1-NN of 4000 x 4000 SIFT-like descriptors (the c2 keypoint count after
    border rejection), device-resident and host to host, next to OpenCV's exact and FLANN matchers on this box's CPU."""
    import time
    from cvx_proj_b200.utils import match_descriptors
    rng = np.random.default_rng(0)
    nq = nt = 4000
    d = rng.gamma(0.6, 1.0, size=(nt, 128))
    train = np.minimum(np.rint(d / np.linalg.norm(d, axis=1, keepdims=True) * 512.0), 255.0).astype(np.float32)
    query = np.clip(train[rng.permutation(nt)] + rng.integers(-6, 7, size=(nq, 128)), 0, 255).astype(np.float32)
    q_dev, t_dev = torch.from_numpy(query).to(device), torch.from_numpy(train).to(device)
    ts = []
    for k in range(W + K):
        flush.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); match_descriptors(q_dev, t_dev); e1.record(); e1.synchronize()
        if k >= W:
            ts.append(e0.elapsed_time(e1))
    ms_dev = float(np.median(ts))
    t0 = time.perf_counter()
    for _ in range(K):
        idx, dist = match_descriptors(query, train)
    ms_host = (time.perf_counter() - t0) / K * 1e3
    dump.add("matcher_index", idx)
    dump.add("matcher_distance", dist)
    out = {"what": "exact 1-nearest-neighbour descriptor matching (apap_match_nn) = cv.BFMatcher(NORM_L2).match, bit-identical on "
                   "SIFT descriptors; the reference calls FLANN's approximate matcher (pyviz/utils.py:149-150)",
           "queries": nq, "train": nt, "dim": 128, "ms_device": ms_dev, "ms_host_to_host": ms_host,
           "pairs_per_s": nq * nt / (ms_dev * 1e-3),
           "fp32_frac": 3.0 * nq * nt * 128 / (ms_dev * 1e-3) / 1e12 / fp32_peak,
           "fp32_note": "3 flop (subtract, multiply, add) per component of a (query, train) pair on the packed FP32x2 pipe, "
                        "against the FFMA probe peak of this run", "_launches": (W + 2 * K) * 3}
    try:
        import cv2 as cv
        t0 = time.perf_counter(); cv.BFMatcher(cv.NORM_L2).match(query, train); ms_bf = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter(); cv.FlannBasedMatcher().match(query, train); ms_flann = (time.perf_counter() - t0) * 1e3
        out["cpu"] = {"cv_bfmatcher_ms": ms_bf, "cv_flann_ms": ms_flann, "threads": cv.getNumThreads()}
    except ImportError:
        out["cpu"] = None
    return out


def run_c4_c5(torch, device, flush, mufu_peak, W, K, dump):
    """BASELINE configs c4 (a batch of 64 1080p pairs, 2k keypoints, 100 x 100 grid, ONE launch of K1 + K2) and c5
    (keypoint sweep at a fixed 256 x 256 grid) on one GPU: device-resident, CUDA events, L2 flushed before every launch."""
    from cvx_proj_b200 import _runtime as rt, synth
    from cvx_proj_b200.apap import APAP, scale_anchors, weight_scale

    def timed(fn):
        ts = []
        for k in range(W + K):
            flush.add_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize()
            if k >= W:
                ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    def tensors(sc, st):
        table, tmats = st._prepare(sc.src, sc.dst)
        return table, tmats, scale_anchors(sc.vertices, weight_scale(sc.sigma))

    launches, sweep = 0, []
    for n_kp in (1000, 4000, 16000, 64000):
        sc = synth.make_scene("c5", n_kp=n_kp)
        st = APAP(sc.gamma, sc.sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y], device=device)
        table, tmats, anchors = tensors(sc, st)
        t_dev = st.kp_table_device(torch.from_numpy(table[None]).to(device))
        a_dev, m_dev = torch.from_numpy(anchors[None]).to(device), torch.from_numpy(tmats[None]).to(device)
        cells, n_pad = sc.n_cells, table.shape[0]
        ks, _, nbytes = rt.gram_plan(cells, n_pad, rt.GRAM_TCGEN05)
        partials = torch.empty(nbytes // 4, dtype=torch.float32, device=device)
        out_h = torch.empty((1, cells, 9), dtype=torch.float32, device=device)
        lib, stream = rt.load_library(), rt.stream_ptr(torch, device)
        g2 = float(np.float32(sc.gamma ** 2))
        bound = st.weight_bound_device(torch.from_numpy(np.ascontiguousarray(sc.src[None], dtype=np.float32)).to(device),
                                       None, a_dev)
        ms_gram = timed(lambda: rt.check(lib.apap_gram_partials(t_dev.data_ptr(), a_dev.data_ptr(), 1, cells, n_pad, g2,
                                                                rt.GRAM_TCGEN05, bound.data_ptr(), partials.data_ptr(),
                                                                stream)))
        ms_both = timed(lambda: st.local_homography_device(t_dev, a_dev, m_dev, 1, cells, out_h=out_h, partials=partials,
                                                           t_bound=bound))
        dump.add(f"c5_h_{n_kp}", out_h[0].reshape(sc.mesh_cells, sc.mesh_cells, 3, 3))
        launches += (W + K) * 3
        sweep.append({"n_kp": n_kp, "cells": cells, "k_splits": ks, "gram_ms": ms_gram, "k1_k2_ms": ms_both,
                      "cells_per_s": cells / (ms_both * 1e-3), "xu_frac": 2.0 * cells * n_pad / (ms_gram * 1e-3) / mufu_peak})
    pairs = 64
    scs = [synth.make_scene("c4", seed=k) for k in range(pairs)]
    st = APAP(scs[0].gamma, scs[0].sigma, [scs[0].final_w, scs[0].final_h], [scs[0].offset_x, scs[0].offset_y], device=device)
    prep = [tensors(sc, st) for sc in scs]
    rows = torch.from_numpy(np.stack([q[0] for q in prep])).to(device)
    t_dev = st.kp_table_device(rows)
    m_dev = torch.from_numpy(np.stack([q[1] for q in prep])).to(device)
    a_dev = torch.from_numpy(np.stack([q[2] for q in prep])).to(device)
    cells, n_pad = scs[0].n_cells, rows.shape[1]
    _, _, nbytes = rt.gram_plan(cells, n_pad, rt.GRAM_TCGEN05)
    partials = torch.empty(pairs * nbytes // 4, dtype=torch.float32, device=device)
    out_h = torch.empty((pairs, cells, 9), dtype=torch.float32, device=device)
    raw = np.stack([np.ascontiguousarray(sc.src, dtype=np.float32) for sc in scs])      # c4 scenes have equal match counts
    bound = st.weight_bound_device(torch.from_numpy(raw).to(device), None, a_dev)
    ms_batch = timed(lambda: st.local_homography_device(t_dev, a_dev, m_dev, pairs, cells, out_h=out_h, partials=partials,
                                                        t_bound=bound))
    dump.add("c4_h", out_h.reshape(pairs, scs[0].mesh_cells, scs[0].mesh_cells, 3, 3))
    launches += (W + K) * 2
    c4 = {"workload": _workload_desc("c4") + f", batch of {pairs} pairs in one launch", "batch_ms": ms_batch,
          "cells_per_s": pairs * cells / (ms_batch * 1e-3),
          "xu_frac": 2.0 * pairs * cells * n_pad / (ms_batch * 1e-3) / mufu_peak}
    return {"c4": c4, "c5": {"workload": "c5: 1920x1080 pair, 256x256 grid, keypoint sweep", "points": sweep}, "_launches": launches}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, help="c1..c5 (default c2)")
    ap.add_argument("--c3", default="always", choices=["multi", "always", ""],
                    help="run the c3 pass (strong-scaled over the ranks): always (default, N = 1 included), only with N>1, or never ('')")
    ap.add_argument("--no-extras", action="store_true", help="skip the c4 (batch of 64 pairs) and c5 (keypoint sweep) lines at N = 1")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--gram-engine", default="tcgen05", choices=["tcgen05", "ffma2"],
                    help="kernel of the moving-DLT contraction (default: tensor cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each timed path computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
