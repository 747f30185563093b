#!/usr/bin/env python
"""Cost of the multi-image mode (one centre against K images, run_all.sh:15,29) on the batched paths against the
per-pair loop.  One run prints:
  - the card's name, power limit and top SM clock (queries only);
  - batched RANSAC on K in {1, 4, 16, 64} c2 match sets (the 3 975 pairs of tests.test_sift._pair("c2"), each with its
    own seeded draw of uniform-noise targets at 17 % -- the exact matcher's own rate on that pair -- and at 80 %):
      one apap_ransac_homography_batch call by CUDA events, and k_ransac_sample / k_ransac_fit / k_ransac_score by
      torch.profiler (a run of its own);
      find_homography_ransac_batch host to host, and the part of it spent in the per-pair host tails (adaptive-stop
      scan, OpenCV's fit of the chosen subset, mask, refit);
      a loop of find_homography_ransac and a loop of cv.findHomography(RANSAC) on the host cores;
  - end to end on a c2-size case (centre + 4 others) and a c4-size case (centre + 16 others), the images and keypoints
    of tests/test_case.py: keypoint_pairs_batch against a loop of keypoint_pairs, and stitch_case against a loop of
    keypoint_pairs + stitch_pair, in both ransac modes, the outputs checked equal in the same run.

    python tools/case_time.py [--reps 20] [--out FILE]
"""
import argparse
import ctypes
import functools
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200 import utils  # noqa: E402
from cvx_proj_b200.driver import stitch_case, stitch_pair  # noqa: E402
from cvx_proj_b200.utils import (find_homography_ransac, find_homography_ransac_batch, keypoint_pairs,  # noqa: E402
                                 keypoint_pairs_batch)
from sift_time import c2_pair, host_ms  # noqa: E402
from tests.test_case import _scene  # noqa: E402

KERNELS = ("k_ransac_sample", "k_ransac_fit", "k_ransac_score")
MAX_ITERS = 2000
THR = 5.0
_c2_pair = functools.lru_cache(maxsize=None)(c2_pair)


def c2_sets(k, share):
    """``k`` copies of the c2 correspondences, each with its own seeded share of targets replaced by uniform noise."""
    img_c, _, raw_c, raw_o = _c2_pair()
    h, w = img_c.shape[:2]
    sets = []
    for j in range(k):
        r = np.random.default_rng(1000 + j)
        o = raw_o.copy()
        m = int(round(share * len(o)))
        bad = r.choice(len(o), m, replace=False)
        o[bad] = (r.random((m, 2)) * [w, h]).astype(np.float32)
        sets.append((raw_c, o))
    return sets


def same_fit(a, b):
    return (a[0] is None) == (b[0] is None) and np.array_equal(a[1], b[1]) and (a[0] is None or np.array_equal(a[0], b[0]))


def same_result(a, b):
    return (a.final_size == b.final_size and all(np.array_equal(getattr(a, f), getattr(b, f)) for f in
                                                  ("mesh", "vertices", "local_homography", "mat", "stitched")))


def kernel_call(lib, dev, sets):
    """A closure that runs apap_ransac_homography_batch on ``sets`` (device buffers prepared once)."""
    b = len(sets)
    ns = [len(s) for s, _ in sets]
    src = torch.from_numpy(np.concatenate([s for s, _ in sets])).to(dev)
    dst = torch.from_numpy(np.concatenate([d for _, d in sets])).to(dev)
    off = torch.from_numpy(np.cumsum([0] + ns).astype(np.int32)).to(dev)
    nb = ctypes.c_size_t()
    rt.check(lib.apap_ransac_batch_workspace_bytes(b, MAX_ITERS, ctypes.byref(nb)), "apap_ransac_batch_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    sub = torch.empty((b, MAX_ITERS, 4), dtype=torch.int32, device=dev)
    hyps = torch.empty((b, MAX_ITERS, 9), dtype=torch.float64, device=dev)
    cnt = torch.empty((b, MAX_ITERS), dtype=torch.int32, device=dev)
    n_s = torch.empty(b, dtype=torch.int32, device=dev)
    st = rt.stream_ptr(torch, dev)

    def call():
        rt.check(lib.apap_ransac_homography_batch(src.data_ptr(), dst.data_ptr(), off.data_ptr(), b, max(ns), THR,
                                                  MAX_ITERS, ws.data_ptr(), nb.value, sub.data_ptr(), hyps.data_ptr(),
                                                  cnt.data_ptr(), n_s.data_ptr(), st), "apap_ransac_homography_batch")
    return call


def event_us(call, reps):
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def profiled_us(call, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        for name in KERNELS:
            if name in e.key:
                kern[name] = (getattr(e, "device_time_total", None) or e.cuda_time_total) / max(e.count, 1)
    return kern


def batch_with_tails(sets, reps):
    """find_homography_ransac_batch host to host, and the summed time of its per-pair host tails, per call."""
    tails, orig = [], utils._ransac_tail

    def timed(*a, **k):
        t0 = time.perf_counter()
        out = orig(*a, **k)
        tails.append(time.perf_counter() - t0)
        return out
    srcs, dsts = [s for s, _ in sets], [d for _, d in sets]
    utils._ransac_tail = timed
    try:
        find_homography_ransac_batch(srcs, dsts, THR)
        tails.clear()
        t = host_ms(lambda: find_homography_ransac_batch(srcs, dsts, THR), reps)
    finally:
        utils._ransac_tail = orig
    per_call = np.array(tails).reshape(reps, len(sets)).sum(axis=1) * 1e3
    return t, float(np.median(per_call))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    _, dev = rt.torch_cuda()
    lib = rt.load_library()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"card: {torch.cuda.get_device_name(dev)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    say(f"host cores: {os.cpu_count()}, cv.getNumThreads() = {cv.getNumThreads()}, OpenCV {cv.__version__}")
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "ransac": [], "e2e": []}
    say(f"== batched RANSAC: c2 match sets, max_iters {MAX_ITERS}, threshold {THR}")
    for share in (0.17, 0.8):
        for k in (1, 4, 16, 64):
            sets = c2_sets(k, share)
            reps = max(3, args.reps // k)
            call = kernel_call(lib, dev, sets)
            call_us = event_us(call, args.reps)
            kern = profiled_us(call, args.reps)
            (batch_ms, batch_min), tails_ms = batch_with_tails(sets, reps)
            loop_ms = host_ms(lambda: [find_homography_ransac(s, d, THR) for s, d in sets], reps)
            cv_ms = host_ms(lambda: [cv.findHomography(s, d, cv.RANSAC, THR) for s, d in sets], reps)
            got = find_homography_ransac_batch([s for s, _ in sets], [d for _, d in sets], THR)
            loop = [find_homography_ransac(s, d, THR) for s, d in sets]
            ocv = [cv.findHomography(s, d, cv.RANSAC, THR) for s, d in sets]
            eq_loop = all(same_fit(a, b) for a, b in zip(got, loop))
            eq_cv = all(same_fit(a, b) for a, b in zip(got, ocv))
            say(f"{100 * share:.0f} % outliers, K = {k}: apap_ransac_homography_batch (CUDA events, {args.reps} calls) "
                f"median {call_us[0]:.1f} us, min {call_us[1]:.1f} us; " +
                ", ".join(f"{n} {kern.get(n, float('nan')):.1f} us" for n in KERNELS) + " (profiler)")
            say(f"  find_homography_ransac_batch {batch_ms:.2f} ms (min {batch_min:.2f}), of which host tails "
                f"{tails_ms:.2f} ms; loop of find_homography_ransac {loop_ms[0]:.2f} ms; loop of cv.findHomography "
                f"{cv_ms[0]:.2f} ms ({reps} reps, medians); batch == loop: {eq_loop}, == OpenCV: {eq_cv}")
            res["ransac"].append({"outliers": share, "k": k, "call_us": call_us[0],
                                  **{n + "_us": v for n, v in kern.items()}, "batch_ms": batch_ms,
                                  "tails_ms": tails_ms, "loop_ms": loop_ms[0], "cv_loop_ms": cv_ms[0],
                                  "equal_loop": eq_loop, "equal_cv": eq_cv})
    for name, k in (("c2", 4), ("c4", 16)):
        centre, others, raw_c, raw_os = _scene(name, k)
        say(f"== end to end: {name} ({centre.shape[1]} x {centre.shape[0]}), centre + {k} others, {len(raw_c)} "
            f"keypoints, mesh 100")
        for mode in ("opencv", "gpu"):
            kp_b = keypoint_pairs_batch(centre, others, raw_c, raw_os, ransac=mode)
            kp_l = [keypoint_pairs(centre, o, raw_c, ko, ransac=mode) for o, ko in zip(others, raw_os)]
            eq_kp = all(all(np.array_equal(a, b) for a, b in zip(x, y)) for x, y in zip(kp_b, kp_l))
            got = stitch_case(centre, others, raw_c, raw_os, ransac=mode)
            want = [stitch_pair(centre, o, *p) for o, p in zip(others, kp_l)]
            eq = all(same_result(a, b) for a, b in zip(got, want))
            reps = 3
            t_kb = host_ms(lambda: keypoint_pairs_batch(centre, others, raw_c, raw_os, ransac=mode), reps)
            t_kl = host_ms(lambda: [keypoint_pairs(centre, o, raw_c, ko, ransac=mode) for o, ko in zip(others, raw_os)],
                           reps)
            t_sc = host_ms(lambda: stitch_case(centre, others, raw_c, raw_os, ransac=mode), reps)
            t_sl = host_ms(lambda: [stitch_pair(centre, o, *keypoint_pairs(centre, o, raw_c, ko, ransac=mode))
                                    for o, ko in zip(others, raw_os)], reps)
            say(f"  ransac={mode!r}: keypoint_pairs_batch {t_kb[0]:.1f} ms vs loop of keypoint_pairs {t_kl[0]:.1f} ms "
                f"(equal: {eq_kp}); stitch_case {t_sc[0]:.1f} ms vs loop of keypoint_pairs + stitch_pair "
                f"{t_sl[0]:.1f} ms (equal: {eq}) ({reps} reps, medians)")
            res["e2e"].append({"case": name, "k": k, "ransac": mode, "kp_batch_ms": t_kb[0], "kp_loop_ms": t_kl[0],
                               "stitch_case_ms": t_sc[0], "stitch_loop_ms": t_sl[0], "equal_kp": eq_kp, "equal": eq})
    say(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
