#!/usr/bin/env python
"""Cost of the GPU RANSAC (csrc/ransac.cu, utils.find_homography_ransac) at the bench shape c2 (3840 x 2160, the
tools/sift_time.py pair).  The match set is the exact matcher's on that pair (what keypoint_pairs hands to RANSAC);
for the higher outlier shares a seeded part of its targets is replaced by uniform noise over the image.  One run
prints:
  - the card's name, power limit and top SM clock (queries only);
  - per outlier share: the iterations OpenCV's loop runs, the device time of one apap_ransac_homography call (CUDA
    events) and of k_ransac_sample / k_ransac_fit / k_ransac_score (torch.profiler, a run of its own);
  - host to host: find_homography_ransac against cv.findHomography(RANSAC) on the host cores, the result checked
    equal; keypoint_pairs with ransac="opencv" and ransac="gpu".

    python tools/ransac_time.py [--reps 50] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200.utils import (find_homography_ransac, keypoint_pairs, match_descriptors,  # noqa: E402
                                 sift_describe)
from sift_time import c2_pair, host_ms  # noqa: E402

KERNELS = ("k_ransac_sample", "k_ransac_fit", "k_ransac_score")
MAX_ITERS = 2000


def iterations_run(counts, n_sampled, n, confidence=0.995, max_iters=MAX_ITERS):
    from cvx_proj_b200.utils import _ransac_update_num_iters
    niters, best, it = max_iters, 0, 0
    while it < niters and it < n_sampled:
        if counts[it] > max(best, 3):
            best = int(counts[it])
            niters = _ransac_update_num_iters(confidence, (n - best) / n, 4, niters)
        it += 1
    return it


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    torch_, dev = rt.torch_cuda()
    lib = rt.load_library()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"card: {torch.cuda.get_device_name(dev)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    say(f"host cores: {os.cpu_count()}, cv.getNumThreads() = {cv.getNumThreads()}, OpenCV {cv.__version__}")
    img_c, img_o, raw_c, raw_o = c2_pair()
    idx, _ = match_descriptors(sift_describe(img_c, raw_c, equalize=True), sift_describe(img_o, raw_o, equalize=True))
    qi = np.flatnonzero(idx >= 0)
    centre, other0 = raw_c[qi], raw_o[idx[qi]]
    n = len(centre)
    wrong = int(np.sum(idx[qi] != qi))
    say(f"c2: {n} matches, {wrong} ({100 * wrong / n:.0f} %) not the generating pair")
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "matches": n, "cases": []}
    st = rt.stream_ptr(torch_, dev)
    nb = ctypes.c_size_t()
    rt.check(lib.apap_ransac_workspace_bytes(MAX_ITERS, ctypes.byref(nb)), "apap_ransac_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    sub = torch.empty((MAX_ITERS, 4), dtype=torch.int32, device=dev)
    hyps = torch.empty((MAX_ITERS, 9), dtype=torch.float64, device=dev)
    cnt = torch.empty(MAX_ITERS, dtype=torch.int32, device=dev)
    ns = torch.empty(1, dtype=torch.int32, device=dev)
    r = np.random.default_rng(5)
    for share in (None, 0.5, 0.7, 0.8, 0.9):
        other = other0.copy()
        label = f"as matched ({100 * wrong / n:.0f} %)"
        if share is not None:
            k = int(share * n)
            bad = r.choice(n, k, replace=False)
            other[bad] = (r.random((k, 2)) * [img_o.shape[1], img_o.shape[0]]).astype(np.float32)
            label = f"{100 * share:.0f} % replaced"
        s_dev, d_dev = torch.from_numpy(centre).to(dev), torch.from_numpy(other).to(dev)

        def call():
            rt.check(lib.apap_ransac_homography(s_dev.data_ptr(), d_dev.data_ptr(), n, 5.0, MAX_ITERS, ws.data_ptr(),
                                                nb.value, sub.data_ptr(), hyps.data_ptr(), cnt.data_ptr(),
                                                ns.data_ptr(), st), "apap_ransac_homography")
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        n_s = int(ns.item())
        its = iterations_run(cnt.cpu().numpy(), n_s, n)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                call()
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            for name in KERNELS:
                if name in e.key:
                    kern[name] = (getattr(e, "device_time_total", None) or e.cuda_time_total) / max(e.count, 1)
        want = cv.findHomography(centre, other, cv.RANSAC, 5.0)
        got = find_homography_ransac(centre, other, 5.0)
        same = np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        gpu_ms = host_ms(lambda: find_homography_ransac(centre, other, 5.0), args.reps)
        cv_ms = host_ms(lambda: cv.findHomography(centre, other, cv.RANSAC, 5.0), args.reps)
        refit_ms = host_ms(lambda: cv.findHomography(centre[got[1].ravel() > 0], other[got[1].ravel() > 0], 0),
                           args.reps)
        inl = int(got[1].sum())
        say(f"{label}: {inl} inliers, OpenCV's loop runs {its} of {n_s} sampled hypotheses")
        say(f"  apap_ransac_homography device time (CUDA events, {args.reps} calls): median {np.median(ts):.1f} us, "
            f"min {np.min(ts):.1f} us")
        say("  " + ", ".join(f"{k} {kern.get(k, float('nan')):.1f} us" for k in KERNELS) +
            f" (profiler, {args.reps} calls)")
        say(f"  find_homography_ransac host to host: median {gpu_ms[0]:.3f} ms (min {gpu_ms[1]:.3f}); "
            f"cv.findHomography(RANSAC): median {cv_ms[0]:.3f} ms (min {cv_ms[1]:.3f}); "
            f"of which the refit cv.findHomography(inliers, 0): {refit_ms[0]:.3f} ms; equal: {same}")
        res["cases"].append({"case": label, "inliers": inl, "iterations": its, "sampled": n_s,
                             "call_us": float(np.median(ts)), **{k + "_us": v for k, v in kern.items()},
                             "gpu_h2h_ms": gpu_ms[0], "cv_ms": cv_ms[0], "refit_ms": refit_ms[0], "equal": bool(same)})
    for mode in ("opencv", "gpu"):
        keypoint_pairs(img_c, img_o, raw_c, raw_o, ransac=mode)
        t = host_ms(lambda: keypoint_pairs(img_c, img_o, raw_c, raw_o, ransac=mode), args.reps)
        say(f"keypoint_pairs(ransac={mode!r}) host to host: median {t[0]:.2f} ms, min {t[1]:.2f} ms")
        res[f"keypoint_pairs_{mode}_ms"] = t[0]
    say(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
