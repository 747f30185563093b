#!/usr/bin/env python
"""Cost of the histogram equalisation (csrc/equalize.cu) and of the array-level keypoint-pair producer
(utils.keypoint_pairs) at the bench shape c2 (3840 x 2160, the tools/sift_time.py pair).  One run prints:
  - the card's name and power limit (queries only);
  - k_eq_hist, k_eq_lut and k_eq_apply from torch.profiler, the L2 flushed by a 256 MiB write before every launch, with
    bytes over time against the data-sheet HBM bandwidth; k_eq_hist again on a flat image (every byte of a channel in
    one bin: the contention worst case);
  - k_sift_base through the LUT against the plain instance, alternating in the same profiled run;
  - device time of one apap_equalize_hist call (CUDA events), with and without the equalised image written;
  - host to host: equalize_hist vs OpenCV's per-channel cv.equalizeHist on the host cores, sift_describe(equalize=True),
    keypoint_pairs vs (host equalisation + coarse_matching(describe="gpu") + findHomography) vs the all-OpenCV chain
    with FLANN (the reference's).

    python tools/producer_time.py [--iters 200]
"""
import argparse
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
from cvx_proj_b200.utils import (coarse_matching, equalize_hist, keypoint_pairs, sift_describe,  # noqa: E402
                                 sift_sample_table)
from sift_time import HBM_TBPS, c2_pair, host_ms  # noqa: E402


def cv_equalize(img):
    return cv.merge([cv.equalizeHist(c) for c in cv.split(img)])


def kernel_name(key):
    for n in ("k_eq_hist", "k_eq_lut", "k_eq_apply"):
        if n in key:
            return n
    if "k_sift_base" in key:
        return "k_sift_base_lut" if ("<true>" in key or "ILb1E" in key) else "k_sift_base"
    return None


def profiled(fn, flush, reps=50):
    """{kernel: mean device us} of ``reps`` launches of ``fn``, each after an L2 flush."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            flush.fill_(1)
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        n = kernel_name(e.key)
        if n:
            out[n] = (getattr(e, "device_time_total", None) or e.cuda_time_total) / max(e.count, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    torch_, dev = rt.torch_cuda()
    lib = rt.load_library()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(f"card: {torch.cuda.get_device_name(dev)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    img_c, img_o, raw_c, raw_o = c2_pair()
    h, w = img_c.shape[:2]
    px = h * w
    k = len(raw_c)
    print(f"c2: {w}x{h} ({3 * px / 1e6:.1f} MB per image), {k} keypoints")
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "w": w, "h": h, "keypoints": k}

    st = rt.stream_ptr(torch_, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    d_img = torch.from_numpy(img_c).to(dev)
    d_flat = torch.full_like(d_img, 128)
    hist = torch.empty(768, dtype=torch.int32, device=dev)
    lut = torch.empty(768, dtype=torch.uint8, device=dev)
    out = torch.empty_like(d_img)

    def eq(img, dst):
        rt.check(lib.apap_equalize_hist(img.data_ptr(), h, w, hist.data_ptr(), lut.data_ptr(), dst, st), "apap_equalize_hist")

    for _ in range(5):
        eq(d_img, out.data_ptr())
        eq(d_flat, None)
    torch.cuda.synchronize()
    for label, fn in (("apap_equalize_hist (hist + LUT)", lambda: eq(d_img, None)),
                      ("apap_equalize_hist (hist + LUT + apply)", lambda: eq(d_img, out.data_ptr()))):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.iters)]
        for e0, e1 in evs:
            flush.fill_(1)
            e0.record()
            fn()
            e1.record()
        torch.cuda.synchronize()
        us = np.array([e0.elapsed_time(e1) * 1e3 for e0, e1 in evs])
        print(f"{label} device time (L2 flushed, {args.iters} launches): median {np.median(us):.1f} us, min {us.min():.1f} us")
        res["eq_call_us" if "apply" not in label else "eq_call_apply_us"] = float(np.median(us))

    floor = lambda b: b / (HBM_TBPS * 1e12) * 1e6  # noqa: E731
    kern = profiled(lambda: eq(d_img, out.data_ptr()), flush)
    for name, nbytes, what in (("k_eq_hist", 3 * px, "3 px read"), ("k_eq_lut", 768 * 4 + 768, "hist read + LUT written"),
                               ("k_eq_apply", 6 * px, "3 px read + 3 px written")):
        if name in kern:
            t = kern[name]
            gbs = nbytes / (t * 1e-6) / 1e9
            print(f"{name} (profiler, 50 launches): {t:.2f} us; {nbytes / 1e6:.3g} MB ({what}) -> {gbs:.0f} GB/s = "
                  f"{gbs / (HBM_TBPS * 1e3) * 100:.1f} % of {HBM_TBPS} TB/s (floor {floor(nbytes):.2f} us)")
            res[f"{name}_us"] = t
    kflat = profiled(lambda: eq(d_flat, None), flush)
    if "k_eq_hist" in kflat:
        t = kflat["k_eq_hist"]
        print(f"k_eq_hist on a flat image (every byte of a channel in one bin): {t:.2f} us = "
              f"{3 * px / (t * 1e-6) / 1e9:.0f} GB/s")
        res["k_eq_hist_flat_us"] = t

    table, ori = sift_sample_table(1.0, -1.0, h, w)
    d_pts = torch.from_numpy(raw_c).to(dev)
    d_tab = torch.from_numpy(table).to(dev)
    base = torch.empty((h, w), dtype=torch.float32, device=dev)
    desc = torch.empty((k, 128), dtype=torch.float32, device=dev)
    eq(d_img, None)

    def both():
        rt.check(lib.apap_sift_describe(d_img.data_ptr(), h, w, d_pts.data_ptr(), k, d_tab.data_ptr(), table.shape[0],
                                        float(ori), base.data_ptr(), desc.data_ptr(), st), "apap_sift_describe")
        flush.fill_(1)
        rt.check(lib.apap_sift_describe_lut(d_img.data_ptr(), h, w, lut.data_ptr(), d_pts.data_ptr(), k, d_tab.data_ptr(),
                                            table.shape[0], float(ori), base.data_ptr(), desc.data_ptr(), st),
                 "apap_sift_describe_lut")
    both()
    kb = profiled(both, flush)
    if "k_sift_base" in kb and "k_sift_base_lut" in kb:
        print(f"k_sift_base (profiler, 50 launches each, alternating): plain {kb['k_sift_base']:.1f} us, through the LUT "
              f"{kb['k_sift_base_lut']:.1f} us")
        res.update(base_plain_us=kb["k_sift_base"], base_lut_us=kb["k_sift_base_lut"])

    equalize_hist(img_c)
    m_gpu, _ = host_ms(lambda: equalize_hist(img_c), 20)
    m_cv, _ = host_ms(lambda: cv_equalize(img_c), 20)
    print(f"equalize_hist host to host (numpy in, numpy out): median {m_gpu:.2f} ms; cv.equalizeHist per channel on the "
          f"host ({os.cpu_count()} cores, cv.getNumThreads() = {cv.getNumThreads()}): median {m_cv:.2f} ms")
    res.update(equalize_h2h_ms=m_gpu, equalize_cv_ms=m_cv, host_cores=os.cpu_count())
    sift_describe(img_c, raw_c, equalize=True)
    m, _ = host_ms(lambda: sift_describe(img_c, raw_c, equalize=True), 20)
    print(f"sift_describe(equalize=True) host to host: median {m:.2f} ms")
    res.update(sift_describe_eq_h2h_ms=m)

    def old_chain():
        kc, _, ko, _, matches = coarse_matching(cv_equalize(img_c), cv_equalize(img_o), raw_c, raw_o, describe="gpu")
        src = np.float32([kc[mm.queryIdx].pt for mm in matches])
        dst = np.float32([ko[mm.trainIdx].pt for mm in matches])
        hh, mask = cv.findHomography(src, dst, cv.RANSAC, 5.0)
        return np.linalg.inv(hh)

    def opencv_chain():
        ext = cv.SIFT.create(nfeatures=128)
        kc, fc = ext.compute(cv_equalize(img_c), [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_c])
        ko, fo = ext.compute(cv_equalize(img_o), [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_o])
        matches = cv.FlannBasedMatcher().match(fc, fo)
        src = np.float32([kc[mm.queryIdx].pt for mm in matches])
        dst = np.float32([ko[mm.trainIdx].pt for mm in matches])
        hh, mask = cv.findHomography(src, dst, cv.RANSAC, 5.0)
        return np.linalg.inv(hh)

    keypoint_pairs(img_c, img_o, raw_c, raw_o)
    old_chain()
    m_kp, mn_kp = host_ms(lambda: keypoint_pairs(img_c, img_o, raw_c, raw_o), 20)
    m_old, _ = host_ms(old_chain, 10)
    m_cvc, _ = host_ms(opencv_chain, 3)
    print(f"keypoint_pairs host to host (two numpy images in, (final_src, final_dst, H) out): median {m_kp:.2f} ms, "
          f"min {mn_kp:.2f} ms")
    print(f"host equalisation + coarse_matching(describe='gpu') + findHomography: median {m_old:.2f} ms")
    print(f"all-OpenCV chain (equalizeHist, SIFT.compute, FLANN, findHomography): median {m_cvc:.1f} ms")
    res.update(keypoint_pairs_ms=m_kp, coarse_gpu_chain_ms=m_old, opencv_flann_chain_ms=m_cvc)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
