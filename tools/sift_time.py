#!/usr/bin/env python
"""Cost of the SIFT descriptors at given keypoints (utils.sift_describe, csrc/sift.cu) at the bench shape c2
(3840 x 2160, the tools/n3_host_cost.py pair), against cv.SIFT.compute on the host cores.  One run prints:
  - the card's name and power limit (queries only);
  - device time of one apap_sift_describe call (both kernels), the L2 flushed by a 256 MiB write before every launch;
  - k_sift_base and k_sift_desc split out by a separate torch.profiler run (same flushed launches);
  - sift_describe host to host (numpy image and points in, numpy descriptors out);
  - coarse_matching(describe="gpu") vs describe="opencv" host to host (both images, matcher, DMatch list);
  - cv.SIFT.compute per image on the host.

    python tools/sift_time.py [--iters 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200 import synth  # noqa: E402
from cvx_proj_b200.utils import coarse_matching, sift_describe, sift_sample_table  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU


def c2_pair():
    sc = synth.make_scene("c2")
    rng = np.random.default_rng(1)
    img_c = synth.make_image(sc.width, sc.height, seed=2)
    hinv = np.linalg.inv(sc.h_gt)
    img_o = cv.warpPerspective(img_c, hinv, (sc.width, sc.height))
    raw_c = sc.dst.astype(np.float32)
    raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
    keep = np.all((raw_o > 8) & (raw_o < [sc.width - 8, sc.height - 8]) & (raw_c > 8) & (raw_c < [sc.width - 8, sc.height - 8]),
                  axis=1)
    raw_c, raw_o = raw_c[keep], raw_o[keep]
    return img_c, img_o, raw_c, raw_o + rng.normal(0, 0.3, raw_o.shape).astype(np.float32)


def host_ms(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


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
    k = len(raw_c)
    print(f"c2: {w}x{h}, {k} keypoints (size 1, angle -1, as the reference builds them)")

    table, ori = sift_sample_table(1.0, -1.0, h, w)
    d_img = torch.from_numpy(img_c).to(dev)
    d_pts = torch.from_numpy(raw_c).to(dev)
    d_tab = torch.from_numpy(table).to(dev)
    base = torch.empty((h, w), dtype=torch.float32, device=dev)
    desc = torch.empty((k, 128), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = rt.stream_ptr(torch_, dev)

    def launch():
        rt.check(lib.apap_sift_describe(d_img.data_ptr(), h, w, d_pts.data_ptr(), k, d_tab.data_ptr(), table.shape[0],
                                        float(ori), base.data_ptr(), desc.data_ptr(), st), "apap_sift_describe")

    for _ in range(10):
        flush.fill_(1)
        launch()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.iters)]
    for e0, e1 in evs:
        flush.fill_(1)
        e0.record()
        launch()
        e1.record()
    torch.cuda.synchronize()
    dev_us = np.array([e0.elapsed_time(e1) * 1e3 for e0, e1 in evs])
    print(f"apap_sift_describe device time (L2 flushed, {args.iters} launches): median {np.median(dev_us):.1f} us, "
          f"min {dev_us.min():.1f} us, max {dev_us.max():.1f} us")

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            flush.fill_(1)
            launch()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if e.key.startswith(("_ZN4apap11k_sift", "apap::k_sift")) or "k_sift_" in e.key:
            name = "k_sift_base" if "k_sift_base" in e.key else "k_sift_desc"
            kern[name] = (getattr(e, "device_time_total", None) or e.cuda_time_total) / max(e.count, 1)
    px = h * w
    base_bytes = 3 * px + 4 * px
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "w": w, "h": h, "keypoints": k,
           "describe_device_us_median": float(np.median(dev_us)), "describe_device_us_min": float(dev_us.min())}
    if "k_sift_base" in kern:
        t = kern["k_sift_base"]
        gbs = base_bytes / (t * 1e-6) / 1e9
        print(f"k_sift_base (profiler, 50 launches): {t:.1f} us; {base_bytes / 1e6:.1f} MB (3 px read + 4 px written) -> "
              f"{gbs:.0f} GB/s = {gbs / (HBM_TBPS * 1e3) * 100:.0f} % of {HBM_TBPS} TB/s (floor {base_bytes / (HBM_TBPS * 1e12) * 1e6:.1f} us)")
        res.update(base_us=t, base_gbs=gbs)
    if "k_sift_desc" in kern:
        t = kern["k_sift_desc"]
        print(f"k_sift_desc (profiler, 50 launches): {t:.1f} us = {k / (t * 1e-6) / 1e6:.1f} M keypoints/s")
        res.update(desc_us=t, desc_mkps=k / (t * 1e-6) / 1e6)

    sift_describe(img_c, raw_c)
    m, mn = host_ms(lambda: sift_describe(img_c, raw_c), 20)
    print(f"sift_describe host to host (numpy {img_c.nbytes / 1e6:.1f} MB image in, numpy out): median {m:.2f} ms, min {mn:.2f} ms")
    res.update(sift_describe_h2h_ms=m)

    coarse_matching(img_c, img_o, raw_c, raw_o, describe="gpu")
    m_gpu, _ = host_ms(lambda: coarse_matching(img_c, img_o, raw_c, raw_o, describe="gpu"), 10)
    m_cv, _ = host_ms(lambda: coarse_matching(img_c, img_o, raw_c, raw_o, describe="opencv"), 3)
    print(f"coarse_matching host to host: describe='gpu' {m_gpu:.2f} ms, describe='opencv' {m_cv:.1f} ms "
          f"({m_cv / m_gpu:.0f}x)")
    res.update(coarse_gpu_ms=m_gpu, coarse_opencv_ms=m_cv)

    kps = [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_c]
    ext = cv.SIFT.create(nfeatures=128)
    m, mn = host_ms(lambda: ext.compute(img_c, kps), 3)
    print(f"cv.SIFT.compute on the host ({os.cpu_count()} cores, cv.getNumThreads() = {cv.getNumThreads()}): "
          f"median {m:.1f} ms, min {mn:.1f} ms per image")
    res.update(cv_compute_ms=m, host_cores=os.cpu_count())
    print(json.dumps(res))


if __name__ == "__main__":
    main()
