#!/usr/bin/env python
"""Cost of the SIFT descriptors at given keypoints (utils.sift_describe, csrc/sift.cu) at the bench shape c2
(3840 x 2160, synth.make_pair("c2")), against cv.SIFT.compute on the host cores.  One run prints:
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
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200 import synth  # noqa: E402
from cvx_proj_b200.utils import coarse_matching, sift_describe, sift_sample_table  # noqa: E402
from timing import HBM_TBS, card, host_ms, kernel_times, l2_flush, name_in  # noqa: E402

KERNELS = ("k_sift_base", "k_sift_desc")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    torch_, dev = rt.torch_cuda()
    lib = rt.load_library()
    res = card(dev)
    img_c, img_o, raw_c, raw_o = synth.make_pair("c2")
    h, w = img_c.shape[:2]
    k = len(raw_c)
    print(f"c2: {w}x{h}, {k} keypoints (size 1, angle -1, as the reference builds them)")

    table, ori = sift_sample_table(1.0, -1.0, h, w)
    d_img = torch.from_numpy(img_c).to(dev)
    d_pts = torch.from_numpy(raw_c).to(dev)
    d_tab = torch.from_numpy(table).to(dev)
    base = torch.empty((h, w), dtype=torch.float32, device=dev)
    desc = torch.empty((k, 128), dtype=torch.float32, device=dev)
    flush = l2_flush(dev)
    st = rt.stream_ptr(torch_, dev)

    def launch():
        rt.check(lib.apap_sift_describe(d_img.data_ptr(), h, w, d_pts.data_ptr(), k, d_tab.data_ptr(), table.shape[0],
                                        float(ori), base.data_ptr(), desc.data_ptr(), st), "apap_sift_describe")

    for _ in range(10):
        flush.fill_(1)
        launch()
    torch.cuda.synchronize()
    # All launches are queued and their events read after one synchronise.  With a synchronise after every call, as
    # timing.event_us does, the median stays but the min rises by about 0.6 us and the max by about 34 us (host delays
    # between the flush and the launch; measured on a B200 at 1000 W).
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

    kern = {n: float(np.mean(v)) for n, v in kernel_times([launch], name_in(KERNELS), 50, flush).items()}
    px = h * w
    base_bytes = 3 * px + 4 * px
    res.update(w=w, h=h, keypoints=k, describe_device_us_median=float(np.median(dev_us)),
               describe_device_us_min=float(dev_us.min()))
    if "k_sift_base" in kern:
        t = kern["k_sift_base"]
        gbs = base_bytes / (t * 1e-6) / 1e9
        print(f"k_sift_base (profiler, 50 launches): {t:.1f} us; {base_bytes / 1e6:.1f} MB (3 px read + 4 px written) -> "
              f"{gbs:.0f} GB/s = {gbs / (HBM_TBS * 1e3) * 100:.0f} % of {HBM_TBS} TB/s (floor {base_bytes / (HBM_TBS * 1e12) * 1e6:.1f} us)")
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
