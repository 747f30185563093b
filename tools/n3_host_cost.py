#!/usr/bin/env python
"""Row N3 of SURVEY 8f (the keypoint-pair producer: pyviz/utils.py:142-151 coarse_matching + pyviz/baseline_stitch_test.py:40
cv.findHomography): what it costs on the host, and how far its outputs are defined at bit level -- the measurements
behind DESIGN section 7.  CPU only (OpenCV); synthetic pairs of the bench shapes (cvx_proj_b200.synth).

    python tools/n3_host_cost.py [c1 c2 ...]
"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402

from cvx_proj_b200 import synth  # noqa: E402


def timed(fn, reps=3):
    best, out = float("inf"), None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3, out


for name in (sys.argv[1:] or ["c1", "c2"]):
    # the other view = the centre image warped by the scene's ground-truth homography (so descriptors do match)
    img_c, img_o, raw_c, raw_o = synth.make_pair(name)
    kc = [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_c]
    ko = [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_o]
    ext = cv.SIFT.create(nfeatures=128)
    t_desc, (kc2, fc) = timed(lambda: ext.compute(img_c, kc))
    _, (ko2, fo) = timed(lambda: ext.compute(img_o, ko))
    t_flann, m_flann = timed(lambda: cv.FlannBasedMatcher().match(fc, fo))
    t_bf, m_bf = timed(lambda: cv.BFMatcher(cv.NORM_L2).match(fc, fo))
    same = sum(a.trainIdx == b.trainIdx for a, b in zip(m_flann, m_bf))
    runs = [tuple(m.trainIdx for m in cv.FlannBasedMatcher().match(fc, fo)) for _ in range(3)]
    stable = sum(len(set(col)) == 1 for col in zip(*runs))
    src = np.float32([kc2[m.queryIdx].pt for m in m_flann])
    dst = np.float32([ko2[m.trainIdx].pt for m in m_flann])
    t_ransac, (h, mask) = timed(lambda: cv.findHomography(src, dst, cv.RANSAC, 5.0), reps=5)
    print(f"{name}: {img_c.shape[1]}x{img_c.shape[0]}, {len(kc)} keypoints given (size 1, as the reference builds them)")
    print(f"  SIFT.compute at the given keypoints     {t_desc:9.1f} ms per image (Gaussian pyramid of the whole image + 128-d descriptors)")
    print(f"  FlannBasedMatcher().match (reference)   {t_flann:9.1f} ms   {len(m_flann)} matches")
    print(f"  BFMatcher(NORM_L2).match  (exact 1-NN)  {t_bf:9.1f} ms   FLANN agrees with the exact neighbour on {same} of {len(m_bf)} "
          f"({100.0 * same / max(len(m_bf), 1):.1f} %), {stable} of {len(m_bf)} identical over 3 FLANN runs")
    print(f"  cv.findHomography(RANSAC, 5.0)          {t_ransac:9.2f} ms   inliers {int(mask.sum())} of {len(src)}")
