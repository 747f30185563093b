"""RANSAC homography (cvx_proj_b200.utils.find_homography_ransac, csrc/ransac.cu, keypoint_pairs(ransac="gpu")): the
restatement of OpenCV's loop (oracle/ransac_oracle.py) against the live cv.findHomography on the CPU, the kernels
against its per-hypothesis record and the host wrapper against OpenCV on the GPU.

Everything is bit-equal to OpenCV except H when the best hypothesis has exactly 4 inliers: OpenCV then refits and
LM-refines those 4 points, which is not restated, and H is held to 1e-9 relative (the mask stays exact)."""
import functools

import cv2 as cv
import numpy as np
import pytest

from oracle import ransac_oracle as ro
from tests import test_sift as ts

H_TRUE = np.array([[1.02, 0.03, 12.0], [-0.02, 0.98, -7.0], [1e-5, -2e-5, 1.0]])


def _case(n, outliers, sigma, seed, scale=1000.0):
    """``n`` correspondences under H_TRUE with Gaussian noise ``sigma`` px; a share ``outliers`` of the targets
    replaced by uniform noise over the ``scale`` square."""
    r = np.random.default_rng(seed)
    src = (r.random((n, 2)) * scale).astype(np.float32)
    p = np.c_[src, np.ones(n)] @ H_TRUE.T
    dst = (p[:, :2] / p[:, 2:] + r.normal(0, sigma, (n, 2))).astype(np.float32)
    k = int(round(outliers * n))
    bad = r.choice(n, k, replace=False)
    dst[bad] = (r.random((k, 2)) * scale).astype(np.float32)
    return src, dst


@functools.lru_cache(maxsize=None)
def _c2_pairs(outliers=0.0):
    """The c2 keypoint pairs (3 975 centre / other points of tests.test_sift's pair) with a share of the targets
    replaced by uniform noise over the image."""
    _, img_o, raw_c, raw_o = ts._pair("c2")
    raw_o = raw_o.copy()
    r = np.random.default_rng(80)
    k = int(round(outliers * len(raw_o)))
    bad = r.choice(len(raw_o), k, replace=False)
    raw_o[bad] = (r.random((k, 2)) * [img_o.shape[1], img_o.shape[0]]).astype(np.float32)
    return raw_c, raw_o


def _grid():
    """A seeded draw from N x outliers x sigma x maxIters x confidence x threshold, each value of every axis used."""
    ns = [4, 5, 6, 8, 20, 100, 1000]
    outl = [0, 0.2, 0.5, 0.7, 0.8, 0.9]
    sig = [0.3, 2, 4]
    iters = [1, 2, 50, 2000]
    conf = [0.9, 0.995, 0.999]
    thr = [1, 3, 5]
    r = np.random.default_rng(2024)
    cases = []
    for i in range(48):
        n = ns[i % len(ns)]
        o = outl[i % len(outl)]
        cases.append((n, o, sig[r.integers(3)], iters[i % 4], conf[r.integers(3)], thr[r.integers(3)], i))
    return cases


GRID = _grid()
C2 = [(0.0, 2000, 0.995, 5), (0.17, 2000, 0.995, 5), (0.5, 2000, 0.995, 5), (0.8, 2000, 0.995, 5),
      (0.9, 50, 0.999, 3), (0.7, 2, 0.9, 1)]


def _near_collinear(k):
    """Random near-collinear sets: 12..40 points within 3e-5..3e-4 px of a line over a 100 px span, mapped by an
    affine map (seed k).  Subsets of such points pass checkSubset's FLT_EPSILON bound while LtL has an almost
    two-dimensional null space."""
    r = np.random.default_rng(1000 + k)
    n = int(r.integers(12, 41))
    t = r.random(n) * 100.0
    p = (np.c_[t, 0.7 * t + 5] + r.normal(0, r.uniform(3e-5, 3e-4), (n, 2))).astype(np.float32)
    return p, (p * 1.3 + 2).astype(np.float32)


def _edge(name):
    """``(src, dst)`` of the named edge case."""
    if name == "near-collinear":                                 # a line plus 1e-4 px noise, dst = 1.5 src
        t = np.linspace(0, 100, 30, dtype=np.float32)
        line = np.c_[t, 2 * t].astype(np.float32)
        near = line + np.random.default_rng(3).normal(0, 1e-4, line.shape).astype(np.float32)
        return near, near * 1.5
    if name.startswith("near-collinear-"):
        return _near_collinear(int(name.rsplit("-", 1)[1]))
    if name == "duplicates":
        src, dst = _case(40, 0.3, 0.3, 5)
        src[10:20], dst[10:20] = src[0], dst[0]
        return src, dst
    if name == "8K":
        return _case(500, 0.5, 2, 11, scale=7680.0)
    if name.startswith("nonfinite-"):                            # nonfinite-{nan,inf,-inf}-{src,dst}
        bad, which = name[len("nonfinite-"):].rsplit("-", 1)
        src, dst = _case(50, 0.5, 0.3, 1)
        (src, dst)[which == "dst"][[3, 7], 0] = float(bad)
        return src, dst
    raise KeyError(name)


EDGES = (["near-collinear", "duplicates", "8K"] + [f"near-collinear-{k}" for k in range(12)] +
         [f"nonfinite-{b}-{w}" for b in ("nan", "inf", "-inf") for w in ("src", "dst")])


def _data(case):
    n, o, s, _, _, _, seed = case
    return _case(n, o, s, seed)


def _assert_same(got_h, got_mask, want_h, want_mask, exact_h=True, what=""):
    assert (got_h is None) == (want_h is None), what
    assert np.array_equal(got_mask, want_mask), what
    if want_h is None:
        return
    assert got_h.dtype == np.float64 and got_h.shape == (3, 3), what
    if exact_h:
        assert np.array_equal(got_h, want_h), (what, np.abs(got_h - want_h).max())
    else:
        assert np.allclose(got_h, want_h, rtol=1e-9, atol=1e-12), (what, np.abs(got_h - want_h).max())


def _best_is_4(rec):
    return rec["best"] >= 0 and rec["counts"][rec["best"]] == 4


def _vs_opencv(src, dst, thr, conf, iters, what):
    want_h, want_mask = cv.findHomography(src, dst, cv.RANSAC, thr, maxIters=iters, confidence=conf)
    h, mask, rec = ro.find_homography(src, dst, thr, conf, iters)
    _assert_same(h, mask, want_h, want_mask, exact_h=not _best_is_4(rec), what=what)
    return rec


# ----------------------------------------------------------------------------------------------- CPU: oracle vs OpenCV
@pytest.mark.parametrize("case", GRID, ids=lambda c: "n{}-o{}-s{}-it{}-c{}-t{}".format(*c[:6]))
def test_oracle_equals_live_opencv_grid(case):
    src, dst = _data(case)
    _vs_opencv(src, dst, case[5], case[4], case[3], str(case))


@pytest.mark.parametrize("c2", C2, ids=lambda c: "o{}-it{}-c{}-t{}".format(*c))
def test_oracle_equals_live_opencv_c2_pairs(c2):
    src, dst = _c2_pairs(c2[0])
    assert len(src) == 3975
    _vs_opencv(src, dst, c2[3], c2[2], c2[1], str(c2))


def test_oracle_pieces_equal_opencv():
    """The minimal-set fit is OpenCV's runKernel bit for bit (findHomography(4 points, 0) runs it alone); the RNG is
    cv::RNG(-1)'s multiply-with-carry."""
    src, dst = _case(200, 0.5, 2, 7)
    subsets, valid, counts, hs = ro.record(src, dst, 3.0, 300)
    assert len(subsets) == 300 and valid.all()
    for s, h in zip(subsets, hs):
        assert np.array_equal(h, cv.findHomography(src[s], dst[s], 0)[0])
    rng = ro.RNG()
    assert rng.next() == (0xFFFFFFFF * 4164903690 + 0xFFFFFFFF) & 0xFFFFFFFF
    assert rng.state == (0xFFFFFFFF * 4164903690 + 0xFFFFFFFF) & ((1 << 64) - 1)
    assert ro.RNG(5).uniform(0, 7) == ((5 * 4164903690) & 0xFFFFFFFF) % 7 and ro.RNG(5).uniform(3, 3) == 3


def _line_but_one(n):
    t = np.arange(n, dtype=np.float32)
    p = np.c_[t, t].astype(np.float32)
    p[n // 2] = (0.0, 1000.0)
    return p


def _first_accept(p):
    rng, attempts = ro.RNG(), 0
    while True:
        attempts += 1
        idx = []
        for _ in range(4):
            j = rng.uniform(0, len(p))
            while j in idx:
                j = rng.uniform(0, len(p))
            idx.append(j)
        if ro.check_subset(p[idx], p[idx]):
            return attempts


def test_jacobi_equals_cv_eigen():
    """The restated cv::eigen on the LtL of every hypothesis of near-collinear sets (almost two-dimensional null
    space) and of an ordinary set: eigenvalues and eigenvectors bit for bit."""
    mats = []
    ltl_of = ro.jacobi

    def spy(a):
        mats.append(np.array(a, np.float64))
        return ltl_of(a)
    ro.jacobi = spy
    try:
        for name in ("near-collinear", "near-collinear-0", "near-collinear-1", "near-collinear-2"):
            ro.record(*_edge(name), 3.0, 60)
        ro.record(*_case(200, 0.5, 2, 7), 3.0, 60)
    finally:
        ro.jacobi = ltl_of
    assert len(mats) >= 200
    for a in mats:
        w, v = ro.jacobi(a)
        _, wc, vc = cv.eigen(np.triu(a) + np.triu(a, 1).T)
        assert np.array_equal(w, wc.ravel()) and np.array_equal(v, vc)


@pytest.mark.parametrize("name", [e for e in EDGES if e.startswith("near-collinear-")])
def test_oracle_equals_live_opencv_near_collinear(name):
    src, dst = _edge(name)
    _vs_opencv(src, dst, 3.0, 0.995, 2000, name)


def test_attempt_limit_is_10000():
    """Points on a line but one, mapped to themselves: a subset passes checkSubset only with the off-line point drawn
    last.  At n = 2000 the first pass takes between 1 000 and 10 000 attempts and OpenCV finds a model; at n = 20000
    it takes more than 10 000 and OpenCV finds none."""
    p = _line_but_one(2000)
    assert 1000 < _first_accept(p) < ro.MAX_ATTEMPTS
    rec = _vs_opencv(p, p, 5.0, 0.995, 2000, "n 2000")
    assert rec["best"] >= 0
    p = _line_but_one(20000)
    assert _first_accept(p) > ro.MAX_ATTEMPTS
    want_h, want_mask = cv.findHomography(p, p, cv.RANSAC, 5.0)
    h, mask, rec = ro.find_homography(p, p, 5.0)
    assert want_h is None and h is None and rec["iterations"] == 0 and not want_mask.any() and not mask.any()


def test_collinear_and_edge_sets():
    t = np.linspace(0, 100, 30, dtype=np.float32)
    line = np.c_[t, 2 * t].astype(np.float32)
    _vs_opencv(line, line, 5.0, 0.995, 2000, "collinear")
    for name in EDGES:
        with np.errstate(all="ignore"):
            _vs_opencv(*_edge(name), 5.0, 0.995, 2000, name)


def test_oracle_scan_and_fewer_than_4_points():
    assert ro.scan([], 10, 0.995, 2000) == (-1, 0)
    assert ro.scan([3, 3, 3], 10, 0.995, 3) == (-1, 3)
    best, it = ro.scan([5, 10, 2, 10], 10, 0.995, 2000)
    assert best == 1 and it == 2                                # all 10 inliers: RANSACUpdateNumIters -> 0
    src, dst = _case(3, 0, 0.3, 1)
    with pytest.raises(cv.error):
        cv.findHomography(src, dst, cv.RANSAC, 5.0)
    with pytest.raises(ValueError):
        ro.find_homography(src, dst)


# ----------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in GRID if c[0] > 4][::2] + ["c2-80"] + EDGES, ids=str)
def test_kernels_equal_oracle_record(case):
    """Subsets, hypotheses (bit for bit), counts, best index and iterations equal the oracle's record."""
    import torch
    from cvx_proj_b200 import _runtime as rt
    if isinstance(case, str):
        src, dst = _c2_pairs(0.8) if case == "c2-80" else _edge(case)
        thr, conf, iters = (5.0, 0.995, 2000) if case == "c2-80" else (3.0, 0.995, 300)
    else:
        src, dst = _data(case)
        thr, conf, iters = float(case[5]), case[4], case[3]
    with np.errstate(all="ignore"):
        subsets, valid, counts, hs = ro.record(src, dst, thr, iters)
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    s_dev, d_dev = torch.from_numpy(src).to(dev), torch.from_numpy(dst).to(dev)
    nb = ctypes_size(lib, iters)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    sub = torch.full((iters, 4), -7, dtype=torch.int32, device=dev)
    hyps = torch.empty((iters, 9), dtype=torch.float64, device=dev)
    cnt = torch.empty(iters, dtype=torch.int32, device=dev)
    ns = torch.empty(1, dtype=torch.int32, device=dev)
    rt.check(lib.apap_ransac_homography(s_dev.data_ptr(), d_dev.data_ptr(), len(src), thr, iters, ws.data_ptr(), nb,
                                        sub.data_ptr(), hyps.data_ptr(), cnt.data_ptr(), ns.data_ptr(),
                                        rt.stream_ptr(torch, dev)), "apap_ransac_homography")
    k = int(ns.item())
    assert k == len(subsets)
    assert np.array_equal(sub.cpu().numpy()[:k], subsets)
    assert np.array_equal(cnt.cpu().numpy()[:k], counts)
    assert np.array_equal(hyps.cpu().numpy()[:k], hs.reshape(-1, 9), equal_nan=True)
    assert np.array_equal(counts == -1, ~valid)
    best, it = ro.scan(counts, len(src), conf, iters)
    with np.errstate(all="ignore"):
        want = ro.find_homography(src, dst, thr, conf, iters)[2]
    assert (best, it) == (want["best"], want["iterations"])


def ctypes_size(lib, iters):
    import ctypes
    from cvx_proj_b200 import _runtime as rt
    nb = ctypes.c_size_t()
    rt.check(lib.apap_ransac_workspace_bytes(iters, ctypes.byref(nb)), "apap_ransac_workspace_bytes")
    return nb.value


@pytest.mark.gpu
@pytest.mark.parametrize("case", GRID, ids=lambda c: "n{}-o{}-s{}-it{}-c{}-t{}".format(*c[:6]))
def test_find_homography_ransac_equals_opencv(case):
    import torch
    from cvx_proj_b200.utils import find_homography_ransac
    src, dst = _data(case)
    thr, conf, iters = case[5], case[4], case[3]
    want_h, want_mask = cv.findHomography(src, dst, cv.RANSAC, thr, maxIters=iters, confidence=conf)
    exact = not _best_is_4(ro.find_homography(src, dst, thr, conf, iters)[2])
    h, mask = find_homography_ransac(src, dst, thr, confidence=conf, max_iters=iters)
    _assert_same(h, mask, want_h, want_mask, exact, f"numpy {case}")
    h, mask = find_homography_ransac(torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda(), thr, confidence=conf,
                                     max_iters=iters)
    _assert_same(h, mask, want_h, want_mask, exact, f"tensor {case}")


@pytest.mark.gpu
@pytest.mark.parametrize("c2", C2, ids=lambda c: "o{}-it{}-c{}-t{}".format(*c))
def test_find_homography_ransac_c2_pairs(c2):
    from cvx_proj_b200.utils import find_homography_ransac
    src, dst = _c2_pairs(c2[0])
    want_h, want_mask = cv.findHomography(src, dst, cv.RANSAC, c2[3], maxIters=c2[1], confidence=c2[2])
    exact = not _best_is_4(ro.find_homography(src, dst, c2[3], c2[2], c2[1])[2])
    h, mask = find_homography_ransac(src, dst, c2[3], confidence=c2[2], max_iters=c2[1])
    _assert_same(h, mask, want_h, want_mask, exact, str(c2))


@pytest.mark.gpu
def test_find_homography_ransac_edge_cases():
    from cvx_proj_b200.utils import find_homography_ransac
    p = _line_but_one(2000)
    for src, dst, what in [(p, p, "attempt limit late"), (_line_but_one(20000), _line_but_one(20000), "no model")]:
        want_h, want_mask = cv.findHomography(src, dst, cv.RANSAC, 5.0)
        h, mask = find_homography_ransac(src, dst, 5.0)
        _assert_same(h, mask, want_h, want_mask, True, what)
    t = np.linspace(0, 100, 30, dtype=np.float32)
    line = np.c_[t, 2 * t].astype(np.float32)
    cases = [(line, line, "collinear")] + [(*_edge(e), e) for e in EDGES]
    for src, dst, what in cases:
        want_h, want_mask = cv.findHomography(src, dst, cv.RANSAC, 5.0)
        with np.errstate(all="ignore"):
            exact = not _best_is_4(ro.find_homography(src, dst, 5.0)[2])
        h, mask = find_homography_ransac(src, dst, 5.0)
        _assert_same(h, mask, want_h, want_mask, exact, what)
    # 4 points: OpenCV's single fit; threshold <= 0 -> 3
    src, dst = _case(4, 0, 0.3, 3)
    _assert_same(*find_homography_ransac(src, dst), *cv.findHomography(src, dst, cv.RANSAC, 5.0), True, "n 4")
    src, dst = _case(100, 0.5, 2, 3)
    _assert_same(*find_homography_ransac(src, dst, 0.0), *cv.findHomography(src, dst, cv.RANSAC, 0.0), True, "thr 0")


@pytest.mark.gpu
def test_find_homography_ransac_errors():
    import torch
    from cvx_proj_b200 import _runtime as rt
    from cvx_proj_b200.utils import find_homography_ransac
    src, dst = _case(20, 0, 0.3, 1)
    with pytest.raises(ValueError, match="at least 4"):
        find_homography_ransac(src[:3], dst[:3])
    with pytest.raises(ValueError, match="at least 4"):
        find_homography_ransac(src, dst[:10])
    with pytest.raises(ValueError, match="confidence"):
        find_homography_ransac(src, dst, confidence=1.0)
    with pytest.raises(ValueError, match="max_iters"):
        find_homography_ransac(src, dst, max_iters=rt.RANSAC_MAX_ITERS + 1)
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    s, d = torch.from_numpy(src).to(dev), torch.from_numpy(dst).to(dev)
    ws = torch.empty(1024, dtype=torch.uint8, device=dev)
    out = torch.empty(64, dtype=torch.int32, device=dev)
    hy = torch.empty(90, dtype=torch.float64, device=dev)
    st = rt.stream_ptr(torch, dev)
    good = [s.data_ptr(), d.data_ptr(), 20, 5.0, 10, ws.data_ptr(), 1024, out.data_ptr(), hy.data_ptr(),
            out.data_ptr() + 160, out.data_ptr() + 200, st]
    rt.check(lib.apap_ransac_homography(*good), "apap_ransac_homography")
    for i, v in ((2, 4), (3, 0.0), (3, float("nan")), (4, 0), (4, rt.RANSAC_MAX_ITERS + 1), (0, None), (5, None),
                 (6, 16), (0, s.data_ptr() + 4), (7, out.data_ptr() + 4), (8, hy.data_ptr() + 4),
                 (9, out.data_ptr() + 162), (10, out.data_ptr() + 202)):
        args = list(good)
        args[i] = v
        with pytest.raises(rt.ApapError):
            rt.check(lib.apap_ransac_homography(*args), "apap_ransac_homography")
    import ctypes
    nb = ctypes.c_size_t()
    with pytest.raises(rt.ApapError):
        rt.check(lib.apap_ransac_workspace_bytes(0, ctypes.byref(nb)), "apap_ransac_workspace_bytes")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c1", "c2", "c2-80"])
def test_keypoint_pairs_gpu_ransac_is_bit_identical(case):
    from cvx_proj_b200.utils import keypoint_pairs
    img_c, img_o, raw_c, raw_o = ts._pair(case[:2])
    if case == "c2-80":                                          # 80 % of the other image's points moved at random
        raw_o = raw_o.copy()
        r = np.random.default_rng(81)
        bad = r.choice(len(raw_o), int(0.8 * len(raw_o)), replace=False)
        raw_o[bad] = (r.random((len(bad), 2)) * [img_o.shape[1], img_o.shape[0]]).astype(np.float32)
    want = keypoint_pairs(img_c, img_o, raw_c, raw_o)
    got = keypoint_pairs(img_c, img_o, raw_c, raw_o, ransac="gpu")
    assert all(np.array_equal(a, b) for a, b in zip(got, want)), case
    with pytest.raises(ValueError, match="ransac"):
        keypoint_pairs(img_c, img_o, raw_c, raw_o, ransac="cpu")
