"""One centre against several images (the reference's multi-image mode, run_all.sh:15,29): the batched RANSAC kernels
(apap_ransac_homography_batch) against the oracle's per-pair record, find_homography_ransac_batch and
keypoint_pairs_batch against their per-pair calls, and driver.stitch_case against stitch_pair(*keypoint_pairs(...)),
each bit for bit."""
import ctypes
import functools

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import synth
from oracle import ransac_oracle as ro
from tests import test_ransac as tr

pytestmark = pytest.mark.gpu


# ----------------------------------------------------------------------------------------------- fixtures
@functools.lru_cache(maxsize=None)
def _scene(name, k):
    """A centre image of the bench shape ``name`` and ``k`` others warped from it by different homographies (rotation,
    shift, a little perspective), with the centre keypoints and their noisy images in each other view."""
    cfg = synth.CONFIGS[name]
    w, h = cfg["width"], cfg["height"]
    centre = synth.make_image(w, h, seed=2)
    r = np.random.default_rng(5)
    raw_c = (r.random((cfg["n_kp"], 2)) * [w - 48, h - 48] + 24).astype(np.float32)
    others, raw_os = [], []
    for j in range(k):
        a = 0.015 * (j + 1) * (-1) ** j
        hom = np.array([[np.cos(a), -np.sin(a), 0.02 * w * (j + 1)], [np.sin(a), np.cos(a), -0.015 * h * (j + 1)],
                        [2e-6 * (j + 1), -3e-6 * j, 1.0]])
        hinv = np.linalg.inv(hom)
        others.append(cv.warpPerspective(centre, hinv, (w, h)))
        raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
        raw_os.append(raw_o + r.normal(0, 0.3, raw_o.shape).astype(np.float32))
    return centre, others, raw_c, raw_os


def _per_pair_centres(raw_c, k):
    """Ragged per-pair centre keypoint sets: a different prefix of the centre keypoints for each pair."""
    return [raw_c[:len(raw_c) - 37 * j] for j in range(k)]


def _lib_batch(sets, thr, iters):
    """``apap_ransac_homography_batch`` on ``[(src, dst), ...]``: per pair ``(subsets, hyps, counts, n_sampled)``."""
    import torch
    from cvx_proj_b200 import _runtime as rt
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    b = len(sets)
    ns = [len(s) for s, _ in sets]
    src = torch.from_numpy(np.concatenate([s for s, _ in sets]).astype(np.float32)).to(dev)
    dst = torch.from_numpy(np.concatenate([d for _, d in sets]).astype(np.float32)).to(dev)
    off = torch.from_numpy(np.cumsum([0] + ns).astype(np.int32)).to(dev)
    nb = ctypes.c_size_t()
    rt.check(lib.apap_ransac_batch_workspace_bytes(b, iters, ctypes.byref(nb)), "apap_ransac_batch_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    sub = torch.full((b, iters, 4), -7, dtype=torch.int32, device=dev)
    hyps = torch.empty((b, iters, 9), dtype=torch.float64, device=dev)
    cnt = torch.empty((b, iters), dtype=torch.int32, device=dev)
    n_s = torch.full((b,), -7, dtype=torch.int32, device=dev)
    rt.check(lib.apap_ransac_homography_batch(src.data_ptr(), dst.data_ptr(), off.data_ptr(), b, max(ns), thr, iters,
                                              ws.data_ptr(), nb.value, sub.data_ptr(), hyps.data_ptr(), cnt.data_ptr(),
                                              n_s.data_ptr(), rt.stream_ptr(torch, dev)),
             "apap_ransac_homography_batch")
    sub, hyps, cnt, n_s = sub.cpu().numpy(), hyps.cpu().numpy(), cnt.cpu().numpy(), n_s.cpu().numpy()
    return [(sub[p], hyps[p], cnt[p], int(n_s[p])) for p in range(b)]


def _ragged_sets():
    """Grid cases of test_ransac, the c2 sets at 0 / 50 / 80 % outliers, near-collinear sets, and 5-, 4- and 3-point
    sets, with names."""
    sets = [(f"grid-{c}", tr._data(c)) for c in tr.GRID if c[0] > 4][::3]
    sets += [(f"c2-{o}", tr._c2_pairs(o)) for o in (0.0, 0.5, 0.8)]
    sets += [(e, tr._edge(e)) for e in ("near-collinear", "near-collinear-0", "near-collinear-1", "duplicates")]
    sets += [("n5", tr._case(5, 0, 0.3, 8)), ("n4", tr._case(4, 0, 0.3, 8)), ("n3", tr._case(3, 0, 0.3, 8))]
    return sets


# ----------------------------------------------------------------------------------------------- kernel record
@pytest.mark.parametrize("iters,which", [(300, "ragged"), (6, "attempt-limit")])
def test_batch_record_equals_oracle(iters, which):
    """Every pair's subsets, n_sampled, hypothesis bits and counts equal the oracle's single-pair record; pairs of 4
    and 3 points are not sampled.  The attempt-limit batch holds a set whose first subset takes 1 000 - 10 000
    candidates, one that never finds one (no model) and an ordinary set."""
    if which == "ragged":
        named = _ragged_sets()
    else:
        p, q = tr._line_but_one(2000), tr._line_but_one(20000)
        named = [("late", (p, p)), ("no-model", (q, q)), ("ordinary", tr._case(200, 0.5, 2, 7))]
    thr = 3.0
    got = _lib_batch([s for _, s in named], thr, iters)
    for (name, (src, dst)), (sub, hyps, cnt, k) in zip(named, got):
        if len(src) < 5:
            assert k == 0, name
            continue
        with np.errstate(all="ignore"):
            subsets, valid, counts, hs = ro.record(src, dst, thr, iters)
        assert k == len(subsets), name
        assert np.array_equal(sub[:k], subsets), name
        assert np.array_equal(cnt[:k], counts), name
        assert np.array_equal(hyps[:k], hs.reshape(-1, 9), equal_nan=True), name
        assert np.array_equal(counts == -1, ~valid), name
    if which == "attempt-limit":
        assert got[0][3] > 0 and got[1][3] == 0


def test_batch_of_one_equals_single_call():
    import torch
    from cvx_proj_b200 import _runtime as rt
    src, dst = tr._c2_pairs(0.5)
    iters, thr = 2000, 5.0
    (sub, hyps, cnt, k), = _lib_batch([(src, dst)], thr, iters)
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    s_dev, d_dev = torch.from_numpy(src).to(dev), torch.from_numpy(dst).to(dev)
    nb = tr.ctypes_size(lib, iters)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    sub1 = torch.full((iters, 4), -7, dtype=torch.int32, device=dev)
    hyps1 = torch.empty((iters, 9), dtype=torch.float64, device=dev)
    cnt1 = torch.empty(iters, dtype=torch.int32, device=dev)
    ns1 = torch.empty(1, dtype=torch.int32, device=dev)
    rt.check(lib.apap_ransac_homography(s_dev.data_ptr(), d_dev.data_ptr(), len(src), thr, iters, ws.data_ptr(), nb,
                                        sub1.data_ptr(), hyps1.data_ptr(), cnt1.data_ptr(), ns1.data_ptr(),
                                        rt.stream_ptr(torch, dev)), "apap_ransac_homography")
    assert k == int(ns1.item()) > 0
    assert np.array_equal(sub[:k], sub1.cpu().numpy()[:k])
    assert np.array_equal(cnt[:k], cnt1.cpu().numpy()[:k])
    assert np.array_equal(hyps[:k].view(np.uint64), hyps1.cpu().numpy()[:k].view(np.uint64))


def test_batch_bad_arguments():
    import torch
    from cvx_proj_b200 import _runtime as rt
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    src, dst = tr._case(20, 0, 0.3, 1)
    s = torch.from_numpy(np.concatenate([src, src])).to(dev)
    d = torch.from_numpy(np.concatenate([dst, dst])).to(dev)
    off = torch.tensor([0, 20, 40], dtype=torch.int32, device=dev)
    nb = ctypes.c_size_t()
    rt.check(lib.apap_ransac_batch_workspace_bytes(2, 10, ctypes.byref(nb)), "apap_ransac_batch_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    out = torch.empty(128, dtype=torch.int32, device=dev)
    hy = torch.empty(180, dtype=torch.float64, device=dev)
    st = rt.stream_ptr(torch, dev)
    good = [s.data_ptr(), d.data_ptr(), off.data_ptr(), 2, 20, 5.0, 10, ws.data_ptr(), nb.value, out.data_ptr(),
            hy.data_ptr(), out.data_ptr() + 320, out.data_ptr() + 400, st]
    rt.check(lib.apap_ransac_homography_batch(*good), "apap_ransac_homography_batch")
    torch.cuda.synchronize()
    assert out[100:102].tolist() == [10, 10]                   # n_sampled of both pairs
    for i, v in ((2, None), (2, off.data_ptr() + 2), (3, 0), (3, rt.RANSAC_MAX_ITERS // 10 + 1), (4, -1), (5, 0.0),
                 (5, float("inf")), (6, 0), (0, None), (7, None), (8, nb.value - 1), (0, s.data_ptr() + 4),
                 (9, out.data_ptr() + 4), (10, hy.data_ptr() + 4), (11, out.data_ptr() + 322),
                 (12, out.data_ptr() + 402)):
        args = list(good)
        args[i] = v
        with pytest.raises(rt.ApapError):
            rt.check(lib.apap_ransac_homography_batch(*args), "apap_ransac_homography_batch")
    for b, it in ((0, 10), (2, 0), (2, rt.RANSAC_MAX_ITERS // 2 + 1)):
        with pytest.raises(rt.ApapError):
            rt.check(lib.apap_ransac_batch_workspace_bytes(b, it, ctypes.byref(nb)), "apap_ransac_batch_workspace_bytes")


# ----------------------------------------------------------------------------------------------- Python batch
def _assert_fit_equal(got, want, what):
    (gh, gm), (wh, wm) = got, want
    assert (gh is None) == (wh is None), what
    assert np.array_equal(gm, wm), what
    if wh is not None:
        assert np.array_equal(gh, wh), what


def test_find_homography_ransac_batch_equals_single_calls():
    """Ragged sets, the no-model case, a best hypothesis of exactly 4 inliers and a 4-point set, as numpy arrays and as
    CUDA tensors, at the c2 threshold and at 1 px."""
    import torch
    from cvx_proj_b200.utils import find_homography_ransac, find_homography_ransac_batch
    q = tr._line_but_one(20000)
    best4 = tr._case(6, 0.5, 3.0, 0)
    four = tr._case(4, 0, 0.3, 3)
    for thr in (5.0, 1.0):
        sets = [s for _, s in _ragged_sets() if len(s[0]) >= 4] + [(q, q), best4, four]
        srcs, dsts = [s for s, _ in sets], [d for _, d in sets]
        with np.errstate(all="ignore"):
            got = find_homography_ransac_batch(srcs, dsts, thr)
            want = [find_homography_ransac(s, d, thr) for s, d in sets]
        for i, (g, w) in enumerate(zip(got, want)):
            _assert_fit_equal(g, w, (thr, i))
        assert got[-3][0] is None and not got[-3][1].any()     # no model
        tens = find_homography_ransac_batch([torch.from_numpy(s).cuda() for s in srcs],
                                            [torch.from_numpy(d).cuda() for d in dsts], thr)
        for i, (g, w) in enumerate(zip(tens, want)):
            _assert_fit_equal(g, w, ("tensor", thr, i))
    # the best hypothesis of best4 at 1 px has exactly 4 inliers: OpenCV LM-refines them, held to 1e-9
    assert tr._best_is_4(ro.find_homography(*best4, 1.0)[2])
    for src, dst in (best4, four):
        want_h, want_mask = cv.findHomography(src, dst, cv.RANSAC, 1.0)
        h, mask = got[-2] if src is best4[0] else got[-1]
        assert np.array_equal(mask, want_mask)
        assert np.allclose(h, want_h, rtol=1e-9, atol=1e-12)


def test_find_homography_ransac_batch_errors():
    from cvx_proj_b200 import _runtime as rt
    from cvx_proj_b200.utils import find_homography_ransac_batch
    src, dst = tr._case(20, 0, 0.3, 1)
    assert find_homography_ransac_batch([], []) == []
    with pytest.raises(ValueError, match="target sets"):
        find_homography_ransac_batch([src, src], [dst])
    with pytest.raises(ValueError, match="pair 1 needs at least 4"):
        find_homography_ransac_batch([src, src[:3]], [dst, dst[:3]])
    with pytest.raises(ValueError, match="pair 0 needs at least 4"):
        find_homography_ransac_batch([src], [dst[:10]])
    with pytest.raises(ValueError, match="confidence"):
        find_homography_ransac_batch([src], [dst], confidence=0.0)
    with pytest.raises(ValueError, match="max_iters"):
        find_homography_ransac_batch([src] * 3, [dst] * 3, max_iters=rt.RANSAC_MAX_ITERS // 2)
    src4, dst4 = tr._case(4, 0, 0.3, 3)                          # 4-point sets are not sampled: no limit to reach
    assert len(find_homography_ransac_batch([src4] * 3, [dst4] * 3, max_iters=rt.RANSAC_MAX_ITERS)) == 3


# ----------------------------------------------------------------------------------------------- producer
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("images", ["numpy", "tensor"])
@pytest.mark.parametrize("centres", ["shared", "per-pair"])
def test_keypoint_pairs_batch_equals_single_calls(ransac, images, centres):
    import torch
    from cvx_proj_b200.utils import keypoint_pairs, keypoint_pairs_batch
    centre, others, raw_c, raw_os = _scene("c1", 3)
    kcs = [raw_c] * 3 if centres == "shared" else _per_pair_centres(raw_c, 3)
    want = [keypoint_pairs(centre, o, kc, ko, ransac=ransac) for o, kc, ko in zip(others, kcs, raw_os)]
    if images == "tensor":
        centre, others = torch.from_numpy(centre).cuda(), [torch.from_numpy(o).cuda() for o in others]
    got = keypoint_pairs_batch(centre, others, raw_c if centres == "shared" else kcs, raw_os, ransac=ransac)
    assert len(got) == 3
    for i, (g, w) in enumerate(zip(got, want)):
        assert all(np.array_equal(a, b) for a, b in zip(g, w)), i
        assert len(g[0]) > 100, i


def test_keypoint_pairs_batch_errors():
    from cvx_proj_b200.utils import keypoint_pairs_batch
    centre, others, raw_c, raw_os = _scene("c1", 3)
    assert keypoint_pairs_batch(centre, [], raw_c, []) == []
    with pytest.raises(ValueError, match="ransac"):
        keypoint_pairs_batch(centre, others, raw_c, raw_os, ransac="cpu")
    with pytest.raises(ValueError, match="keypoint sets"):
        keypoint_pairs_batch(centre, others, raw_c, raw_os[:2])
    with pytest.raises(ValueError, match="centre sets"):
        keypoint_pairs_batch(centre, others, [raw_c] * 2, raw_os)
    with pytest.raises(ValueError, match="pair 1 has 3 matches"):
        keypoint_pairs_batch(centre, others[:2], [raw_c, raw_c[:3]], raw_os[:2])


# ----------------------------------------------------------------------------------------------- driver
def _assert_results_equal(got, want, what):
    assert got.final_size == want.final_size, what
    for field in ("mesh", "vertices", "local_homography", "mat"):
        a, b = getattr(got, field), getattr(want, field)
        assert a.dtype == b.dtype and np.array_equal(a, b), (what, field)
    assert (got.stitched is None) == (want.stitched is None), what
    if want.stitched is not None:
        assert isinstance(got.stitched, np.ndarray) and np.array_equal(got.stitched, want.stitched), what


@pytest.mark.parametrize("name,k,ransac", [("c1", 3, "opencv"), ("c1", 3, "gpu"), ("c2", 2, "gpu"), ("c4", 6, "gpu")])
def test_stitch_case_equals_stitch_pair(name, k, ransac):
    from cvx_proj_b200.driver import stitch_case, stitch_pair
    from cvx_proj_b200.utils import keypoint_pairs
    centre, others, raw_c, raw_os = _scene(name, k)
    kcs = _per_pair_centres(raw_c, k) if name == "c1" else [raw_c] * k     # c4: ragged match counts, 1 762 .. 1 245
    got = stitch_case(centre, others, kcs if name == "c1" else raw_c, raw_os, ransac=ransac)
    assert len(got) == k
    for i, (o, kc, ko) in enumerate(zip(others, kcs, raw_os)):
        want = stitch_pair(centre, o, *keypoint_pairs(centre, o, kc, ko, ransac=ransac))
        _assert_results_equal(got[i], want, (name, i))


def test_stitch_case_options():
    """``stitch=False``, given warp and blend images (the de-hazed pair of the script), another mesh, and errors."""
    from cvx_proj_b200.driver import stitch_case, stitch_pair
    from cvx_proj_b200.utils import keypoint_pairs
    centre, others, raw_c, raw_os = _scene("c1", 3)
    pairs = [keypoint_pairs(centre, o, raw_c, ko) for o, ko in zip(others, raw_os)]
    got = stitch_case(centre, others, raw_c, raw_os, stitch=False, mesh_size=40, gamma=0.3, sigma=60)
    for i, (o, p) in enumerate(zip(others, pairs)):
        _assert_results_equal(got[i], stitch_pair(centre, o, *p, stitch=False, mesh_size=40, gamma=0.3, sigma=60),
                              ("no stitch", i))
    warps = [(255 - o) for o in others]
    blend = synth.make_image(centre.shape[1], centre.shape[0], seed=9)
    got = stitch_case(centre, others, raw_c, raw_os, warp_imgs=warps, blend_img=blend)
    for i, (o, p) in enumerate(zip(others, pairs)):
        _assert_results_equal(got[i], stitch_pair(centre, o, *p, warp_img=warps[i], blend_img=blend), ("given", i))
    assert stitch_case(centre, [], raw_c, []) == []
    with pytest.raises(ValueError, match="warp images"):
        stitch_case(centre, others, raw_c, raw_os, warp_imgs=warps[:2])
