"""Per-channel histogram equalisation (cvx_proj_b200.utils.equalize_hist, csrc/equalize.cu), SIFT description through
the equalisation LUT (sift_describe(..., equalize=True)) and the array-level keypoint-pair producer
(utils.keypoint_pairs): the numpy restatement (oracle/equalize_oracle.py) against the live cv.equalizeHist on the CPU,
the kernels against it and against OpenCV on the GPU."""
import functools

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import synth
from oracle import equalize_oracle as eo
from oracle import sift_oracle as so
from tests import test_sift as ts


def _cv_equalize(img):
    return cv.merge([cv.equalizeHist(c) for c in cv.split(img)])


@functools.lru_cache(maxsize=None)
def _image(name):
    """The named test image, uint8 [H, W, 3]."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "noise":                                          # 3 w = 903: not a multiple of 16
        return rng.integers(0, 256, (200, 301, 3), dtype=np.uint8)
    if name == "flat":                                           # every channel takes OpenCV's setTo path
        return np.full((64, 80, 3), 77, np.uint8)
    if name == "one_flat":                                       # channel 1 flat, the other two not
        img = rng.integers(0, 256, (50, 61, 3), dtype=np.uint8)
        img[..., 1] = 200
        return img
    if name == "1x1":
        return np.uint8([[[3, 200, 255]]])
    if name == "1xN":
        return rng.integers(0, 256, (1, 37, 3), dtype=np.uint8)
    if name == "two_valued":
        return np.where(rng.random((33, 47, 3)) < 0.3, 10, 240).astype(np.uint8)
    if name == "bin0":                                           # bin 0 populated in every channel
        img = rng.integers(0, 256, (41, 53, 3), dtype=np.uint8)
        img[::7, ::5] = 0
        return img
    if name == "only255":                                        # only bin 255 populated
        return np.full((19, 23, 3), 255, np.uint8)
    if name == "skewed":                                         # a narrow normal: large jumps in the LUT
        return np.clip(rng.normal(60, 12, (300, 257, 3)), 0, 255).astype(np.uint8)
    if name in ("c1", "c2", "c3"):                               # values in 1..255: i0 >= 1
        w, h = {"c1": (1024, 768), "c2": (3840, 2160), "c3": (7680, 4320)}[name]
        return synth.make_image(w, h, seed=2)
    if name.startswith("odd"):                                   # odd{h}x{w}
        h, w = (int(v) for v in name[3:].split("x"))
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if name == "big":                                            # 18 M pixels per channel: sums > 2^24 round to float
        img = np.empty((4500, 4000, 3), np.uint8)
        for c in range(3):
            img[..., c] = np.clip(rng.normal(100 + 40 * c, 30 + 10 * c, (4500, 4000)), 0, 255).astype(np.uint8)
        return img
    raise KeyError(name)


CASES = ["noise", "flat", "one_flat", "1x1", "1xN", "two_valued", "bin0", "only255", "skewed", "c1", "c2",
         "odd7x5", "odd13x11", "odd1x17", "big"]


# ----------------------------------------------------------------------------------------------- CPU: oracle vs OpenCV
@pytest.mark.parametrize("name", CASES)
def test_oracle_equals_live_opencv(name):
    img = _image(name)
    assert np.array_equal(eo.equalize(img), _cv_equalize(img)), name


def test_oracle_lut_paths():
    """setTo path (all i0), lut[i0] = 0 with the top bin at 255, and the int -> float rounding above 2^24."""
    flat = eo.luts(_image("only255"))
    assert (flat == 255).all()
    lut = eo.channel_lut(np.bincount([5, 5, 9, 200], minlength=256))
    assert lut[5] == 0 and lut[9] == 128 and lut[200] == 255 and lut[199] == 128
    big = _image("big")
    hist = eo.histograms(big)
    assert hist.sum(axis=1).tolist() == [4500 * 4000] * 3 and (hist.cumsum(axis=1) > 1 << 24).any()


# --------------------------------------------------------------------------------------------------------- GPU
def _lib_equalize(img_dev, out=None):
    """(hist, lut) of apap_equalize_hist on a device image, and the image written to ``out`` when given."""
    import torch
    from cvx_proj_b200 import _runtime as rt
    torch_, dev = rt.torch_cuda(img_dev.device)
    hist = torch.full((768,), 12345, dtype=torch.int32, device=dev)   # the launcher zeroes it
    lut = torch.empty(768, dtype=torch.uint8, device=dev)
    rt.check(rt.load_library().apap_equalize_hist(img_dev.data_ptr(), img_dev.shape[0], img_dev.shape[1], hist.data_ptr(),
                                                  lut.data_ptr(), out, rt.stream_ptr(torch_, dev)), "apap_equalize_hist")
    return hist.cpu().numpy().reshape(3, 256), lut.cpu().numpy().reshape(3, 256)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_kernel_hist_and_lut_equal_oracle(name):
    import torch
    img = _image(name)
    hist, lut = _lib_equalize(torch.from_numpy(img).cuda())
    assert np.array_equal(hist.astype(np.int64), eo.histograms(img)), name
    assert np.array_equal(lut, eo.luts(img)), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES + ["c3"])
def test_equalize_hist_equals_opencv(name):
    from cvx_proj_b200.utils import equalize_hist
    img = _image(name)
    got = equalize_hist(img)
    assert got.dtype == np.uint8 and got.shape == img.shape
    assert np.array_equal(got, _cv_equalize(img)), name


@pytest.mark.gpu
def test_equalize_hist_tensors_and_unaligned_views():
    import torch
    from cvx_proj_b200.utils import equalize_hist
    img = _image("odd211x173")                                   # 3 w = 519 bytes per row
    dev = torch.device("cuda", torch.cuda.current_device())
    d_img = torch.from_numpy(img).to(dev)
    got = equalize_hist(d_img)
    assert got.is_cuda and got.dtype == torch.uint8 and np.array_equal(got.cpu().numpy(), _cv_equalize(img))
    for r0 in (1, 2, 5):                                          # views whose base is not 16-byte aligned
        view = d_img[r0:]
        assert view.data_ptr() % 16 != 0
        want = _cv_equalize(np.ascontiguousarray(img[r0:]))
        assert np.array_equal(equalize_hist(view).cpu().numpy(), want), r0
        # an output of the same 16-byte phase takes the vector path with an unaligned head
        buf = torch.zeros(view.numel() + 32, dtype=torch.uint8, device=dev)
        at = (view.data_ptr() - buf.data_ptr()) % 16
        hist, lut = _lib_equalize(view, buf.data_ptr() + at)
        assert buf.data_ptr() + at != view.data_ptr() and (buf.data_ptr() + at - view.data_ptr()) % 16 == 0
        out = buf[at:at + view.numel()].view(view.shape).cpu().numpy()
        assert np.array_equal(out, want) and np.array_equal(lut, eo.luts(img[r0:])), r0
        assert not buf[:at].any() and not buf[at + view.numel():].any()
    with pytest.raises(ValueError, match="uint8"):
        equalize_hist(img.astype(np.float32))
    with pytest.raises(ValueError, match="uint8"):
        equalize_hist(img[..., :2])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ts.CASES)
def test_sift_describe_equalize_equals_equalized_image(name):
    from cvx_proj_b200.utils import equalize_hist, sift_describe
    img, pts, size, angle = ts._case(name)
    got = sift_describe(img, pts, size, angle, equalize=True)
    eq = equalize_hist(img)
    assert np.array_equal(got.view(np.uint32), sift_describe(eq, pts, size, angle).view(np.uint32)), name
    assert np.array_equal(got.view(np.uint32), so.describe(_cv_equalize(img), pts, size, angle).view(np.uint32)), name
    ts._gate(got, ts._cv_describe(_cv_equalize(img), pts, size, angle), name + " equalised")


@pytest.mark.gpu
def test_sift_describe_equalize_c2_pair_and_tensors():
    import torch
    from cvx_proj_b200.utils import equalize_hist, sift_describe
    img_c, img_o, raw_c, raw_o = ts._pair("c2")
    for img, pts, name in ((img_c, raw_c, "c2 centre"), (img_o, raw_o, "c2 other")):
        got = sift_describe(img, pts, equalize=True)
        assert np.array_equal(got.view(np.uint32), sift_describe(equalize_hist(img), pts).view(np.uint32)), name
        ts._gate(got, ts._cv_describe(_cv_equalize(img), pts), name + " equalised")
    d_img = torch.from_numpy(img_c).cuda()
    got = sift_describe(d_img, torch.from_numpy(raw_c).cuda(), equalize=True)
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), sift_describe(img_c, raw_c, equalize=True))
    assert sift_describe(img_c, np.zeros((0, 2), np.float32), equalize=True).shape == (0, 128)


def _chain(img_c, img_o, raw_c, raw_o):
    """keypoint_pairs written out: equalize_hist -> sift_describe -> match_descriptors -> findHomography -> inv."""
    from cvx_proj_b200.utils import equalize_hist, match_descriptors, sift_describe
    fc = sift_describe(equalize_hist(img_c), raw_c)
    fo = sift_describe(equalize_hist(img_o), raw_o)
    idx, _ = match_descriptors(fc, fo)
    q = np.flatnonzero(idx >= 0)
    centre, other = raw_c[q], raw_o[idx[q]]
    h, mask = cv.findHomography(centre, other, cv.RANSAC, 5.0)
    mask = mask.ravel().astype(bool)
    return other[mask], centre[mask], np.linalg.inv(h)


def _corners_px(h_a, h_b, w, h):
    c = np.float64([[0, 0], [w, 0], [w, h], [0, h]])[None]
    return np.abs(cv.perspectiveTransform(c, h_a) - cv.perspectiveTransform(c, h_b)).max()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c1", "c2"])
def test_keypoint_pairs_equals_the_written_out_chain_and_opencv(case):
    from cvx_proj_b200.utils import keypoint_pairs
    img_c, img_o, raw_c, raw_o = ts._pair(case)
    src, dst, h = keypoint_pairs(img_c, img_o, raw_c, raw_o)
    w_src, w_dst, w_h = _chain(img_c, img_o, raw_c, raw_o)
    assert src.dtype == dst.dtype == np.float32 and h.dtype == np.float64 and h.shape == (3, 3)
    assert np.array_equal(src, w_src) and np.array_equal(dst, w_dst) and np.array_equal(h, w_h)
    assert len(src) > 0.75 * len(raw_c)
    # the all-OpenCV chain: cv.equalizeHist, cv.SIFT.compute, cv.BFMatcher, findHomography
    ext = cv.SIFT.create(nfeatures=128)
    _, fc = ext.compute(_cv_equalize(img_c), [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_c])
    _, fo = ext.compute(_cv_equalize(img_o), [cv.KeyPoint(float(x), float(y), 1) for x, y in raw_o])
    cv_idx = np.array([m.trainIdx for m in cv.BFMatcher(cv.NORM_L2).match(fc, fo)])
    from cvx_proj_b200.utils import equalize_hist, match_descriptors, sift_describe
    idx, _ = match_descriptors(sift_describe(equalize_hist(img_c), raw_c), sift_describe(equalize_hist(img_o), raw_o))
    assert np.mean(idx == cv_idx) >= 0.995
    hc, mask = cv.findHomography(raw_c, raw_o[cv_idx], cv.RANSAC, 5.0)
    assert _corners_px(h, np.linalg.inv(hc), img_o.shape[1], img_o.shape[0]) < 1.0


@pytest.mark.gpu
def test_keypoint_pairs_equalize_false_empty_and_errors():
    import torch
    from cvx_proj_b200 import _runtime as rt
    from cvx_proj_b200.utils import keypoint_pairs
    img_c, img_o, raw_c, raw_o = ts._pair("c1")
    want = keypoint_pairs(img_c, img_o, raw_c, raw_o)
    got = keypoint_pairs(_cv_equalize(img_c), _cv_equalize(img_o), raw_c, raw_o, equalize=False)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    d_got = keypoint_pairs(torch.from_numpy(img_c).cuda(), torch.from_numpy(img_o).cuda(), raw_c, raw_o)
    assert all(np.array_equal(a, b) for a, b in zip(d_got, want))
    with pytest.raises(ValueError, match="matches"):
        keypoint_pairs(img_c, img_o, np.zeros((0, 2), np.float32), raw_o)
    with pytest.raises(ValueError, match="matches"):
        keypoint_pairs(img_c, img_o, raw_c[:3], raw_o)
    with pytest.raises(ValueError, match="matches"):
        keypoint_pairs(img_c, img_o, raw_c, np.zeros((0, 2), np.float32))
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    img = torch.zeros((4, 4, 3), dtype=torch.uint8, device=dev)
    hist = torch.empty(768, dtype=torch.int32, device=dev)
    lut = torch.empty(768, dtype=torch.uint8, device=dev)
    st = rt.stream_ptr(torch, dev)
    for args in ((None, 4, 4, hist.data_ptr(), lut.data_ptr()), (img.data_ptr(), 4, 4, None, lut.data_ptr()),
                 (img.data_ptr(), 4, 4, hist.data_ptr(), None), (img.data_ptr(), 0, 4, hist.data_ptr(), lut.data_ptr()),
                 (img.data_ptr(), 4, -1, hist.data_ptr(), lut.data_ptr()),
                 (img.data_ptr(), 1 << 16, 1 << 15, hist.data_ptr(), lut.data_ptr())):           # h w > INT_MAX
        with pytest.raises(rt.ApapError):
            rt.check(lib.apap_equalize_hist(*args, None, st), "apap_equalize_hist")
    from cvx_proj_b200.utils import sift_sample_table
    table, ori = sift_sample_table(1.0, -1.0, 4, 4)
    d_tab = torch.from_numpy(table).to(dev)
    pts = torch.zeros((1, 2), dtype=torch.float32, device=dev)
    base = torch.empty((4, 4), dtype=torch.float32, device=dev)
    desc = torch.empty((1, 128), dtype=torch.float32, device=dev)
    for lut_p, h in ((None, 4), (lut.data_ptr(), 1 << 24), (lut.data_ptr(), 0)):
        with pytest.raises(rt.ApapError):
            rt.check(lib.apap_sift_describe_lut(img.data_ptr(), h, 4, lut_p, pts.data_ptr(), 1, d_tab.data_ptr(),
                                                int(table.shape[0]), float(ori), base.data_ptr(), desc.data_ptr(), st),
                     "apap_sift_describe_lut")
