"""SIFT descriptors at given keypoints (cvx_proj_b200.utils.sift_describe, csrc/sift.cu): the numpy restatement
(oracle/sift_oracle.py) against the live cv.SIFT.compute on the CPU, the kernels against the restatement bit for bit
and against OpenCV on the GPU, and coarse_matching(describe="gpu")."""
import functools

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import synth
from oracle import sift_oracle as so

EXACT = {"ramp", "flat"}          # no blur rounding reaches these: OpenCV's bytes exactly


def _gate(got, want, name):
    """max |d| <= 2, >= 99.9 % of the components equal, |d| = 2 in <= 1e-5 of them; ramp and flat exactly equal."""
    assert got.shape == want.shape, name
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    if name in EXACT:
        assert np.array_equal(got, want), name
        return
    assert d.max(initial=0) <= 2, (name, d.max())
    assert (d == 0).mean() >= 0.999, (name, (d == 0).mean())
    assert (d == 2).sum() <= 1e-5 * d.size, (name, (d == 2).sum())


def _cv_describe(img, pts, size=1.0, angle=-1.0):
    kps = [cv.KeyPoint(float(x), float(y), size, angle) for x, y in pts]
    out, feats = cv.SIFT.create(nfeatures=128).compute(img, kps)
    assert len(out) == len(kps)                                   # compute keeps every provided keypoint
    return feats if feats is not None else np.zeros((0, 128), np.float32)


@functools.lru_cache(maxsize=None)
def _pair(name):
    """A synthetic pair of the bench shape ``name`` (tools/n3_host_cost.py): centre image, the other view warped by the
    scene's homography, centre keypoints and their (noisy) images in the other view."""
    sc = synth.make_scene(name)
    rng = np.random.default_rng(1)
    img_c = synth.make_image(sc.width, sc.height, seed=2)
    hinv = np.linalg.inv(sc.h_gt)
    img_o = cv.warpPerspective(img_c, hinv, (sc.width, sc.height))
    raw_c = sc.dst.astype(np.float32)
    raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
    keep = np.all((raw_o > 8) & (raw_o < [sc.width - 8, sc.height - 8]) & (raw_c > 8) & (raw_c < [sc.width - 8, sc.height - 8]),
                  axis=1)
    raw_c, raw_o = raw_c[keep], raw_o[keep]
    raw_o = raw_o + rng.normal(0, 0.3, raw_o.shape).astype(np.float32)
    return img_c, img_o, raw_c, raw_o


def _border_points(h, w):
    """Points on, next to and outside every border, half-pixel positions (cvRound: half to even) included."""
    xs = np.float32([-7, -1, -0.5, 0, 0.5, 1, 1.5, 2.5, w / 2, w - 2.5, w - 1.5, w - 1, w - 0.5, w, w + 4])
    ys = np.float32([-7, -1, -0.5, 0, 0.5, 1, 2.5, h / 2, h - 2.5, h - 1, h - 0.5, h, h + 4])
    return np.stack(np.meshgrid(xs, ys), -1).reshape(-1, 2)


def _case(name):
    """(image, points, size, angle) of the named case."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "c1":
        img, _, pts, _ = _pair("c1")
        return img, pts, 1.0, -1.0
    if name == "c1_other":
        _, img, _, pts = _pair("c1")
        return img, pts, 1.0, -1.0
    if name.startswith("c1_size"):                              # c1_size{s}_angle{a}
        size, angle = name[len("c1_size"):].split("_angle")
        img, _, pts, _ = _pair("c1")
        return img, pts, float(size), float(angle)
    if name == "noise":
        img = rng.integers(0, 256, (97, 131, 3), dtype=np.uint8)
        pts = np.concatenate([rng.uniform(-3, [134, 100], (300, 2)), _border_points(97, 131)]).astype(np.float32)
        return img, pts, 1.0, -1.0
    if name == "ramp":                                          # horizontal gradients only: Ori = 0 -> o0 = -1
        img = np.repeat(np.repeat(np.arange(0, 250, 2, dtype=np.uint8)[None, :, None], 90, 0), 3, 2)
        pts = np.concatenate([rng.uniform(-2, [127, 92], (200, 2)), _border_points(90, 125)]).astype(np.float32)
        return img, pts, 1.0, -1.0
    if name == "flat":
        img = np.full((50, 70, 3), 77, np.uint8)
        return img, _border_points(50, 70), 1.0, -1.0
    if name.startswith("odd"):                                  # odd{h}x{w}: smaller than the blur, multiple reflections
        h, w = (int(v) for v in name[3:].split("x"))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        return img, np.concatenate([rng.uniform(-2, [w + 1, h + 1], (40, 2)), _border_points(h, w)]).astype(np.float32), 1.0, -1.0
    raise KeyError(name)


CASES = ["c1", "c1_other", "noise", "ramp", "flat", "odd9x7", "odd5x13", "odd3x2", "odd1x1", "odd16x1", "odd211x173"] + \
        [f"c1_size{s}_angle{a}" for s in (2.0, 3.0) for a in (-1.0, 0.0, 45.0, 200.0)]


# ----------------------------------------------------------------------------------------------- CPU: oracle vs OpenCV
def test_gray_and_taps_bit_exact_with_opencv():
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (64, 256, 3), dtype=np.uint8)
    img[0, :, :] = 255; img[1, :, :] = 0
    assert np.array_equal(so.gray(img), cv.cvtColor(img, cv.COLOR_BGR2GRAY))
    taps = so.gaussian_taps()
    want = cv.getGaussianKernel(13, float(so.blur_sigma()), cv.CV_32F).ravel()
    assert taps.shape == (13,) and np.array_equal(taps.view(np.uint32), want.view(np.uint32))
    assert so.blur_sigma() == np.float32(1.5198685)


def test_kernel_taps_are_opencvs():
    """The 13 taps written into csrc/sift.cu as float literals are cv.getGaussianKernel's bits."""
    import os
    import re
    src = open(os.path.join(os.path.dirname(__file__), "..", "cvx_proj_b200", "csrc", "sift.cu")).read()
    body = re.search(r"kSiftTaps\[[^\]]*\]\s*=\s*\{([^}]*)\}", src).group(1)
    lits = np.float32([float.fromhex(t.strip().rstrip("f")) for t in body.split(",")])
    want = cv.getGaussianKernel(13, float(so.blur_sigma()), cv.CV_32F).ravel()
    assert np.array_equal(lits.view(np.uint32), want.view(np.uint32))


def test_host_sample_table_equals_the_oracle_loop():
    from cvx_proj_b200.utils import sift_sample_table
    for size in (1.0, 2.0, 3.0, 0.3, 7.5):
        for angle in (-1.0, 0.0, 45.0, 200.0, 359.5):
            for hw in ((2160, 3840), (3, 2), (1, 1)):
                got, ori = sift_sample_table(size, angle, *hw)
                want, want_ori = so.sample_table(size, angle, *hw)
                assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))
                assert ori == want_ori
    assert sift_sample_table(1.0, -1.0, 768, 1024)[1] == np.float32(361.0)
    assert sift_sample_table(1.0, 0.0, 768, 1024)[1] == 0.0


@pytest.mark.parametrize("name", CASES)
def test_oracle_vs_live_opencv(name):
    img, pts, size, angle = _case(name)
    _gate(so.describe(img, pts, size, angle), _cv_describe(img, pts, size, angle), name)


def test_oracle_vs_live_opencv_c2_pair():
    """The bench shape c2 (3840 x 2160, about 4 000 keypoints), both views; the exact matcher picks the same train index
    on the restated descriptors as on OpenCV's for >= 99.5 % of the queries."""
    img_c, img_o, raw_c, raw_o = _pair("c2")
    fc, fo = so.describe(img_c, raw_c), so.describe(img_o, raw_o)
    wc, wo = _cv_describe(img_c, raw_c), _cv_describe(img_o, raw_o)
    _gate(fc, wc, "c2 centre")
    _gate(fo, wo, "c2 other")
    got = [m.trainIdx for m in cv.BFMatcher(cv.NORM_L2).match(fc, fo)]
    want = [m.trainIdx for m in cv.BFMatcher(cv.NORM_L2).match(wc, wo)]
    assert np.mean(np.equal(got, want)) >= 0.995


def test_ramp_takes_the_o0_minus_one_path():
    """On a horizontal ramp every gradient has Ori = 0, which with angle -1 (ori = 361) gives o0 = -1: the first trilinear
    contribution lands in bin n+1 of the previous cell and is folded into its bin 1.  The restatement keeps that and
    equals OpenCV."""
    img, pts, size, angle = _case("ramp")
    got = so.describe(img, pts, size, angle)
    assert got.any() and np.array_equal(got, _cv_describe(img, pts))
    inner = got[(pts[:, 0] > 8) & (pts[:, 0] < 116) & (pts[:, 1] > 8) & (pts[:, 1] < 81)]
    assert len(inner) and (inner.reshape(-1, 16, 8)[:, :, 1] > 0).any()


# --------------------------------------------------------------------------------------------------------- GPU
def _kernel_base(img):
    """base_scratch of apap_sift_describe for one keypoint: the blurred gray image the descriptors read."""
    import torch
    from cvx_proj_b200 import _runtime as rt
    from cvx_proj_b200.utils import sift_sample_table
    torch_, dev = rt.torch_cuda()
    h, w = img.shape[:2]
    table, ori = sift_sample_table(1.0, -1.0, h, w)
    d_img = torch.from_numpy(img).to(dev)
    d_pts = torch.zeros((1, 2), dtype=torch.float32, device=dev)
    d_tab = torch.from_numpy(table).to(dev)
    base = torch.full((h, w), float("nan"), dtype=torch.float32, device=dev)
    desc = torch.empty((1, 128), dtype=torch.float32, device=dev)
    lib = rt.load_library()
    rt.check(lib.apap_sift_describe(d_img.data_ptr(), h, w, d_pts.data_ptr(), 1, d_tab.data_ptr(), table.shape[0], float(ori),
                                    base.data_ptr(), desc.data_ptr(), rt.stream_ptr(torch_, dev)), "apap_sift_describe")
    return base.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_kernel_equals_oracle_and_opencv(name):
    from cvx_proj_b200.utils import sift_describe
    img, pts, size, angle = _case(name)
    got = sift_describe(img, pts, size, angle)
    want = so.describe(img, pts, size, angle)
    assert got.dtype == np.float32 and got.shape == (len(pts), 128)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), name
    _gate(got, _cv_describe(img, pts, size, angle), name)
    base = _kernel_base(img)
    assert np.array_equal(base.view(np.uint32), so.base_image(img).view(np.uint32)), name


@pytest.mark.gpu
def test_kernel_c2_pair_equals_oracle_and_opencv():
    from cvx_proj_b200.utils import sift_describe
    img_c, img_o, raw_c, raw_o = _pair("c2")
    for img, pts, name in ((img_c, raw_c, "c2 centre"), (img_o, raw_o, "c2 other")):
        got = sift_describe(img, pts)
        assert np.array_equal(got.view(np.uint32), so.describe(img, pts).view(np.uint32)), name
        _gate(got, _cv_describe(img, pts), name)
    assert np.array_equal(_kernel_base(img_c).view(np.uint32), so.base_image(img_c).view(np.uint32))


@pytest.mark.gpu
def test_sift_describe_tensors_keypoint_lists_and_edge_cases():
    import torch
    from cvx_proj_b200.utils import sift_describe
    img, pts, _, _ = _case("c1")
    want = so.describe(img, pts)
    dev = torch.device("cuda", torch.cuda.current_device())
    d_img = torch.from_numpy(img).to(dev)
    got = sift_describe(d_img, torch.from_numpy(pts).to(dev))               # CUDA tensors in -> stays on the device
    assert got.is_cuda and got.dtype == torch.float32 and np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(sift_describe(d_img, pts).cpu().numpy(), want)  # host points, device image
    kps = [cv.KeyPoint(float(x), float(y), 1) for x, y in pts]
    assert np.array_equal(sift_describe(img, kps), want)
    kps2 = [cv.KeyPoint(float(x), float(y), 2.0, 45.0) for x, y in pts[:50]]
    assert np.array_equal(sift_describe(img, kps2), so.describe(img, pts[:50], 2.0, 45.0))
    out = sift_describe(img, np.zeros((0, 2), np.float32))                # K = 0
    assert out.shape == (0, 128) and out.dtype == np.float32
    assert sift_describe(img, []).shape == (0, 128)
    one = sift_describe(img, pts[:1])                                     # K = 1
    assert one.shape == (1, 128) and np.array_equal(one, want[:1])
    assert not sift_describe(img, np.float32([[-50, -50], [np.nan, 3], [np.inf, 1e30]])).any()
    with pytest.raises(ValueError, match="mixed sizes"):
        sift_describe(img, [cv.KeyPoint(10, 10, 1), cv.KeyPoint(20, 20, 2)])
    with pytest.raises(ValueError, match="mixed angles"):
        sift_describe(img, [cv.KeyPoint(10, 10, 1, 0), cv.KeyPoint(20, 20, 1, 90)])
    with pytest.raises(ValueError, match="octave"):
        sift_describe(img, [cv.KeyPoint(10, 10, 1, -1, 0, 1)])
    with pytest.raises(ValueError, match="angle"):
        sift_describe(img, pts, angle=400.0)
    with pytest.raises(ValueError, match="size"):
        sift_describe(img, pts, size=0.0)
    with pytest.raises(ValueError, match="uint8"):
        sift_describe(img.astype(np.float32), pts)


@pytest.mark.gpu
def test_coarse_matching_describe_gpu_on_a_synthetic_pair():
    """coarse_matching(describe="gpu") on the c1 pair of the OpenCV-descriptor mirror test: same return layout, nearly
    all matches the true correspondences, cv.findHomography recovers the homography, and the train index equals the
    describe="opencv" path for >= 99.5 % of the queries."""
    from cvx_proj_b200.utils import coarse_matching
    sc = synth.make_scene("c1")
    img_c = synth.make_image(sc.width, sc.height, seed=2)
    hinv = np.linalg.inv(sc.h_gt)
    img_o = cv.warpPerspective(img_c, hinv, (sc.width, sc.height))
    raw_c = sc.dst.astype(np.float32)
    raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
    keep = np.all((raw_o > 16) & (raw_o < [sc.width - 16, sc.height - 16]) & (raw_c > 16) & (raw_c < [sc.width - 16, sc.height - 16]), axis=1)
    raw_c, raw_o = raw_c[keep], raw_o[keep]
    kc, fc, ko, fo, matches = coarse_matching(img_c, img_o, raw_c, raw_o, describe="gpu")
    assert len(matches) == len(kc) == fc.shape[0] and all(isinstance(m, cv.DMatch) for m in matches)
    assert fc.dtype == np.float32 and fc.shape[1] == 128 and fo.shape == (len(ko), 128)
    assert all(isinstance(k, cv.KeyPoint) for k in kc)
    assert np.array_equal(fc, so.describe(img_c, raw_c)) and np.array_equal(fo, so.describe(img_o, raw_o))
    bf = cv.BFMatcher(cv.NORM_L2).match(fc, fo)
    assert [m.trainIdx for m in matches] == [m.trainIdx for m in bf]
    assert np.mean([m.trainIdx == m.queryIdx for m in matches]) > 0.8
    src = np.float32([kc[m.queryIdx].pt for m in matches]); dst = np.float32([ko[m.trainIdx].pt for m in matches])
    h, mask = cv.findHomography(src, dst, cv.RANSAC, 5.0)
    assert mask.sum() > 0.8 * len(matches) and np.abs(h / h[2, 2] - hinv / hinv[2, 2]).max() < 0.05 * np.abs(hinv / hinv[2, 2]).max()
    ref = coarse_matching(img_c, img_o, raw_c, raw_o)[4]
    assert np.mean([a.trainIdx == b.trainIdx for a, b in zip(matches, ref)]) >= 0.995
    with pytest.raises(ValueError, match="describe"):
        coarse_matching(img_c, img_o, raw_c, raw_o, describe="cuda")
