"""Exposure compensation of a panorama: ``oracle.gain_oracle`` pinned against the live ``cv.detail.GainCompensator``
(gains, ``apply`` and the whole compensate-then-feather chain), the statistics kernel (``k_gain_stats``) and the blends
with gains against the oracle, and ``driver.stitch_panorama(exposure="gain")`` against the oracle composite."""
import ctypes
import re

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import _runtime as rt
from cvx_proj_b200 import synth
from oracle import feather_oracle as fo
from oracle import gain_oracle as go
from tests.test_feather import _cases
from tests.test_panorama import _random_case, _random_image, _scene_2d

gpu = pytest.mark.gpu


def _masks(ps):
    return [np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8) for p in ps]


def _opencv_gains(layers, origins, size):
    """GainCompensator() fed as exposure_gains' contract says: every layer pasted into the canvas."""
    ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
    comp = cv.detail.GainCompensator()
    comp.feed([(0, 0)] * len(ps), [cv.UMat(p) for p in ps], [cv.UMat(m) for m in _masks(ps)])
    return np.asarray(comp.getMatGains(), dtype=np.float64).reshape(-1)


def _opencv_chain(layers, origins, size, sharpness=0.02):
    """OpenCV's pipeline: feed, apply per layer, FeatherBlender fed the compensated layers with the original masks.
    Returns (panorama, OpenCV's gains)."""
    ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
    ms = _masks(ps)
    comp = cv.detail.GainCompensator()
    comp.feed([(0, 0)] * len(ps), [cv.UMat(p) for p in ps], [cv.UMat(m) for m in ms])
    blender = cv.detail.FeatherBlender(sharpness)
    blender.prepare((0, 0, size[0], size[1]))
    for k, (p, m) in enumerate(zip(ps, ms)):
        blender.feed(comp.apply(k, (0, 0), p.copy(), m).astype(np.int16), m, (0, 0))
    res, _ = blender.blend(None, None)
    return res.astype(np.uint8), np.asarray(comp.getMatGains(), dtype=np.float64).reshape(-1)


def _extra_cases():
    """(name, layers, origins, size) beyond test_feather's shapes."""
    r = np.random.default_rng(17)
    out = []
    a, b = _random_image(r, 20, 30, black=0.0), _random_image(r, 20, 30, black=0.0)
    out.append(("disjoint", [a, b], [(0, 0), (40, 25)], (80, 50)))
    c = _random_image(r, 30, 40, black=0.0)
    c[:, 20:] = 0                                    # the rectangles overlap, the masks do not: N = 1
    d = _random_image(r, 30, 20, black=0.0)
    out.append(("rects-meet-masks-not", [c, d, _random_image(r, 25, 25)], [(0, 0), (20, 0), (10, 5)], (45, 35)))
    out.append(("all-zero", [_random_image(r, 30, 30), np.zeros((20, 20, 3), np.uint8), _random_image(r, 25, 25)],
                [(0, 0), (5, 5), (10, 3)], (40, 35)))
    out.append(("one", [_random_image(r, 33, 45)], [(0, 0)], (45, 33)))
    out.append(("c1-scene", *_scene_layers("c1", 3)))
    return out


def _scene_layers(name, k):
    """Brightness-shifted layers of a synthetic scene of the size of ``name``: the centre and ``k`` shifted copies, each
    scaled by its own factor, the way hazy photographs of one case differ."""
    cfg = synth.CONFIGS[name]
    w, h = cfg["width"], cfg["height"]
    centre = synth.make_image(w, h, seed=2)
    layers, origins = [], []
    for j in range(k):
        f = 0.75 + 0.15 * j
        layers.append(np.clip(np.rint(centre * f), 0, 255).astype(np.uint8))
        origins.append((int((j - k / 2) * 0.15 * w), int((-1) ** j * 0.1 * h)))
    layers.append(centre)
    origins.append((int(0.2 * w), int(0.15 * h)))
    xs = [o[0] for o in origins]
    ys = [o[1] for o in origins]
    origins = [(x - min(xs), y - min(ys)) for x, y in origins]
    return layers, origins, (max(xs) - min(xs) + w, max(ys) - min(ys) + h)


def _all_cases():
    return _cases() + _extra_cases()


# ----------------------------------------------------------------------------------------------- CPU
def test_opencv_build_solves_without_eigen():
    """With Eigen, singleFeed solves with a float32 LLT instead of cv::solve; the oracle restates the cv::solve path."""
    assert re.search(r"Eigen:\s+NO", cv.getBuildInformation())


CASE_NAMES = ("ragged", "wide", "holes", "full", "one", "tall", "disjoint", "rects-meet-masks-not", "all-zero", "one",
              "c1-scene")


def test_case_names_cover_every_case():
    assert tuple(c[0] for c in _all_cases()) == CASE_NAMES


@pytest.mark.parametrize("case", range(len(CASE_NAMES)), ids=[f"{k}-{n}" for k, n in enumerate(CASE_NAMES)])
def test_oracle_gains_are_opencv(case):
    name, layers, origins, size = _all_cases()[case]
    want = _opencv_gains(layers, origins, size)
    got = go.gains(layers, origins, size)
    assert got.shape == want.shape and np.allclose(got, want, rtol=1e-12, atol=0), (name, got, want)
    if name == "disjoint":
        assert (got == 1).all()
    if name == "all-zero":
        assert got[1] == 1
    if name == "one":
        assert (got == 1).all()
    if name == "rects-meet-masks-not":
        count, _ = go.stats(layers, origins, size)
        assert count[0][1] == 0 and count[0][2] > 0 and count[1][2] > 0


@pytest.mark.parametrize("case", range(len(CASE_NAMES)), ids=[f"{k}-{n}" for k, n in enumerate(CASE_NAMES)])
def test_shipped_solve_is_opencv(case):
    """utils.solve_gains (the host half of exposure_gains) fed the exact statistics gives getMatGains()."""
    from cvx_proj_b200.utils import solve_gains
    name, layers, origins, size = _all_cases()[case]
    got = solve_gains(*go.stats(layers, origins, size))
    want = _opencv_gains(layers, origins, size)
    assert got.dtype == np.float64 and np.allclose(got, want, rtol=1e-12, atol=0), (name, got, want)
    assert np.array_equal(got, go.gains(layers, origins, size)), name


def test_oracle_sums_are_fsum():
    import math
    name, layers, origins, size = _cases()[0]
    count, sums = go.stats(layers, origins, size)
    ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
    ms = [p.max(axis=-1) > 0 for p in ps]
    for i, j in ((0, 1), (1, 0), (2, 5), (7, 3)):
        both = ms[i] & ms[j]
        norms = np.sqrt((ps[i][both].astype(np.int64) ** 2).sum(axis=-1).astype(np.float64))
        assert float(sums[i][j]) * 2.0 ** -52 == math.fsum(norms), (i, j)


def test_scaled_sqrt_is_an_integer_below_2_61():
    q = np.arange(1, 3 * 255 * 255 + 1, dtype=np.float64)
    e = np.sqrt(q) * 2.0 ** 52
    assert (e == np.floor(e)).all() and e.max() < 2.0 ** 61 and e.min() >= 2.0 ** 52


def test_apply_is_opencv_apply():
    r = np.random.default_rng(3)
    v = np.arange(256, dtype=np.uint8).reshape(1, 256, 1).repeat(3, axis=2)
    mask = np.full((1, 256), 255, np.uint8)
    comp = cv.detail.GainCompensator()
    for g in [0.5, 1.5, 2.5, 0.3, 3.0, 1.0, 0.0] + list(r.uniform(0.2, 3.0, 2000)):
        comp.setMatGains(np.array([[g]]))
        want = comp.apply(0, (0, 0), v.copy(), mask)
        assert np.array_equal(go.apply(v, g), want), g


@pytest.mark.parametrize("sharpness", [0.02, 1.0])
def test_oracle_composite_is_opencv_chain(sharpness):
    """Equal wherever no layer's v g rounds differently under OpenCV's gain and the oracle's; with OpenCV's own gains
    the oracle composite is OpenCV's everywhere."""
    for name, layers, origins, size in _all_cases():
        want, g_cv = _opencv_chain(layers, origins, size, sharpness)
        assert np.array_equal(go.feather_blend(layers, origins, size, g_cv, sharpness), want), name
        g_or = go.gains(layers, origins, size)
        ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
        differ = np.zeros((size[1], size[0]), bool)
        for p, a, b in zip(ps, g_cv, g_or):
            differ |= (go.apply(p, a) != go.apply(p, b)).any(axis=-1)
        got = go.feather_blend(layers, origins, size, g_or, sharpness)
        assert np.array_equal(got[~differ], want[~differ]), name


def test_gain_argument_errors_before_any_launch():
    from cvx_proj_b200.utils import blend_layers, exposure_gains, feather_blend
    img = np.zeros((4, 5, 3), np.uint8)
    with pytest.raises(ValueError, match="257"):
        exposure_gains([img] * 257, [(0, 0)] * 257, (5, 4))
    with pytest.raises(ValueError, match="layers"):
        exposure_gains([], [], (5, 4))
    with pytest.raises(ValueError, match="origin"):
        exposure_gains([img, img], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="uint8"):
        exposure_gains([img.astype(np.float32)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="positive"):
        exposure_gains([img], [(0, 0)], (5, 0))
    for fn in (blend_layers, feather_blend):
        for bad in ([1.0], [1.0, float("nan")], [1.0, float("inf")], [[1.0, 1.0]], "ab", [1.0, 1.0, 1.0]):
            with pytest.raises(ValueError, match="gains"):
                fn([img, img], [(0, 0), (1, 1)], (5, 4), gains=bad)


def test_stitch_panorama_exposure_errors_before_any_keypoint_work():
    from cvx_proj_b200.driver import stitch_panorama
    img = np.zeros((4, 5, 3), np.uint8)
    for bad in ("gains", "", None, "GAIN"):
        with pytest.raises(ValueError, match="exposure"):
            stitch_panorama(img, [img], None, [None], exposure=bad)


def test_gain_stats_bytes_host_checks():
    lib = rt.load_library()
    nb = ctypes.c_size_t()
    assert lib.apap_gain_stats_bytes(3, ctypes.byref(nb)) == 0 and nb.value == 4 * 9 * 8
    assert lib.apap_gain_stats_bytes(256, ctypes.byref(nb)) == 0 and nb.value == 4 * 256 * 256 * 8
    assert lib.apap_gain_stats_bytes(0, ctypes.byref(nb)) == -1
    assert lib.apap_gain_stats_bytes(257, ctypes.byref(nb)) == -1


# ----------------------------------------------------------------------------------------------- GPU: kernels
def _gpu_stats(layers, origins, size):
    """apap_gain_stats' result as Python ints, from numpy or tensor layers."""
    import torch
    from cvx_proj_b200.utils import _layer_descs, gain_stats_ints
    on_device = not isinstance(layers[0], np.ndarray)
    dev = layers[0].device if on_device else torch.device("cuda", torch.cuda.current_device())
    devs, desc = _layer_descs(torch, dev, layers, origins, on_device)
    lib = rt.load_library()
    nb = ctypes.c_size_t()
    rt.check(lib.apap_gain_stats_bytes(len(devs), ctypes.byref(nb)), "bytes")
    stats = torch.full((nb.value // 8,), -1, dtype=torch.int64, device=dev)    # the call must clear it
    rt.check(lib.apap_gain_stats(desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), len(devs), size[1], size[0],
                                 stats.data_ptr(), nb.value, rt.stream_ptr(torch, dev)), "apap_gain_stats")
    return gain_stats_ints(stats.cpu().numpy(), len(devs))


def _assert_stats(got, want, name=""):
    count, sums = got
    wc, ws = want
    n = len(wc)
    for i in range(n):
        for j in range(n):
            assert count[i][j] == (wc[i][j] if i <= j else 0), (name, i, j, count[i][j], wc[i][j])
            assert sums[i][j] == (ws[i][j] if i != j else 0), (name, i, j)


@gpu
def test_gain_stats_equal_oracle_integers():
    for name, layers, origins, size in _all_cases():
        _assert_stats(_gpu_stats(layers, origins, size), go.stats(layers, origins, size), name)


@gpu
def test_gain_stats_c2_size_beyond_2_64():
    r = np.random.default_rng(21)
    w, h = 4222, 2560
    big = r.integers(200, 256, (h, w, 3), dtype=np.uint8)
    big2 = r.integers(1, 256, (h - 100, w - 50, 3), dtype=np.uint8)
    small = _random_image(r, 300, 500)
    layers, origins = [big, big2, small], [(0, 0), (30, 60), (3000, 1500)]
    want = go.stats(layers, origins, (w, h))
    assert want[1][0][1] > 1 << 64 and want[1][1][0] > 1 << 64
    got = _gpu_stats(layers, origins, (w, h))
    _assert_stats(got, want, "c2")
    assert _gpu_stats(layers, origins, (w, h)) == got                  # two calls, the same bits


@gpu
@pytest.mark.parametrize("n", [2, 33, 129, 256])
def test_gain_stats_many_layers_on_one_region(n):
    layers, origins = _random_case(40 + n, (70, 21), n, (60, 20))
    want = go.stats(layers, origins, (70, 21))
    _assert_stats(_gpu_stats(layers, origins, (70, 21)), want, n)


@gpu
def test_gain_stats_tensor_views_and_numpy():
    """Crops of a larger tensor at odd byte offsets, read in place; numpy and tensor inputs give the same integers."""
    import torch
    from cvx_proj_b200.utils import exposure_gains
    r = np.random.default_rng(11)
    big = _random_image(r, 300, 701, black=0.05)
    big_t = torch.from_numpy(big).cuda()
    crops = [(0, 0, 300, 701), (3, 1, 120, 333), (17, 5, 18, 6), (100, 257, 101, 258), (5, 7, 200, 8), (9, 11, 10, 600)]
    layers_t = [big_t[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    layers_np = [big[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    assert any(t.data_ptr() % 4 for t in layers_t) and any(t.stride(0) != 3 * t.shape[1] for t in layers_t)
    origins = [(-5, 3), (100, -20), (650, 280), (0, 0), (333, 100), (150, 200)]
    canvas = (701, 310)
    want = go.stats(layers_np, origins, canvas)
    _assert_stats(_gpu_stats(layers_t, origins, canvas), want, "tensor")
    _assert_stats(_gpu_stats(layers_np, origins, canvas), want, "numpy")
    g = go.gains_from_stats(*want)
    assert np.array_equal(exposure_gains(layers_t, origins, canvas), g)
    assert np.array_equal(exposure_gains(layers_np, origins, canvas), g)


@gpu
def test_exposure_gains_equal_oracle():
    from cvx_proj_b200.utils import exposure_gains
    for name, layers, origins, size in _all_cases():
        got = exposure_gains(layers, origins, size)
        assert got.dtype == np.float64 and got.shape == (len(layers),)
        assert np.array_equal(got, go.gains(layers, origins, size)), name


@gpu
def test_blends_with_gains_equal_oracle():
    from cvx_proj_b200.utils import blend_layers, exposure_gains, feather_blend
    r = np.random.default_rng(12)
    for name, layers, origins, size in _all_cases():
        n = len(layers)
        ones = np.ones(n)
        assert np.array_equal(blend_layers(layers, origins, size, gains=ones), blend_layers(layers, origins, size)), name
        assert np.array_equal(feather_blend(layers, origins, size, gains=ones), feather_blend(layers, origins, size)), name
        for gains in (exposure_gains(layers, origins, size), np.full(n, 3.0), np.full(n, 0.3), r.uniform(0.3, 2.5, n)):
            assert np.array_equal(blend_layers(layers, origins, size, gains=gains),
                                  go.blend_layers(layers, origins, size, gains)), (name, gains)
            assert np.array_equal(feather_blend(layers, origins, size, 0.05, gains=gains),
                                  go.feather_blend(layers, origins, size, gains, 0.05)), (name, gains)


@gpu
def test_blends_with_gains_many_layers():
    from cvx_proj_b200.utils import blend_layers, feather_blend
    r = np.random.default_rng(13)
    layers, origins = _random_case(7, (257, 131), 256, (200, 120))
    g = r.uniform(0.3, 3.0, 256)
    assert np.array_equal(blend_layers(layers, origins, (257, 131), gains=g), go.blend_layers(layers, origins, (257, 131), g))
    assert np.array_equal(feather_blend(layers[:128], origins[:128], (257, 131), gains=g[:128]),
                          go.feather_blend(layers[:128], origins[:128], (257, 131), g[:128]))


@gpu
def test_gain_c_entry_checks():
    import torch
    lib = rt.load_library()
    t = torch.zeros((4, 5, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((4, 5, 3), dtype=torch.uint8, device="cuda")
    stats = torch.empty(64, dtype=torch.int64, device="cuda")
    lut = torch.zeros((1, 256), dtype=torch.uint8, device="cuda")
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    st = rt.stream_ptr(torch, out.device)
    P = ctypes.POINTER(ctypes.c_longlong)

    def desc(d):
        return np.asarray(d, dtype=np.int64).reshape(-1, 6)

    good = [t.data_ptr(), 4, 5, 15, 0, 0]

    def stats_call(d, n, nbytes=32, ptr=None):
        a = desc(d)
        return lib.apap_gain_stats(a.ctypes.data_as(P), n, 4, 5, stats.data_ptr() if ptr is None else ptr, nbytes, st)
    assert stats_call(good, 1) == 0
    torch.cuda.synchronize()
    assert stats.cpu().numpy()[0] == 0 and (stats.cpu().numpy()[1:4] == 0).all()
    for d, n, kw in ((good, 0, {}), ([good] * 257, 257, {"nbytes": 1 << 22}), (good, 1, {"nbytes": 31}),
                     ([0, 4, 5, 15, 0, 0], 1, {}), ([t.data_ptr(), 4, 5, 14, 0, 0], 1, {}), (good, 1, {"ptr": 0})):
        assert stats_call(d, n, **kw) == -1, (n, kw)
    assert stats_call(good, 1, ptr=stats.data_ptr() + 4) == -2
    a = desc(good)
    assert lib.apap_blend_layers_gain(a.ctypes.data_as(P), 1, 4, 5, lut.data_ptr(), out.data_ptr(), 60, st) == 0
    assert lib.apap_blend_layers_gain(a.ctypes.data_as(P), 1, 4, 5, None, out.data_ptr(), 60, st) == -1
    assert lib.apap_blend_layers_gain(a.ctypes.data_as(P), 1, 4, 5, lut.data_ptr(), out.data_ptr(), 59, st) == -1
    assert lib.apap_feather_blend_gain(a.ctypes.data_as(P), 1, 4, 5, 0.02, lut.data_ptr(), ws.data_ptr(), 256,
                                       out.data_ptr(), 60, st) == 0
    assert lib.apap_feather_blend_gain(a.ctypes.data_as(P), 1, 4, 5, 0.02, None, ws.data_ptr(), 256,
                                       out.data_ptr(), 60, st) == -1
    assert lib.apap_feather_blend_gain(a.ctypes.data_as(P), 1, 4, 5, 0.0, lut.data_ptr(), ws.data_ptr(), 256,
                                       out.data_ptr(), 60, st) == -1
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------- GPU: driver
def _layers_of(res, warps, blend, monkeypatch):
    from tests.test_feather import _feather_layers
    return _feather_layers(res, warps, blend, monkeypatch)


def _check_exposure(monkeypatch, centre, others, raw_c, raw_os, ransac, blend, live=False, **kw):
    from cvx_proj_b200.driver import stitch_panorama
    from tests.test_case import _assert_results_equal
    res = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend=blend, exposure="gain", **kw)
    plain = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend=blend, **kw)
    none = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend=blend, exposure="none", **kw)
    assert np.array_equal(none.panorama, plain.panorama)
    assert res.final_size == plain.final_size and np.array_equal(res.origins, plain.origins)
    for i, (g, w) in enumerate(zip(res.pairs, plain.pairs)):
        _assert_results_equal(g, w, i)
    warps = kw.get("warp_imgs") or others
    bimg = kw.get("blend_img") if kw.get("blend_img") is not None else centre
    layers, origins, size = _layers_of(res, warps, bimg, monkeypatch)
    g = go.gains(layers, origins, size)
    assert not np.allclose(g, 1.0)
    want = go.blend_layers(layers, origins, size, g) if blend == "mean" else go.feather_blend(layers, origins, size, g)
    assert np.array_equal(res.panorama, want)
    if live:
        cv_pano, g_cv = _opencv_chain(layers, origins, size)
        assert np.allclose(g, g_cv, rtol=1e-12, atol=0)
        ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
        differ = np.zeros((size[1], size[0]), bool)
        for p, a, b in zip(ps, g_cv, g):
            differ |= (go.apply(p, a) != go.apply(p, b)).any(axis=-1)
        assert np.array_equal(res.panorama[~differ], cv_pano[~differ])


def _dimmed(imgs):
    return [np.clip(np.rint(img * (0.7 + 0.2 * j)), 0, 255).astype(np.uint8) for j, img in enumerate(imgs)]


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("blend", ["mean", "feather"])
def test_stitch_panorama_exposure_gain_c1(ransac, blend, monkeypatch):
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    _check_exposure(monkeypatch, centre, others, raw_c, raw_os, ransac, blend, live=blend == "feather",
                    warp_imgs=_dimmed(others))


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("blend", ["mean", "feather"])
def test_stitch_panorama_exposure_gain_c4(ransac, blend, monkeypatch):
    from tests.test_case import _scene
    centre, others, raw_c, raw_os = _scene("c4", 6)
    _check_exposure(monkeypatch, centre, others, raw_c, raw_os, ransac, blend, warp_imgs=_dimmed(others))


@gpu
def test_stitch_panorama_exposure_no_other_image():
    from cvx_proj_b200.driver import stitch_panorama
    centre, _, raw_c, _ = _scene_2d("c1", 1)
    for blend in ("mean", "feather"):
        a = stitch_panorama(centre, [], raw_c, [], blend=blend, exposure="gain")
        b = stitch_panorama(centre, [], raw_c, [], blend=blend)
        assert a.pairs == [] and a.final_size == b.final_size and np.array_equal(a.panorama, b.panorama)
