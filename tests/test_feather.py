"""The feather blend of a panorama: ``oracle.feather_oracle`` pinned against the live ``cv.detail.FeatherBlender`` and
``cv.distanceTransform``, the kernels (``utils.feather_blend``) against the oracle, and
``driver.stitch_panorama(blend="feather")`` against the oracle composite."""
import ctypes

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import _runtime as rt
from cvx_proj_b200 import synth
from oracle import feather_oracle as fo
from tests.test_panorama import _random_case, _random_image, _scene_2d

gpu = pytest.mark.gpu
FLT_MIN = float(np.finfo(np.float32).tiny)
SHARPNESS = (0.02, 1.0, 5.0, 1e-3, 1e-6, FLT_MIN)    # FLT_MIN: the smallest sharpness accepted


def _opencv(layers, origins, size, sharpness=0.02):
    """cv.detail.FeatherBlender fed as utils.feather_blend's contract says: every layer pasted into the canvas."""
    blender = cv.detail.FeatherBlender(sharpness)
    blender.prepare((0, 0, size[0], size[1]))
    for img, origin in zip(layers, origins):
        p = fo.paste(img, origin, size)
        blender.feed(p.astype(np.int16), np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8), (0, 0))
    res, _ = blender.blend(None, None)
    return res


def _cases():
    """(name, layers, origins, size): the CPU cases, each also run on the GPU."""
    r = np.random.default_rng(5)
    out = []
    layers, origins = _random_case(0, (61, 47), 9, (40, 30))      # ragged, 1 x 1 and 1 px wide, negative, clipped
    out.append(("ragged", layers, origins, (61, 47)))
    layers, origins = _random_case(1, (1500, 40), 12, (1200, 35))  # rows of several 1024-pixel tiles
    out.append(("wide", layers, origins, (1500, 40)))
    holes = _random_image(r, 50, 70, black=0.02)
    holes[20:23, 30:40] = 0
    out.append(("holes", [holes, _random_image(r, 30, 30)], [(-5, -3), (40, 25)], (80, 60)))
    full = r.integers(1, 256, (33, 45, 3), dtype=np.uint8)          # no empty pixel in the whole canvas
    out.append(("full", [full, _random_image(r, 10, 12)], [(0, 0), (5, 7)], (45, 33)))
    out.append(("one", [_random_image(r, 33, 45)], [(0, 0)], (45, 33)))
    out.append(("tall", [_random_image(r, 300, 3), _random_image(r, 280, 1)], [(0, 0), (1, 5)], (4, 300)))
    return out


# ----------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("density", [0.001, 0.02, 0.3, 0.9])
def test_oracle_distance_is_opencv_l1(density):
    r = np.random.default_rng(int(density * 1000))
    for h, w in ((37, 53), (1, 40), (40, 1), (1, 1), (120, 90)):
        mask = np.where(r.random((h, w)) < density, 0, 255).astype(np.uint8)
        assert np.array_equal(fo.l1_distance(mask), cv.distanceTransform(mask, cv.DIST_L1, 3)), (h, w)


def test_oracle_distance_single_zero_and_none():
    mask = np.full((31, 47), 255, np.uint8)
    want = cv.distanceTransform(mask, cv.DIST_L1, 3)
    assert (want == np.finfo(np.float32).max).all()
    assert np.array_equal(fo.l1_distance(mask), want)
    mask[30, 2] = 0
    assert np.array_equal(fo.l1_distance(mask), cv.distanceTransform(mask, cv.DIST_L1, 3))
    one = np.full((1, 1), 255, np.uint8)
    assert np.array_equal(fo.l1_distance(one), cv.distanceTransform(one, cv.DIST_L1, 3))


@pytest.mark.parametrize("sharpness", SHARPNESS)
def test_oracle_is_opencv_feather_blender(sharpness):
    for name, layers, origins, size in _cases():
        want = _opencv(layers, origins, size, sharpness)
        assert want.min() >= 0 and want.max() <= 255, name        # fits uint8
        got = fo.feather_blend(layers, origins, size, sharpness)
        assert np.array_equal(got, want.astype(np.uint8)), (name, sharpness)


def test_oracle_one_layer_loses_one():
    img = _random_image(np.random.default_rng(2), 20, 30)
    got = fo.feather_blend([img], [(0, 0)], (30, 20), 1.0)
    mask = img.max(axis=-1) > 0
    d = cv.distanceTransform(mask.astype(np.uint8) * 255, cv.DIST_L1, 3)
    sure = d >= 1                                                   # weight 1 at sharpness 1
    assert np.array_equal(got[sure], np.maximum(img[sure].astype(int) - 1, 0))
    assert np.array_equal(got, _opencv([img], [(0, 0)], (30, 20), 1.0).astype(np.uint8))


def test_oracle_128_saturated_layers():
    full = np.full((5, 6, 3), 255, np.uint8)
    want = _opencv([full] * 128, [(0, 0)] * 128, (6, 5))
    assert (want == 254).all()
    assert (fo.feather_blend([full] * 128, [(0, 0)] * 128, (6, 5)) == 254).all()
    assert (_opencv([full] * 129, [(0, 0)] * 129, (6, 5)) < 0).all()     # int16 wraps: why 128 is the limit


@pytest.mark.parametrize("seed", range(4))
def test_oracle_output_range(seed):
    layers, origins = _random_case(seed + 20, (90, 70), 24, (60, 50))
    for s in SHARPNESS:
        raw = _opencv(layers, origins, (90, 70), s)
        assert raw.min() >= 0 and raw.max() <= 255


@pytest.mark.parametrize("sharpness", SHARPNESS + (0.1, 1.5e-5, 3e-5))
def test_distance_cap_rule(sharpness):
    """fl(D s) >= 1 for every D >= cap up to the largest distance of the canvas, < 1 below, unless the cap is the
    canvas limit W + H - 1 (every finite distance lies below it)."""
    lib = rt.load_library()
    s = np.float32(sharpness)
    for w, h in ((4222, 2560), (45, 33), (40000, 30000)):
        cap = ctypes.c_int()
        rc = lib.apap_feather_distance_cap(float(s), h, w, ctypes.byref(cap))
        if rc != 0:
            assert w + h - 1 > 65535 and np.float32(65535) * s < 1
            continue
        c = cap.value
        assert 1 <= c <= 65535
        d = np.arange(0, w + h, dtype=np.float32)
        ok = d * s >= np.float32(1)
        if c < w + h - 1:
            assert ok[c:].all() and not ok[:c].any()
        else:
            assert c == w + h - 1 and not ok[:c].any()


def test_feather_blend_argument_errors_before_any_launch():
    from cvx_proj_b200.utils import feather_blend
    img = np.zeros((4, 5, 3), np.uint8)
    with pytest.raises(ValueError, match="129"):
        feather_blend([img] * 129, [(0, 0)] * 129, (5, 4))
    with pytest.raises(ValueError, match="layers"):
        feather_blend([], [], (5, 4))
    with pytest.raises(ValueError, match="origin"):
        feather_blend([img, img], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match=r"\[h, w, 3\]"):
        feather_blend([np.zeros((4, 5), np.uint8)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="uint8"):
        feather_blend([img.astype(np.float32)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="positive"):
        feather_blend([img], [(0, 0)], (0, 4))
    for bad in (0.0, -0.02, float("nan"), float("inf"), 1e-50, 1e300, 1e-40, 2e-39, FLT_MIN / 2):
        with pytest.raises(ValueError, match="sharpness"):
            feather_blend([img], [(0, 0)], (5, 4), bad)
    with pytest.raises(ValueError, match="16 bits"):
        feather_blend([img], [(0, 0)], (40000, 30000), 1e-6)
    with pytest.raises(ValueError, match=r"2\^30"):                # the library's own message, not the 16-bit one
        feather_blend([img], [(0, 0)], ((1 << 30) + 1, 4))


def test_subnormal_sharpness_is_refused():
    """Below FLT_MIN, OpenCV weights a layer with no empty pixel by min(fl(FLT_MAX s), 1) < 1, where the kernels would
    give it 1; the library refuses such s, and accepts FLT_MIN, where that weight is 1."""
    full = np.random.default_rng(4).integers(1, 256, (20, 30, 3), dtype=np.uint8)
    for s in (1e-40, 2e-39):
        assert np.float32(np.finfo(np.float32).max) * np.float32(s) < 1
        assert not np.array_equal(_opencv([full], [(0, 0)], (30, 20), s).astype(np.uint8),
                                  np.maximum(full.astype(int) - 1, 0))
    lib = rt.load_library()
    cap = ctypes.c_int()
    assert lib.apap_feather_distance_cap(1e-40, 20, 30, ctypes.byref(cap)) == -1
    assert lib.apap_feather_distance_cap(FLT_MIN / 2, 20, 30, ctypes.byref(cap)) == -1
    assert lib.apap_feather_distance_cap(FLT_MIN, 20, 30, ctypes.byref(cap)) == 0 and cap.value == 49
    assert np.array_equal(_opencv([full], [(0, 0)], (30, 20), FLT_MIN).astype(np.uint8),
                          np.maximum(full.astype(int) - 1, 0))


def test_stitch_panorama_blend_errors_before_any_keypoint_work():
    from cvx_proj_b200.driver import stitch_panorama
    img = np.zeros((4, 5, 3), np.uint8)
    with pytest.raises(ValueError, match="median"):
        stitch_panorama(img, [img], None, [None], blend="median")
    with pytest.raises(ValueError, match="at most 127"):
        stitch_panorama(img, [img] * 128, None, [None] * 128, blend="feather")
    for bad in (0.0, float("nan"), 1e-40):
        with pytest.raises(ValueError, match="sharpness"):
            stitch_panorama(img, [img], None, [None], blend="feather", sharpness=bad)


# ----------------------------------------------------------------------------------------------- GPU: kernels
@gpu
@pytest.mark.parametrize("sharpness", SHARPNESS)
def test_feather_blend_equals_oracle(sharpness):
    from cvx_proj_b200.utils import feather_blend
    for name, layers, origins, size in _cases():
        got = feather_blend(layers, origins, size, sharpness)
        assert isinstance(got, np.ndarray) and got.shape == (size[1], size[0], 3) and got.dtype == np.uint8
        assert np.array_equal(got, fo.feather_blend(layers, origins, size, sharpness)), (name, sharpness)


@gpu
def test_feather_blend_equals_opencv_and_order():
    """The same layers in the given and the reversed order, each against the oracle and OpenCV in its order."""
    from cvx_proj_b200.utils import feather_blend
    layers, origins = _random_case(3, (700, 90), 30, (500, 80))
    for order in (slice(None), slice(None, None, -1)):
        ls, os_ = layers[order], origins[order]
        got = feather_blend(ls, os_, (700, 90), 0.05)
        assert np.array_equal(got, fo.feather_blend(ls, os_, (700, 90), 0.05))
        assert np.array_equal(got, _opencv(ls, os_, (700, 90), 0.05).astype(np.uint8))


@gpu
def test_feather_blend_128_layers():
    from cvx_proj_b200.utils import feather_blend
    full = np.full((9, 1030, 3), 255, np.uint8)
    assert (feather_blend([full] * 128, [(0, 0)] * 128, (1030, 9)) == 254).all()
    layers, origins = _random_case(6, (257, 131), 128, (200, 120))
    assert np.array_equal(feather_blend(layers, origins, (257, 131)), fo.feather_blend(layers, origins, (257, 131)))


@gpu
def test_feather_blend_long_uncapped_distances():
    """A c2-size canvas with one far-off empty pixel at sharpness 1e-4: distances in the thousands, none capped."""
    from cvx_proj_b200.utils import feather_blend
    r = np.random.default_rng(8)
    w, h = 4222, 2560
    big = r.integers(1, 256, (h, w, 3), dtype=np.uint8)
    big[h - 3, 7] = 0
    small = _random_image(r, 300, 500)
    layers, origins = [big, small], [(0, 0), (3000, 1500)]
    got = feather_blend(layers, origins, (w, h), 1e-4)
    assert np.array_equal(got, fo.feather_blend(layers, origins, (w, h), 1e-4))


@gpu
def test_feather_blend_tensor_views():
    """Crops of a larger tensor at odd byte offsets, read in place; numpy and tensor inputs give the same bits."""
    import torch
    from cvx_proj_b200.utils import feather_blend
    r = np.random.default_rng(11)
    big = _random_image(r, 300, 701, black=0.05)
    big_t = torch.from_numpy(big).cuda()
    crops = [(0, 0, 300, 701), (3, 1, 120, 333), (17, 5, 18, 6), (100, 257, 101, 258), (5, 7, 200, 8), (9, 11, 10, 600)]
    layers_t = [big_t[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    layers_np = [big[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    assert any(t.data_ptr() % 4 for t in layers_t) and any(t.stride(0) != 3 * t.shape[1] for t in layers_t)
    origins = [(-5, 3), (100, -20), (650, 280), (0, 0), (333, 100), (150, 200)]
    canvas = (701, 310)
    want = fo.feather_blend(layers_np, origins, canvas)
    got = feather_blend(layers_t, origins, canvas)
    assert got.is_cuda and got.device == big_t.device
    assert np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(feather_blend(layers_np, origins, canvas), want)


@gpu
def test_feather_blend_c_entry_checks():
    import torch
    lib = rt.load_library()
    t = torch.zeros((4, 5, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((4, 5, 3), dtype=torch.uint8, device="cuda")
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    st = rt.stream_ptr(torch, out.device)

    def call(desc, n, s=0.02, nbytes=60, ws_ptr=None, ws_bytes=256):
        arr = np.asarray(desc, dtype=np.int64).reshape(-1, 6)
        return lib.apap_feather_blend(arr.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), n, 4, 5, s,
                                      ws.data_ptr() if ws_ptr is None else ws_ptr, ws_bytes, out.data_ptr(), nbytes, st)
    good = [t.data_ptr(), 4, 5, 15, 0, 0]
    assert call(good, 1) == 0
    torch.cuda.synchronize()
    for desc, n, kw in ((good, 0, {}), ([good] * 129, 129, {}), (good, 1, {"nbytes": 59}), (good, 1, {"s": 0.0}),
                        (good, 1, {"s": float("nan")}), (good, 1, {"ws_bytes": 39}), ([0, 4, 5, 15, 0, 0], 1, {}),
                        ([t.data_ptr(), 4, 5, 14, 0, 0], 1, {})):
        assert call(desc, n, **kw) == -1, (n, kw)
    assert call(good, 1, ws_ptr=ws.data_ptr() + 2) == -2


# ----------------------------------------------------------------------------------------------- GPU: driver
def _feather_layers(res, warps, blend, monkeypatch):
    """The layers, origins and canvas of tests.test_panorama._composite: its blend is taken over to return them."""
    import tests.test_panorama as tp
    with monkeypatch.context() as m:
        m.setattr(tp.po, "blend_layers", lambda layers, origins, size: (layers, origins, size))
        return tp._composite(res, warps, blend)


def _check_feather(monkeypatch, centre, others, raw_c, raw_os, ransac, live=False, **kw):
    from cvx_proj_b200.driver import stitch_panorama
    from tests.test_case import _assert_results_equal
    res = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend="feather", **kw)
    mean = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, **kw)
    assert res.final_size == mean.final_size and np.array_equal(res.origins, mean.origins)
    assert len(res.pairs) == len(mean.pairs)
    for i, (g, w) in enumerate(zip(res.pairs, mean.pairs)):
        _assert_results_equal(g, w, i)
    warps = kw.get("warp_imgs") or others
    blend = kw.get("blend_img") if kw.get("blend_img") is not None else centre
    layers, origins, size = _feather_layers(res, warps, blend, monkeypatch)
    assert isinstance(res.panorama, np.ndarray) and res.panorama.shape == (size[1], size[0], 3)
    assert np.array_equal(res.panorama, fo.feather_blend(layers, origins, size))
    if live:
        assert np.array_equal(res.panorama, _opencv(layers, origins, size).astype(np.uint8))
    return res


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
def test_stitch_panorama_feather_c1(ransac, monkeypatch):
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    _check_feather(monkeypatch, centre, others, raw_c, raw_os, ransac, live=True)


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
def test_stitch_panorama_feather_c4(ransac, monkeypatch):
    from tests.test_case import _scene
    centre, others, raw_c, raw_os = _scene("c4", 6)
    _check_feather(monkeypatch, centre, others, raw_c, raw_os, ransac)


@gpu
def test_stitch_panorama_feather_given_images_and_no_other(monkeypatch):
    from cvx_proj_b200.driver import stitch_panorama
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    warps = [(255 - o) for o in others]
    for j, wimg in enumerate(warps):
        wimg[20 + 10 * j:90 + 10 * j, 30:200] = 0
    blend = synth.make_image(centre.shape[1], centre.shape[0], seed=9)
    blend[40:140, 60:400] = 0
    _check_feather(monkeypatch, centre, others, raw_c, raw_os, "opencv", warp_imgs=warps, blend_img=blend, mesh_size=40)
    res = stitch_panorama(centre, [], raw_c, [], blend="feather")
    assert res.pairs == [] and res.final_size == (centre.shape[1], centre.shape[0], 0, 0)
    size = (centre.shape[1], centre.shape[0])
    assert np.array_equal(res.panorama, fo.feather_blend([centre], [(0, 0)], size))
    assert np.array_equal(res.panorama, _opencv([centre], [(0, 0)], size).astype(np.uint8))
