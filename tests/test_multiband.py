"""Multi-band blend of a panorama: ``oracle.multiband_oracle`` pinned against the live
``cv.detail_MultiBandBlender(0, bands, cv.CV_16S)`` (its pyramids against ``cv.pyrDown`` / ``cv.pyrUp``, the blend, and
the compensate-then-blend chain), the kernels (``k_mb_down``, ``k_mb_band``) against the oracle, and
``driver.stitch_panorama(blend="multiband")`` against the oracle composite."""
import ctypes
import math

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import _runtime as rt
from oracle import feather_oracle as fo
from oracle import gain_oracle as go
from oracle import multiband_oracle as mo
from tests.test_feather import _cases
from tests.test_panorama import _random_case, _random_image, _scene_2d

gpu = pytest.mark.gpu

BANDS = (0, 1, 2, 3, 4, 5, 6, 7, 8, 12, 40)          # 0 .. 8 and values above every case's cap


def _masks(ps):
    return [np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8) for p in ps]


def _opencv(layers, origins, size, bands, gains=None):
    """The live CV_16S blender fed as multiband_blend's contract says.  ``gains=True``: OpenCV's pipeline, a
    ``GainCompensator`` fed the same layers and each layer through its ``apply`` with its raw mask kept; returns
    ``(panorama, OpenCV's gains)`` then."""
    ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
    ms = _masks(ps)
    comp = None
    if gains is not None:
        comp = cv.detail.GainCompensator()
        comp.feed([(0, 0)] * len(ps), [cv.UMat(p) for p in ps], [cv.UMat(m) for m in ms])
    b = cv.detail_MultiBandBlender(0, bands, cv.CV_16S)
    b.prepare((0, 0, size[0], size[1]))
    for k, (p, m) in enumerate(zip(ps, ms)):
        if comp is not None:
            p = comp.apply(k, (0, 0), p.copy(), m)
        b.feed(p.astype(np.int16), m, (0, 0))
    res, _ = b.blend(None, None)
    assert res.dtype == np.int16
    out = np.clip(res, 0, 255).astype(np.uint8)                 # convertTo(CV_8U) saturates
    if comp is None:
        return out
    return out, np.asarray(comp.getMatGains(), dtype=np.float64).reshape(-1)


def _edge_case():
    """Layers touching each canvas edge and sticking out of it, so that the boxes meet the reflect pad."""
    r = np.random.default_rng(31)
    w, h = 203, 117                                              # pads of 5 and 11 at 4 bands
    layers = [_random_image(r, 40, 60), _random_image(r, 50, 30), _random_image(r, 30, 70), _random_image(r, 60, 45),
              _random_image(r, 117, 20), _random_image(r, 20, 203), _random_image(r, 25, 25)]
    origins = [(-10, -7), (w - 30, 20), (60, h - 30), (w - 20, h - 40), (w - 20, 0), (0, h - 20), (90, 40)]
    return "edges", layers, origins, (w, h)


def _extra_cases():
    r = np.random.default_rng(17)
    out = []
    a, b = _random_image(r, 20, 30, black=0.0), _random_image(r, 20, 30, black=0.0)
    out.append(("disjoint", [a, b], [(0, 0), (40, 25)], (80, 50)))
    out.append(("all-zero", [_random_image(r, 30, 30), np.zeros((20, 20, 3), np.uint8), _random_image(r, 25, 25)],
                [(0, 0), (5, 5), (10, 3)], (40, 35)))
    out.append(("outside", [_random_image(r, 10, 10), _random_image(r, 30, 30)], [(100, 0), (0, 0)], (40, 35)))
    out.append(_edge_case())
    for w, h in ((1, 37), (37, 1), (300, 5), (1, 1)):          # pads wider than a dimension
        out.append((f"{w}x{h}", [_random_image(r, h, w, black=0.1), _random_image(r, max(1, h - 2), max(1, w // 2))],
                    [(0, 0), (w // 3, h // 4)], (w, h)))
    return out


def _all_cases():
    return _cases() + _extra_cases()


def _full_stack(n):
    """``n`` layers with no empty pixel, all over one 24 x 16 region of a 30 x 20 canvas."""
    r = np.random.default_rng(n)
    return [r.integers(1, 256, (16, 24, 3), dtype=np.uint8) for _ in range(n)], [(3, 2)] * n, (30, 20)


# ----------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("op", ["down", "up"])
def test_oracle_pyramids_are_opencv(op):
    r = np.random.default_rng(3)
    for h in (1, 2, 3, 4, 5, 8, 11, 32, 33):
        for w in (1, 2, 3, 5, 6, 9, 16, 17, 64):
            if op == "down" and (h < 2 or w < 2):
                continue
            x = r.integers(-400, 400, (h, w, 3)).astype(np.int16)
            want = cv.pyrDown(x) if op == "down" else cv.pyrUp(x)
            got = mo.pyr_down(x) if op == "down" else mo.pyr_up(x)
            assert want.shape == got.shape and np.array_equal(want, got), (h, w)


def test_num_bands_is_opencv_cap():
    n = np.arange(1, (1 << 17) + 1)
    cap = np.array([int(math.ceil(math.log(float(v)) / math.log(2.0))) for v in n])
    assert np.array_equal(cap, [(int(v) - 1).bit_length() for v in n])
    assert mo.num_bands(40, 900, 600) == 10 and mo.num_bands(3, 900, 600) == 3 and mo.num_bands(9, 1, 1) == 0


def test_case_names():
    assert [c[0] for c in _all_cases()] == ["ragged", "wide", "holes", "full", "one", "tall", "disjoint", "all-zero",
                                            "outside", "edges", "1x37", "37x1", "300x5", "1x1"]


@pytest.mark.parametrize("case", range(14))
def test_oracle_is_opencv(case):
    name, layers, origins, size = _all_cases()[case]
    for bands in BANDS:
        assert np.array_equal(mo.multiband_blend(layers, origins, size, bands), _opencv(layers, origins, size, bands)), \
            (name, bands)


def test_oracle_leaves_the_byte_range_before_the_clip():
    """The int16 result runs outside [0, 255] at sharp edges: the clip is part of the contract."""
    name, layers, origins, size = _edge_case()
    b = cv.detail_MultiBandBlender(0, 5, cv.CV_16S)
    b.prepare((0, 0, size[0], size[1]))
    for p, m in zip([fo.paste(i, o, size) for i, o in zip(layers, origins)],
                    _masks([fo.paste(i, o, size) for i, o in zip(layers, origins)])):
        b.feed(p.astype(np.int16), m, (0, 0))
    res, _ = b.blend(None, None)
    assert res.min() < 0 and res.max() > 255


def test_oracle_127_layers_and_why_128_are_refused():
    layers, origins, size = _full_stack(127)
    assert np.array_equal(mo.multiband_blend(layers, origins, size, 5), _opencv(layers, origins, size, 5))
    layers, origins, size = _full_stack(128)
    live = _opencv(layers, origins, size, 5)
    # OpenCV's int16 weight sum wraps to -32768 where all 128 cover: those pixels come out 0
    assert (live[2:18, 3:27] == 0).all(axis=-1).mean() > 0.3
    assert not np.array_equal(mo.multiband_blend(layers, origins, size, 5), live)


@pytest.mark.parametrize("case", ["ragged", "holes", "edges", "full"])
def test_oracle_chain_is_opencv(case):
    """GainCompensator.apply then the blender, against the oracle fed OpenCV's own gains."""
    name, layers, origins, size = next(c for c in _all_cases() if c[0] == case)
    layers = [np.clip(np.rint(img * (0.6 + 0.25 * k)), 0, 255).astype(np.uint8) for k, img in enumerate(layers)]
    for bands in (0, 3, 5):
        live, g_cv = _opencv(layers, origins, size, bands, gains=True)
        assert not np.allclose(g_cv, 1.0)
        assert np.array_equal(mo.multiband_blend(layers, origins, size, bands, gains=g_cv), live), (name, bands)


def test_multiband_argument_errors_before_any_launch():
    from cvx_proj_b200.utils import multiband_blend
    img = np.zeros((4, 5, 3), np.uint8)
    for bad in (1.5, True, False, -1, "3", None, np.float32(2)):
        with pytest.raises(ValueError, match="bands"):
            multiband_blend([img], [(0, 0)], (5, 4), bands=bad)
    with pytest.raises(ValueError, match="128"):
        multiband_blend([img] * 128, [(0, 0)] * 128, (5, 4))
    with pytest.raises(ValueError, match="524280"):
        multiband_blend([img], [(0, 0)], (5, 524281))
    with pytest.raises(ValueError, match="layers"):
        multiband_blend([], [], (5, 4))
    for bad in ([1.0], [1.0, float("nan")], "ab"):
        with pytest.raises(ValueError, match="gains"):
            multiband_blend([img, img], [(0, 0), (1, 1)], (5, 4), gains=bad)


def test_stitch_panorama_multiband_errors_before_any_keypoint_work():
    from cvx_proj_b200.driver import stitch_panorama
    img = np.zeros((4, 5, 3), np.uint8)
    for bad in ("multi-band", "MULTIBAND", None):
        with pytest.raises(ValueError, match="blend"):
            stitch_panorama(img, [img], None, [None], blend=bad)
    for bad in (-1, 2.0, True):
        with pytest.raises(ValueError, match="bands"):
            stitch_panorama(img, [img], None, [None], blend="multiband", bands=bad)
    with pytest.raises(ValueError, match="126"):
        stitch_panorama(img, [img] * 127, None, [None] * 127, blend="multiband")


def test_multiband_workspace_bytes_host_checks():
    lib = rt.load_library()
    P = ctypes.POINTER(ctypes.c_longlong)
    nb = ctypes.c_size_t()
    d = np.array([[1 << 20, 4, 5, 15, 0, 0]], dtype=np.int64)

    def call(desc, n, h=4, w=5, bands=5):
        return lib.apap_multiband_workspace_bytes(desc.ctypes.data_as(P), n, h, w, bands, ctypes.byref(nb))
    assert call(d, 1, bands=0) == 0 and nb.value == 0           # no level above 0
    # 5 x 4 at 5 bands: nb = 3, Wp = Hp = 8; both pads pick up the layer, so its boxes are 4 x 4, 2 x 2 and 1 x 1, as
    # are R_1 .. R_3; 8 B a value, each buffer rounded up to 16 B
    assert call(d, 1) == 0 and nb.value == 2 * (128 + 32 + 16)
    assert call(d, 0) == -1 and call(np.repeat(d, 128, 0), 128) == -1
    assert call(d, 1, bands=-1) == -1 and call(d, 1, h=0) == -1
    assert call(np.array([[0, 4, 5, 15, 0, 0]], dtype=np.int64), 1) == -1
    assert call(d, 1, h=524281) == -3


# ----------------------------------------------------------------------------------------------- GPU: kernels
@gpu
@pytest.mark.parametrize("case", range(14))
def test_kernels_equal_oracle(case):
    from cvx_proj_b200.utils import multiband_blend
    name, layers, origins, size = _all_cases()[case]
    r = np.random.default_rng(case)
    for bands in BANDS:
        got = multiband_blend(layers, origins, size, bands)
        assert got.shape == (size[1], size[0], 3) and got.dtype == np.uint8
        assert np.array_equal(got, mo.multiband_blend(layers, origins, size, bands)), (name, bands)
    for gains in (np.ones(len(layers)), r.uniform(0.3, 2.5, len(layers))):
        for bands in (0, 3, 5):
            assert np.array_equal(multiband_blend(layers, origins, size, bands, gains=gains),
                                  mo.multiband_blend(layers, origins, size, bands, gains=gains)), (name, bands)


@gpu
@pytest.mark.parametrize("bands", [5, 13])
def test_kernels_c2_size(bands):
    from cvx_proj_b200.utils import multiband_blend
    r = np.random.default_rng(bands)
    w, h = 4222, 2560
    layers = [_random_image(r, 2400, 2600, black=0.01), _random_image(r, 2000, 2300, black=0.01),
              _random_image(r, 1700, 1900, black=0.01)]
    origins = [(0, 0), (1900, 560), (-100, 1000)]
    assert mo.num_bands(bands, w, h) == min(bands, 13)
    want = mo.multiband_blend(layers, origins, (w, h), bands)
    assert np.array_equal(multiband_blend(layers, origins, (w, h), bands), want)


@gpu
def test_kernels_127_layers():
    from cvx_proj_b200.utils import multiband_blend
    layers, origins, size = _full_stack(127)
    assert np.array_equal(multiband_blend(layers, origins, size, 5), mo.multiband_blend(layers, origins, size, 5))
    layers, origins = _random_case(9, (70, 21), 127, (60, 20))
    g = np.random.default_rng(9).uniform(0.3, 3.0, 127)
    assert np.array_equal(multiband_blend(layers, origins, (70, 21), 4, gains=g),
                          mo.multiband_blend(layers, origins, (70, 21), 4, gains=g))


@gpu
def test_kernels_tensor_views_and_numpy():
    """Crops of a larger tensor at odd byte offsets, read in place: the same bytes as numpy in."""
    import torch
    from cvx_proj_b200.utils import multiband_blend
    r = np.random.default_rng(11)
    big = _random_image(r, 300, 701, black=0.05)
    big_t = torch.from_numpy(big).cuda()
    crops = [(0, 0, 300, 701), (3, 1, 120, 333), (17, 5, 18, 6), (100, 257, 101, 258), (5, 7, 200, 8), (9, 11, 10, 600)]
    layers_t = [big_t[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    layers_np = [big[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    assert any(t.data_ptr() % 4 for t in layers_t) and any(t.stride(0) != 3 * t.shape[1] for t in layers_t)
    origins = [(-5, 3), (100, -20), (650, 280), (0, 0), (333, 100), (150, 200)]
    canvas = (701, 310)
    want = mo.multiband_blend(layers_np, origins, canvas, 5)
    got_t = multiband_blend(layers_t, origins, canvas, 5)
    assert isinstance(got_t, torch.Tensor) and got_t.device == big_t.device
    assert np.array_equal(got_t.cpu().numpy(), want)
    assert np.array_equal(multiband_blend(layers_np, origins, canvas, 5), want)


@gpu
def test_kernels_layer_order_does_not_matter():
    from cvx_proj_b200.utils import multiband_blend
    r = np.random.default_rng(5)
    layers, origins = _random_case(3, (300, 200), 17, (160, 120))
    g = r.uniform(0.4, 2.0, 17)
    perm = r.permutation(17)
    for bands in (2, 5):
        a = multiband_blend(layers, origins, (300, 200), bands)
        b = multiband_blend([layers[i] for i in perm], [origins[i] for i in perm], (300, 200), bands)
        assert np.array_equal(a, b)
        a = multiband_blend(layers, origins, (300, 200), bands, gains=g)
        b = multiband_blend([layers[i] for i in perm], [origins[i] for i in perm], (300, 200), bands, gains=g[perm])
        assert np.array_equal(a, b)
        assert np.array_equal(a, mo.multiband_blend(layers, origins, (300, 200), bands, gains=g))


@gpu
def test_multiband_c_entry_checks():
    import torch
    lib = rt.load_library()
    t = torch.zeros((4, 5, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((4, 5, 3), dtype=torch.uint8, device="cuda")
    lut = torch.zeros((1, 256), dtype=torch.uint8, device="cuda")
    ws = torch.empty(4096, dtype=torch.uint8, device="cuda")
    st = rt.stream_ptr(torch, out.device)
    P = ctypes.POINTER(ctypes.c_longlong)
    a = np.array([[t.data_ptr(), 4, 5, 15, 0, 0]], dtype=np.int64)
    need = ctypes.c_size_t()
    assert lib.apap_multiband_workspace_bytes(a.ctypes.data_as(P), 1, 4, 5, 5, ctypes.byref(need)) == 0

    def call(fn_gain=False, n=1, bands=5, ws_ptr=None, ws_bytes=None, out_bytes=60, lut_ptr=-1, desc=a):
        w = ws.data_ptr() if ws_ptr is None else ws_ptr
        wb = need.value if ws_bytes is None else ws_bytes
        if fn_gain:
            return lib.apap_multiband_blend_gain(desc.ctypes.data_as(P), n, 4, 5, bands,
                                                 lut.data_ptr() if lut_ptr == -1 else lut_ptr, w, wb, out.data_ptr(),
                                                 out_bytes, st)
        return lib.apap_multiband_blend(desc.ctypes.data_as(P), n, 4, 5, bands, w, wb, out.data_ptr(), out_bytes, st)
    for g in (False, True):
        assert call(g) == 0
        assert call(g, n=0) == -1 and call(g, n=128, desc=np.repeat(a, 128, 0)) == -1
        assert call(g, bands=-1) == -1
        assert call(g, ws_bytes=need.value - 1) == -1
        assert call(g, out_bytes=59) == -1
        assert call(g, ws_ptr=0) == -1
        assert call(g, ws_ptr=ws.data_ptr() + 8) == -2
        assert call(g, desc=np.array([[t.data_ptr(), 4, 5, 14, 0, 0]], dtype=np.int64)) == -1
    assert call(True, lut_ptr=None) == -1
    torch.cuda.synchronize()
    assert (out.cpu().numpy() == 0).all()                       # an all-zero layer blends to 0


# ----------------------------------------------------------------------------------------------- GPU: driver
def _check_multiband(monkeypatch, centre, others, raw_c, raw_os, ransac, exposure, live=False, **kw):
    from cvx_proj_b200.driver import stitch_panorama
    from tests.test_case import _assert_results_equal
    from tests.test_feather import _feather_layers
    res = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend="multiband", exposure=exposure, **kw)
    mean = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, **kw)
    assert len(res) == 4 and res.final_size == mean.final_size and np.array_equal(res.origins, mean.origins)
    assert len(res.pairs) == len(mean.pairs)
    for i, (g, w) in enumerate(zip(res.pairs, mean.pairs)):
        _assert_results_equal(g, w, i)
    warps = kw.get("warp_imgs") or others
    layers, origins, size = _feather_layers(res, warps, centre, monkeypatch)
    gains = go.gains(layers, origins, size) if exposure == "gain" else None
    bands = kw.get("bands", 5)
    assert isinstance(res.panorama, np.ndarray) and res.panorama.shape == (size[1], size[0], 3)
    assert np.array_equal(res.panorama, mo.multiband_blend(layers, origins, size, bands, gains=gains))
    if live:
        assert np.array_equal(res.panorama, _opencv(layers, origins, size, bands))


def _dimmed(imgs):
    return [np.clip(np.rint(img * (0.7 + 0.2 * j)), 0, 255).astype(np.uint8) for j, img in enumerate(imgs)]


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("exposure", ["none", "gain"])
def test_stitch_panorama_multiband_c1(ransac, exposure, monkeypatch):
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    _check_multiband(monkeypatch, centre, others, raw_c, raw_os, ransac, exposure, live=exposure == "none",
                     warp_imgs=_dimmed(others))


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("exposure", ["none", "gain"])
def test_stitch_panorama_multiband_c4(ransac, exposure, monkeypatch):
    from tests.test_case import _scene
    centre, others, raw_c, raw_os = _scene("c4", 6)
    _check_multiband(monkeypatch, centre, others, raw_c, raw_os, ransac, exposure, warp_imgs=_dimmed(others), bands=7)


@gpu
def test_stitch_panorama_multiband_no_other_image():
    from cvx_proj_b200.driver import stitch_panorama
    from cvx_proj_b200.utils import multiband_blend
    centre, _, raw_c, _ = _scene_2d("c1", 1)
    for exposure in ("none", "gain"):
        res = stitch_panorama(centre, [], raw_c, [], blend="multiband", exposure=exposure)
        h, w = centre.shape[:2]
        assert res.pairs == [] and res.final_size == (w, h, 0, 0)
        assert np.array_equal(res.panorama, multiband_blend([centre], [(0, 0)], (w, h)))
        assert np.array_equal(res.panorama, mo.multiband_blend([centre], [(0, 0)], (w, h)))
