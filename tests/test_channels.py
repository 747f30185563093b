"""Per-channel exposure compensation of a panorama: ``oracle.channels_oracle`` pinned against the live
``cv.detail.ChannelsCompensator`` (gains bit for bit, ``apply``, and the compensate-then-blend chains), the statistics
kernel (``k_gain_stats<true>``) and the blends with per-channel tables against the oracle, and
``driver.stitch_panorama(exposure="channels")`` against the oracle composite."""
import ctypes

import cv2 as cv
import numpy as np
import pytest

from cvx_proj_b200 import _runtime as rt
from oracle import channels_oracle as co
from oracle import feather_oracle as fo
from oracle import gain_oracle as go
from tests.test_gain import _all_cases, _dimmed, _masks
from tests.test_panorama import _random_case, _random_image, _scene_2d

gpu = pytest.mark.gpu


def _cast(layers, seed):
    """Each layer with its own colour cast: one channel scaled by a factor of its own."""
    r = np.random.default_rng(seed)
    out = []
    for k, img in enumerate(layers):
        f = np.ones(3)
        f[k % 3] = r.uniform(0.6, 1.4)
        out.append(np.clip(np.rint(img * f), 0, 255).astype(np.uint8))
    return out


def _random_sets():
    """(name, layers, origins, size): random placed-layer sets of 1 to 20 layers, ragged and clipped, with holes and
    casts, plus skipped and all-zero layers."""
    out = []
    for s in range(12):
        r = np.random.default_rng(100 + s)
        n = int(r.integers(1, 21))
        size = (int(r.integers(20, 90)), int(r.integers(15, 70)))
        layers, origins = _random_case(200 + s, size, n, (size[0] * 2 // 3, size[1] * 2 // 3))
        if s % 4 == 1:
            layers[0] = np.zeros_like(layers[0])
        if s % 4 == 2:
            origins[-1] = (size[0] + 5, 0)                       # outside the canvas: skipped
        out.append((f"random-{s}", _cast(layers, s), origins, size))
    return out


def _cases():
    return [(name, _cast(layers, k), origins, size) for k, (name, layers, origins, size) in enumerate(_all_cases())] \
        + _random_sets()


def _opencv(layers, origins, size, blender=None):
    """ChannelsCompensator fed as channel_gains' contract says; with ``blender`` (a prepared OpenCV blender) its
    ``apply`` per layer with the raw mask kept, then the blend.  Returns ``(gains [n, 3], panorama or None)``."""
    ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
    ms = _masks(ps)
    comp = cv.detail.ChannelsCompensator()
    comp.feed([(0, 0)] * len(ps), [cv.UMat(p) for p in ps], [cv.UMat(m) for m in ms])
    g = np.array([np.asarray(v, np.float64).reshape(-1)[:3] for v in comp.getMatGains()])
    if blender is None:
        return g, None
    blender.prepare((0, 0, size[0], size[1]))
    for k, (p, m) in enumerate(zip(ps, ms)):
        blender.feed(comp.apply(k, (0, 0), p.copy(), m).astype(np.int16), m, (0, 0))
    res, _ = blender.blend(None, None)
    return g, np.clip(res, 0, 255).astype(np.uint8)


def _differ(layers, origins, size, ga, gb):
    """Pixels where some layer's compensated bytes differ under the gains ``ga`` and ``gb``."""
    d = np.zeros((size[1], size[0]), bool)
    for img, o, a, b in zip(layers, origins, ga, gb):
        p = fo.paste(img, o, size)
        d |= (co.apply(p, a) != co.apply(p, b)).any(axis=-1)
    return d


# ----------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("case", range(len(_cases())))
def test_oracle_gains_are_opencv_bit_for_bit(case):
    name, layers, origins, size = _cases()[case]
    want, _ = _opencv(layers, origins, size)
    got = co.gains(layers, origins, size)
    assert got.shape == (len(layers), 3) and got.dtype == np.float64
    assert np.array_equal(got, want), (name, got, want)


def test_shipped_solve_per_channel_is_opencv():
    """channel_gains' host half: utils.solve_gains on the exact channel sums shifted left by 52."""
    from cvx_proj_b200.utils import solve_gains
    for name, layers, origins, size in _cases():
        count, sums = co.stats(layers, origins, size)
        got = np.stack([solve_gains(count, [[v << 52 for v in row] for row in sums[c]]) for c in range(3)], axis=1)
        assert np.array_equal(got, _opencv(layers, origins, size)[0]), name


def test_channel_counts_are_the_gain_counts():
    for name, layers, origins, size in _cases()[:6]:
        assert co.stats(layers, origins, size)[0] == go.stats(layers, origins, size)[0], name


def test_apply_is_opencv_apply():
    r = np.random.default_rng(4)
    v = np.arange(256, dtype=np.uint8).reshape(1, 256, 1).repeat(3, axis=2)
    mask = np.full((1, 256), 255, np.uint8)
    ties = [(0.5, 1.5, 2.5), (0.0, 1.0, 3.0), (2.5, 0.5, 0.0)]
    for g in ties + [tuple(t) for t in r.uniform(0.0, 3.0, (2000, 3))]:
        comp = cv.detail.ChannelsCompensator()               # setMatGains appends: a fresh one per triple
        comp.setMatGains([np.array([[g[0]], [g[1]], [g[2]], [0.0]])])
        want = comp.apply(0, (0, 0), v.copy(), mask)
        assert np.array_equal(co.apply(v, g), want), g


@pytest.mark.parametrize("blend", ["feather", "multiband"])
def test_oracle_composite_is_opencv_chain(blend):
    """Equal wherever no layer's v g rounds differently under OpenCV's gains and the oracle's (here the gains are
    equal, so everywhere); with OpenCV's own gains the oracle composite is OpenCV's."""
    for name, layers, origins, size in _cases()[:14]:
        if blend == "feather":
            g_cv, want = _opencv(layers, origins, size, cv.detail.FeatherBlender(0.05))
            got = co.feather_blend(layers, origins, size, g_cv, 0.05)
        else:
            g_cv, want = _opencv(layers, origins, size, cv.detail_MultiBandBlender(0, 3, cv.CV_16S))
            got = co.multiband_blend(layers, origins, size, g_cv, 3)
        assert np.array_equal(got, want), (name, blend)
        g_or = co.gains(layers, origins, size)
        d = _differ(layers, origins, size, g_cv, g_or)
        mine = (co.feather_blend(layers, origins, size, g_or, 0.05) if blend == "feather"
                else co.multiband_blend(layers, origins, size, g_or, 3))
        assert np.array_equal(mine[~d], want[~d]), (name, blend)


def test_equal_columns_are_one_gain():
    name, layers, origins, size = _all_cases()[0]
    g = np.random.default_rng(1).uniform(0.3, 2.5, len(layers))
    g3 = np.repeat(g[:, None], 3, axis=1)
    assert np.array_equal(co.blend_layers(layers, origins, size, g3), go.blend_layers(layers, origins, size, g))
    assert np.array_equal(co.feather_blend(layers, origins, size, g3), go.feather_blend(layers, origins, size, g))


def test_channel_argument_errors_before_any_launch():
    from cvx_proj_b200.utils import blend_layers, channel_gains, feather_blend, multiband_blend
    img = np.zeros((4, 5, 3), np.uint8)
    with pytest.raises(ValueError, match="257"):
        channel_gains([img] * 257, [(0, 0)] * 257, (5, 4))
    with pytest.raises(ValueError, match="layers"):
        channel_gains([], [], (5, 4))
    with pytest.raises(ValueError, match="origin"):
        channel_gains([img, img], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="uint8"):
        channel_gains([img.astype(np.float32)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="positive"):
        channel_gains([img], [(0, 0)], (5, 0))
    bads = ([[1.0, 1.0]], [[1.0, 1.0, 1.0]], [[1.0] * 3, [1.0] * 2], [[1.0] * 4] * 2, [[1.0] * 3, [1.0, np.nan, 1.0]],
            [[1.0] * 3, [np.inf, 1.0, 1.0]], np.ones((2, 3, 1)), np.ones((3, 2)), np.ones((2, 1)))
    for fn in (blend_layers, feather_blend, multiband_blend):
        for bad in bads:
            with pytest.raises(ValueError, match="gains"):
                fn([img, img], [(0, 0), (1, 1)], (5, 4), gains=bad)


def test_stitch_panorama_exposure_errors_before_any_keypoint_work():
    from cvx_proj_b200.driver import stitch_panorama
    img = np.zeros((4, 5, 3), np.uint8)
    for bad in ("channel", "Channels", "gain ", ["channels"]):
        with pytest.raises(ValueError, match="exposure.*'channels'"):
            stitch_panorama(img, [img], None, [None], exposure=bad)


# ----------------------------------------------------------------------------------------------- GPU: kernels
def _gpu_stats(layers, origins, size):
    """apap_channel_stats' words as Python ints ``(count, sums[c])``, from numpy or tensor layers."""
    import torch
    from cvx_proj_b200.utils import _layer_descs
    on_device = not isinstance(layers[0], np.ndarray)
    dev = layers[0].device if on_device else torch.device("cuda", torch.cuda.current_device())
    devs, desc = _layer_descs(torch, dev, layers, origins, on_device)
    lib = rt.load_library()
    n = len(devs)
    nb = ctypes.c_size_t()
    rt.check(lib.apap_gain_stats_bytes(n, ctypes.byref(nb)), "bytes")
    stats = torch.full((nb.value // 8,), -1, dtype=torch.int64, device=dev)    # the call must clear it
    rt.check(lib.apap_channel_stats(desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), n, size[1], size[0],
                                    stats.data_ptr(), nb.value, rt.stream_ptr(torch, dev)), "apap_channel_stats")
    w = stats.cpu().numpy().view(np.uint64).reshape(4, n, n)
    return [[int(v) for v in row] for row in w[0]], [[[int(v) for v in row] for row in w[1 + c]] for c in range(3)]


def _assert_stats(got, want, name=""):
    (count, sums), (wc, ws) = got, want
    n = len(wc)
    for i in range(n):
        for j in range(n):
            assert count[i][j] == (wc[i][j] if i <= j else 0), (name, i, j)
            for c in range(3):
                assert sums[c][i][j] == (ws[c][i][j] if i != j else 0), (name, c, i, j)


@gpu
def test_channel_stats_equal_oracle_integers():
    for name, layers, origins, size in _cases():
        _assert_stats(_gpu_stats(layers, origins, size), co.stats(layers, origins, size), name)


@gpu
def test_channel_stats_c2_size():
    r = np.random.default_rng(21)
    w, h = 4222, 2560
    big = r.integers(200, 256, (h, w, 3), dtype=np.uint8)
    big2 = r.integers(1, 256, (h - 100, w - 50, 3), dtype=np.uint8)
    small = _random_image(r, 300, 500)
    layers, origins = [big, big2, small], [(0, 0), (30, 60), (3000, 1500)]
    want = co.stats(layers, origins, (w, h))
    got = _gpu_stats(layers, origins, (w, h))
    _assert_stats(got, want, "c2")
    assert _gpu_stats(layers, origins, (w, h)) == got                  # two calls, the same bits


@gpu
@pytest.mark.parametrize("n", [2, 129, 256])
def test_channel_stats_many_layers_on_one_region(n):
    layers, origins = _random_case(40 + n, (70, 21), n, (60, 20))
    _assert_stats(_gpu_stats(layers, origins, (70, 21)), co.stats(layers, origins, (70, 21)), n)


@gpu
def test_channel_stats_tensor_views_and_numpy():
    """Crops of a larger tensor at odd byte offsets, read in place; numpy and tensor inputs give the same result."""
    import torch
    from cvx_proj_b200.utils import channel_gains
    r = np.random.default_rng(11)
    big = _random_image(r, 300, 701, black=0.05)
    big_t = torch.from_numpy(big).cuda()
    crops = [(0, 0, 300, 701), (3, 1, 120, 333), (17, 5, 18, 6), (100, 257, 101, 258), (5, 7, 200, 8), (9, 11, 10, 600)]
    layers_t = [big_t[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    layers_np = [big[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    assert any(t.data_ptr() % 4 for t in layers_t) and any(t.stride(0) != 3 * t.shape[1] for t in layers_t)
    origins = [(-5, 3), (100, -20), (650, 280), (0, 0), (333, 100), (150, 200)]
    canvas = (701, 310)
    want = co.stats(layers_np, origins, canvas)
    _assert_stats(_gpu_stats(layers_t, origins, canvas), want, "tensor")
    _assert_stats(_gpu_stats(layers_np, origins, canvas), want, "numpy")
    g = co.gains_from_stats(*want)
    assert np.array_equal(channel_gains(layers_t, origins, canvas), g)
    assert np.array_equal(channel_gains(layers_np, origins, canvas), g)


@gpu
def test_channel_gains_equal_opencv():
    from cvx_proj_b200.utils import channel_gains
    for name, layers, origins, size in _cases():
        got = channel_gains(layers, origins, size)
        assert got.dtype == np.float64 and got.shape == (len(layers), 3)
        assert np.array_equal(got, co.gains(layers, origins, size)), name
        assert np.array_equal(got, _opencv(layers, origins, size)[0]), name


@gpu
def test_blends_with_channel_gains_equal_oracle():
    from cvx_proj_b200.utils import blend_layers, channel_gains, feather_blend, multiband_blend
    r = np.random.default_rng(12)
    for name, layers, origins, size in _cases()[:14]:
        n = len(layers)
        for g in (channel_gains(layers, origins, size), np.full((n, 3), 3.0), r.uniform(0.3, 2.5, (n, 3))):
            assert np.array_equal(blend_layers(layers, origins, size, gains=g),
                                  co.blend_layers(layers, origins, size, g)), name
            assert np.array_equal(feather_blend(layers, origins, size, 0.05, gains=g),
                                  co.feather_blend(layers, origins, size, g, 0.05)), name
            assert np.array_equal(multiband_blend(layers, origins, size, 3, gains=g),
                                  co.multiband_blend(layers, origins, size, g, 3)), name


@gpu
def test_equal_columns_give_the_one_gain_bits():
    from cvx_proj_b200.utils import blend_layers, feather_blend, multiband_blend
    r = np.random.default_rng(14)
    for name, layers, origins, size in _cases()[:14]:
        g = r.uniform(0.3, 2.5, len(layers))
        g3 = np.repeat(g[:, None], 3, axis=1)
        assert np.array_equal(blend_layers(layers, origins, size, gains=g3), blend_layers(layers, origins, size, gains=g))
        assert np.array_equal(feather_blend(layers, origins, size, gains=g3),
                              feather_blend(layers, origins, size, gains=g))
        assert np.array_equal(multiband_blend(layers, origins, size, gains=g3),
                              multiband_blend(layers, origins, size, gains=g))


@gpu
def test_layer_order_does_not_change_mean_and_multiband():
    from cvx_proj_b200.utils import blend_layers, multiband_blend
    layers, origins = _random_case(31, (300, 200), 40, (150, 120))
    g = np.random.default_rng(2).uniform(0.3, 2.5, (40, 3))
    perm = np.random.default_rng(3).permutation(40)
    pl, po = [layers[i] for i in perm], [origins[i] for i in perm]
    for fn in (blend_layers, multiband_blend):
        assert np.array_equal(fn(layers, origins, (300, 200), gains=g), fn(pl, po, (300, 200), gains=g[perm]))
    assert np.array_equal(blend_layers(layers, origins, (300, 200), gains=g), co.blend_layers(layers, origins, (300, 200), g))


@gpu
def test_channel_c_entry_checks():
    import torch
    lib = rt.load_library()
    t = torch.zeros((4, 5, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((4, 5, 3), dtype=torch.uint8, device="cuda")
    stats = torch.empty(64, dtype=torch.int64, device="cuda")
    lut = torch.zeros((1, 3, 256), dtype=torch.uint8, device="cuda")
    ws = torch.empty(1 << 16, dtype=torch.uint8, device="cuda")
    st = rt.stream_ptr(torch, out.device)
    P = ctypes.POINTER(ctypes.c_longlong)
    good = np.asarray([t.data_ptr(), 4, 5, 15, 0, 0], dtype=np.int64).reshape(1, 6)

    def stats_call(d, n, nbytes=32, ptr=None):
        a = np.asarray(d, dtype=np.int64).reshape(-1, 6)
        return lib.apap_channel_stats(a.ctypes.data_as(P), n, 4, 5, stats.data_ptr() if ptr is None else ptr, nbytes,
                                      st)
    assert stats_call(good, 1) == 0
    torch.cuda.synchronize()
    assert (stats.cpu().numpy()[:4] == 0).all()
    for d, n, kw in ((good, 0, {}), (np.repeat(good, 257, axis=0), 257, {"nbytes": 1 << 22}), (good, 1, {"nbytes": 31}),
                     ([0, 4, 5, 15, 0, 0], 1, {}), ([t.data_ptr(), 4, 5, 14, 0, 0], 1, {}), (good, 1, {"ptr": 0})):
        assert stats_call(d, n, **kw) == -1, (n, kw)
        assert "channel_stats" in lib.apap_last_error().decode()
    assert stats_call(good, 1, ptr=stats.data_ptr() + 4) == -2
    d = good.ctypes.data_as(P)
    assert lib.apap_blend_layers_channels(d, 1, 4, 5, lut.data_ptr(), out.data_ptr(), 60, st) == 0
    assert lib.apap_blend_layers_channels(d, 1, 4, 5, None, out.data_ptr(), 60, st) == -1
    assert lib.apap_blend_layers_channels(d, 1, 4, 5, lut.data_ptr(), out.data_ptr(), 59, st) == -1
    assert lib.apap_feather_blend_channels(d, 1, 4, 5, 0.02, lut.data_ptr(), ws.data_ptr(), ws.numel(),
                                           out.data_ptr(), 60, st) == 0
    assert lib.apap_feather_blend_channels(d, 1, 4, 5, 0.02, None, ws.data_ptr(), ws.numel(), out.data_ptr(), 60,
                                           st) == -1
    assert lib.apap_multiband_blend_channels(d, 1, 4, 5, 5, lut.data_ptr(), ws.data_ptr(), ws.numel(),
                                             out.data_ptr(), 60, st) == 0
    assert lib.apap_multiband_blend_channels(d, 1, 4, 5, 5, None, ws.data_ptr(), ws.numel(), out.data_ptr(), 60,
                                             st) == -1
    assert lib.apap_multiband_blend_channels(d, 0, 4, 5, 5, lut.data_ptr(), ws.data_ptr(), ws.numel(),
                                             out.data_ptr(), 60, st) == -1
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------- GPU: driver
def _check_channels(monkeypatch, centre, others, raw_c, raw_os, ransac, blend, live=False, **kw):
    from cvx_proj_b200.driver import stitch_panorama
    from tests.test_case import _assert_results_equal
    from tests.test_feather import _feather_layers
    res = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend=blend, exposure="channels", **kw)
    none = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, blend=blend, exposure="none", **kw)
    assert len(res) == 4 and res.final_size == none.final_size and np.array_equal(res.origins, none.origins)
    assert len(res.pairs) == len(none.pairs)
    for i, (g, w) in enumerate(zip(res.pairs, none.pairs)):
        _assert_results_equal(g, w, i)
    layers, origins, size = _feather_layers(res, kw.get("warp_imgs") or others, centre, monkeypatch)
    g = co.gains(layers, origins, size)
    assert not np.allclose(g, g[:, :1])                          # the casts give different gains per channel
    want = {"mean": lambda: co.blend_layers(layers, origins, size, g),
            "feather": lambda: co.feather_blend(layers, origins, size, g),
            "multiband": lambda: co.multiband_blend(layers, origins, size, g)}[blend]()
    assert np.array_equal(res.panorama, want)
    if live and blend != "mean":
        blender = cv.detail.FeatherBlender(0.02) if blend == "feather" else cv.detail_MultiBandBlender(0, 5, cv.CV_16S)
        g_cv, cv_pano = _opencv(layers, origins, size, blender)
        assert np.array_equal(g, g_cv)
        d = _differ(layers, origins, size, g_cv, g)
        assert np.array_equal(res.panorama[~d], cv_pano[~d])


def _tinted(imgs):
    return _cast(_dimmed(imgs), 9)


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("blend", ["mean", "feather", "multiband"])
def test_stitch_panorama_exposure_channels_c1(ransac, blend, monkeypatch):
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    _check_channels(monkeypatch, centre, others, raw_c, raw_os, ransac, blend, live=True, warp_imgs=_tinted(others))


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
@pytest.mark.parametrize("blend", ["mean", "feather", "multiband"])
def test_stitch_panorama_exposure_channels_c4(ransac, blend, monkeypatch):
    from tests.test_case import _scene
    centre, others, raw_c, raw_os = _scene("c4", 6)
    _check_channels(monkeypatch, centre, others, raw_c, raw_os, ransac, blend, warp_imgs=_tinted(others))


@gpu
def test_stitch_panorama_exposure_channels_no_other_image():
    from cvx_proj_b200.driver import stitch_panorama
    centre, _, raw_c, _ = _scene_2d("c1", 1)
    for blend in ("mean", "feather", "multiband"):
        a = stitch_panorama(centre, [], raw_c, [], blend=blend, exposure="channels")
        b = stitch_panorama(centre, [], raw_c, [], blend=blend)
        assert a.pairs == [] and a.final_size == b.final_size and np.array_equal(a.panorama, b.panorama)
