"""One panorama of a case: the N-layer mean blend (``k_blend_layers`` / ``utils.blend_layers``) against its numpy
restatement ``oracle.panorama_oracle.blend_layers``, and ``driver.stitch_panorama`` against ``stitch_pair`` (one other
image) and against the oracle composite of per-pair ``local_warp`` canvases plus the centre (several)."""
import functools

import cv2 as cv
import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from cvx_proj_b200 import synth
from cvx_proj_b200.driver import panorama_size
from oracle import apap_oracle as orc
from oracle import panorama_oracle as po

gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------------------------- CPU
def test_panorama_size_of_one_pair_is_its_final_size():
    for fs in ((2701, 1897, 0, 407), (1920, 1080, 0, 0), (4222, 2560, 1130, 312)):
        size, origins = panorama_size([fs])
        assert size == fs
        assert origins.tolist() == [[0, 0]]


@settings(max_examples=200, deadline=None)
@given(st.lists(st.tuples(st.integers(0, 3000), st.integers(0, 3000), st.integers(1, 3000), st.integers(1, 3000)),
                min_size=1, max_size=20))
def test_panorama_union_contains_every_pair_canvas(boxes):
    """Pair canvases built as final_size builds them (they contain the centre's [0, w) x [0, h) with w = h = 1 here):
    offset ox, extent W >= ox + 1.  The union holds each one at its origin and is the smallest box that does."""
    fs = [(ox + w, oy + h, ox, oy) for ox, oy, w, h in boxes]
    (width, height, ox, oy), origins = panorama_size(fs)
    assert origins.shape == (len(fs), 2)
    for (wk, hk, oxk, oyk), (x0, y0) in zip(fs, origins):
        assert x0 >= 0 and y0 >= 0 and x0 + wk <= width and y0 + hk <= height
        assert (x0 + oxk, y0 + oyk) == (ox, oy)          # every canvas puts the centre at the panorama's (OX, OY)
    assert origins[:, 0].min() == 0 and origins[:, 1].min() == 0
    assert max(x0 + f[0] for f, (x0, _) in zip(fs, origins)) == width
    assert max(y0 + f[1] for f, (_, y0) in zip(fs, origins)) == height


def test_panorama_size_needs_a_pair():
    with pytest.raises(ValueError):
        panorama_size([])


def _random_image(r, h, w, black=0.2):
    img = r.integers(0, 256, (h, w, 3), dtype=np.uint8)
    img[r.random((h, w)) < black] = 0                    # black pixels inside the layer
    img[r.random((h, w)) < 0.05, 0] = 0                  # partly black pixels stay non-empty
    return img


def test_oracle_two_equal_layers_is_uniform_blend():
    r = np.random.default_rng(0)
    for h, w in ((1, 1), (7, 13), (64, 33)):
        a, b = _random_image(r, h, w), _random_image(r, h, w)
        got = po.blend_layers([a, b], [(0, 0), (0, 0)], (w, h))
        assert np.array_equal(got, orc.uniform_blend(a, b))
        assert np.array_equal(got, orc.uniform_blend_float(a, b))


def test_floor_division_by_reciprocal_is_exact():
    """k_blend_layers divides s by n >= 2 as __umulhi(s, ceil(2^32 / n)), ceil(2^32 / n) = floor((2^32 - 1) / n) + 1
    in uint32; n <= 1 takes s itself.  Every n <= 256 and s <= 255 n."""
    for n in range(2, 257):
        m = np.uint64(0xFFFFFFFF // n + 1)
        assert m < 2 ** 32
        s = np.arange(255 * n + 1, dtype=np.uint64)
        assert np.array_equal((s * m) >> np.uint64(32), s // np.uint64(n)), n


def test_blend_layers_argument_errors_before_any_launch():
    from cvx_proj_b200.utils import blend_layers
    img = np.zeros((4, 5, 3), np.uint8)
    with pytest.raises(ValueError, match="257"):
        blend_layers([img] * 257, [(0, 0)] * 257, (5, 4))
    with pytest.raises(ValueError, match="layers"):
        blend_layers([], [], (5, 4))
    with pytest.raises(ValueError, match="origin"):
        blend_layers([img, img], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="origin"):
        blend_layers([img], [(0, 0, 0)], (5, 4))
    with pytest.raises(ValueError, match=r"\[h, w, 3\]"):
        blend_layers([np.zeros((4, 5), np.uint8)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match=r"\[h, w, 3\]"):
        blend_layers([np.zeros((4, 5, 4), np.uint8)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match=r"\[h, w, 3\]"):
        blend_layers([np.zeros((0, 5, 3), np.uint8)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="uint8"):
        blend_layers([img.astype(np.float32)], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match="positive"):
        blend_layers([img], [(0, 0)], (0, 4))


# ----------------------------------------------------------------------------------------------- GPU: kernel
def _random_case(seed, canvas, n, max_wh):
    """``n`` layers of ragged sizes (1 x 1 and 1 px wide ones included) at origins that may be negative or stick out
    of the ``canvas = (width, height)``."""
    r = np.random.default_rng(seed)
    width, height = canvas
    layers, origins = [], []
    for k in range(n):
        if k % 7 == 3:
            h, w = 1, 1
        elif k % 7 == 5:
            h, w = int(r.integers(1, max_wh[1] + 1)), 1
        else:
            h, w = int(r.integers(1, max_wh[1] + 1)), int(r.integers(1, max_wh[0] + 1))
        layers.append(_random_image(r, h, w))
        origins.append((int(r.integers(-w // 2 - 3, width - w // 2 + 3)), int(r.integers(-h // 2 - 3, height - h // 2 + 3))))
    return layers, origins


@gpu
@pytest.mark.parametrize("seed,canvas,n,max_wh", [
    (0, (17, 11), 5, (9, 7)),              # odd widths, one CTA segment
    (1, (1, 1), 3, (2, 2)),                # 1 x 1 canvas
    (2, (1, 40), 6, (1, 30)),              # 1 px wide canvas and layers
    (3, (2501, 37), 12, (1900, 30)),       # segments of 1024 pixels, odd canvas width
    (4, (3000, 64), 40, (2600, 60)),
    (5, (1023, 9), 9, (1100, 12)),         # layers wider than the canvas
    (6, (257, 301), 256, (200, 200)),      # the most layers
])
def test_blend_layers_equals_oracle(seed, canvas, n, max_wh):
    from cvx_proj_b200.utils import blend_layers
    layers, origins = _random_case(seed, canvas, n, max_wh)
    got = blend_layers(layers, origins, canvas)
    assert isinstance(got, np.ndarray) and got.shape == (canvas[1], canvas[0], 3) and got.dtype == np.uint8
    assert np.array_equal(got, po.blend_layers(layers, origins, canvas))


@gpu
def test_blend_layers_tensor_views():
    """Crops of larger tensors (odd start byte, row pitch of the parent), layers in place, out on the device."""
    import torch
    from cvx_proj_b200.utils import blend_layers
    r = np.random.default_rng(11)
    big = _random_image(r, 300, 701)
    big_t = torch.from_numpy(big).cuda()
    crops = [(0, 0, 300, 701), (3, 1, 120, 333), (17, 5, 18, 6), (100, 257, 101, 258), (5, 7, 200, 8), (9, 11, 10, 600)]
    layers_t = [big_t[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    layers_np = [big[r0:r1, c0:c1] for r0, c0, r1, c1 in crops]
    assert any(t.data_ptr() % 4 for t in layers_t) and any(t.stride(0) != 3 * t.shape[1] for t in layers_t)
    origins = [(-5, 3), (100, -20), (650, 280), (0, 0), (333, 100), (150, 200)]
    canvas = (701, 310)
    want = po.blend_layers(layers_np, origins, canvas)
    got = blend_layers(layers_t, origins, canvas)
    assert got.is_cuda and got.device == big_t.device
    assert np.array_equal(got.cpu().numpy(), want)
    # a transposed view (strides that are not (pitch, 3, 1)) is made contiguous first
    tr = big_t[:50, :40].transpose(0, 1)
    assert np.array_equal(blend_layers([tr], [(2, 1)], (45, 60)).cpu().numpy(),
                          po.blend_layers([big[:50, :40].transpose(1, 0, 2)], [(2, 1)], (45, 60)))


@gpu
def test_blend_layers_sum_bound_and_one_layer():
    from cvx_proj_b200.utils import blend_layers
    full = np.full((9, 1030, 3), 255, np.uint8)
    got = blend_layers([full] * 256, [(0, 0)] * 256, (1030, 9))       # s = 255 x 256 = 65 280, n = 256
    assert (got == 255).all()
    odd = [full.copy() for _ in range(256)]
    for k, img in enumerate(odd):
        img[..., k % 3] = k % 256
    assert np.array_equal(blend_layers(odd, [(k % 5, 0) for k in range(256)], (1034, 9)),
                          po.blend_layers(odd, [(k % 5, 0) for k in range(256)], (1034, 9)))
    r = np.random.default_rng(3)
    one = _random_image(r, 33, 45)
    assert np.array_equal(blend_layers([one], [(0, 0)], (45, 33)), one)
    assert np.array_equal(blend_layers([one], [(-3, 2)], (40, 40)), po.blend_layers([one], [(-3, 2)], (40, 40)))


@gpu
def test_blend_layers_two_equal_layers_is_uniform_blend():
    from cvx_proj_b200.apap_utils import uniform_blend
    from cvx_proj_b200.utils import blend_layers
    r = np.random.default_rng(4)
    for h, w in ((1, 1), (5, 7), (1081, 1921)):
        a, b = _random_image(r, h, w), _random_image(r, h, w)
        assert np.array_equal(blend_layers([a, b], [(0, 0), (0, 0)], (w, h)), uniform_blend(a, b))


@gpu
def test_blend_layers_order_independent():
    from cvx_proj_b200.utils import blend_layers
    layers, origins = _random_case(8, (1500, 50), 30, (1200, 45))
    want = blend_layers(layers, origins, (1500, 50))
    for seed in range(3):
        perm = np.random.default_rng(seed).permutation(len(layers))
        got = blend_layers([layers[i] for i in perm], [origins[i] for i in perm], (1500, 50))
        assert np.array_equal(got, want)


@gpu
def test_blend_layers_errors():
    import ctypes

    import torch
    from cvx_proj_b200 import _runtime as rt
    from cvx_proj_b200.utils import blend_layers
    img = np.zeros((4, 5, 3), np.uint8)
    t = torch.zeros((4, 5, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="257"):
        blend_layers([t] * 257, [(0, 0)] * 257, (5, 4))
    with pytest.raises(ValueError, match="all numpy"):
        blend_layers([img, t], [(0, 0)] * 2, (5, 4))
    with pytest.raises(ValueError, match="CUDA tensor"):
        blend_layers([t, torch.zeros((4, 5, 3), dtype=torch.uint8)], [(0, 0)] * 2, (5, 4))
    with pytest.raises(ValueError, match="uint8"):
        blend_layers([t.float()], [(0, 0)], (5, 4))
    with pytest.raises(ValueError, match=r"\[h, w, 3\]"):
        blend_layers([t[..., :2]], [(0, 0)], (5, 4))
    # the C entry point checks its own arguments
    lib = rt.load_library()
    out = torch.empty((4, 5, 3), dtype=torch.uint8, device="cuda")
    st = rt.stream_ptr(torch, out.device)

    def call(desc, n, h=4, w=5, nbytes=60):
        arr = np.asarray(desc, dtype=np.int64).reshape(-1, 6)
        return lib.apap_blend_layers(arr.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), n, h, w, out.data_ptr(),
                                     nbytes, st)
    good = [t.data_ptr(), 4, 5, 15, 0, 0]
    assert call(good, 1) == 0
    torch.cuda.synchronize()
    for desc, n, kw in ((good, 0, {}), ([good] * 257, 257, {}), (good, 1, {"nbytes": 59}), (good, 1, {"h": 0}),
                        (good, 1, {"w": -1}), ([0, 4, 5, 15, 0, 0], 1, {}), ([t.data_ptr(), 0, 5, 15, 0, 0], 1, {}),
                        ([t.data_ptr(), 4, 5, 14, 0, 0], 1, {}), ([t.data_ptr(), 4, 5, 15, -(1 << 31), 0], 1, {})):
        assert call(desc, n, **kw) == -1, (n, kw)


# ----------------------------------------------------------------------------------------------- GPU: driver
@functools.lru_cache(maxsize=None)
def _scene_2d(name, k):
    """Like tests.test_case._scene, but the other images are shifted left and right, up and down, so that the
    panorama's OX and OY come from different pairs."""
    cfg = synth.CONFIGS[name]
    w, h = cfg["width"], cfg["height"]
    centre = synth.make_image(w, h, seed=2)
    r = np.random.default_rng(7)
    raw_c = (r.random((cfg["n_kp"], 2)) * [w - 48, h - 48] + 24).astype(np.float32)
    shifts = [(-0.12, 0.05), (0.06, -0.14), (-0.04, -0.06), (0.1, 0.08)]
    others, raw_os = [], []
    for j in range(k):
        a = 0.02 * (j + 1) * (-1) ** j
        sx, sy = shifts[j % len(shifts)]
        hom = np.array([[np.cos(a), -np.sin(a), sx * w], [np.sin(a), np.cos(a), sy * h], [1e-6 * (j + 1), -2e-6, 1.0]])
        hinv = np.linalg.inv(hom)
        others.append(cv.warpPerspective(centre, hinv, (w, h)))
        raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
        raw_os.append(raw_o + r.normal(0, 0.3, raw_o.shape).astype(np.float32))
    return centre, others, raw_c, raw_os


def _composite(res, warps, blend, gamma=0.5, sigma=100):
    """The oracle panorama from the pair results: each warp image through its grid by the numpy-in / numpy-out
    ``APAP.local_warp`` on its own canvas, placed at its origin, plus the centre image at (OX, OY)."""
    from cvx_proj_b200.apap import APAP
    layers = []
    for p, img in zip(res.pairs, warps):
        w, h, ox, oy = p.final_size
        layers.append(APAP(gamma, sigma, [w, h], [ox, oy]).local_warp(img, p.local_homography.copy(), p.mesh))
    width, height, ox, oy = res.final_size
    return po.blend_layers(layers + [blend], [tuple(o) for o in res.origins] + [(ox, oy)], (width, height))


def _check_case(centre, others, raw_c, raw_os, ransac, **kw):
    from cvx_proj_b200.driver import stitch_case, stitch_panorama
    from tests.test_case import _assert_results_equal
    res = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac, **kw)
    want = stitch_case(centre, others, raw_c, raw_os, ransac=ransac, stitch=False, **kw)
    assert len(res.pairs) == len(others)
    for i, (g, w) in enumerate(zip(res.pairs, want)):
        _assert_results_equal(g, w, i)
    size, origins = panorama_size([p.final_size for p in res.pairs])
    assert res.final_size == size and np.array_equal(res.origins, origins)
    assert isinstance(res.panorama, np.ndarray) and res.panorama.shape == (size[1], size[0], 3)
    warps = kw.get("warp_imgs") or others
    blend = kw.get("blend_img") if kw.get("blend_img") is not None else centre
    assert np.array_equal(res.panorama, _composite(res, warps, blend))
    return res


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
def test_stitch_panorama_one_pair_is_stitch_pair(ransac):
    from cvx_proj_b200.driver import stitch_panorama, stitch_pair
    from cvx_proj_b200.utils import keypoint_pairs
    from tests.test_case import _scene
    centre, others, raw_c, raw_os = _scene("c1", 1)
    want = stitch_pair(centre, others[0], *keypoint_pairs(centre, others[0], raw_c, raw_os[0], ransac=ransac))
    res = stitch_panorama(centre, others, raw_c, raw_os, ransac=ransac)
    assert res.final_size == want.final_size
    assert res.origins.tolist() == [[0, 0]]
    assert np.array_equal(res.panorama, want.stitched)


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
def test_stitch_panorama_shifted_both_ways(ransac):
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    res = _check_case(centre, others, raw_c, raw_os, ransac)
    offs = np.array([p.final_size[2:] for p in res.pairs])
    assert offs[:, 0].max() > 0 and offs[:, 1].max() > 0
    assert offs[:, 0].argmax() != offs[:, 1].argmax()    # OX and OY come from different pairs
    assert (res.origins[:, 0] > 0).any() and (res.origins[:, 1] > 0).any()


@gpu
@pytest.mark.parametrize("ransac", ["opencv", "gpu"])
def test_stitch_panorama_c4_ragged(ransac):
    from tests.test_case import _scene
    centre, others, raw_c, raw_os = _scene("c4", 6)
    _check_case(centre, others, raw_c, raw_os, ransac)


@gpu
def test_stitch_panorama_given_images():
    """The de-hazed images of the script as warp and blend images, with black regions in both."""
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    warps = [(255 - o) for o in others]
    for j, wimg in enumerate(warps):
        wimg[20 + 10 * j:90 + 10 * j, 30:200] = 0
    blend = synth.make_image(centre.shape[1], centre.shape[0], seed=9)
    blend[40:140, 60:400] = 0
    _check_case(centre, others, raw_c, raw_os, "opencv", warp_imgs=warps, blend_img=blend, mesh_size=40)


@gpu
def test_stitch_panorama_no_other_image_and_errors():
    import torch
    from cvx_proj_b200.driver import stitch_panorama
    centre, others, raw_c, raw_os = _scene_2d("c1", 3)
    res = stitch_panorama(centre, [], raw_c, [])
    assert res.pairs == [] and res.final_size == (centre.shape[1], centre.shape[0], 0, 0) and res.origins.shape == (0, 2)
    assert np.array_equal(res.panorama, centre)
    blend = synth.make_image(centre.shape[1], centre.shape[0], seed=9)
    assert np.array_equal(stitch_panorama(torch.from_numpy(centre).cuda(), [], raw_c, [], blend_img=blend).panorama,
                          blend)
    with pytest.raises(ValueError, match="warp images"):
        stitch_panorama(centre, others, raw_c, raw_os, warp_imgs=others[:2])
    with pytest.raises(ValueError, match="at most 255"):
        stitch_panorama(centre, others[:1] * 256, raw_c, raw_os[:1] * 256)
