"""Global-homography warp of the reference's README pipeline (SURVEY.md section 8f, row N4).

Mirror of ``image_warping`` in the reference's ``pyviz/utils.py:93-127`` -- same name, arguments and result:
the canvas is sized from the projected corners of the image to warp (``:99-112``), the image is warped onto it
with ``cv.warpPerspective`` semantics (bilinear, constant border 0, ``:114``) and the base image is either pasted
over the result (``direct_blend=True``, ``:124-125``) or mean-blended where the warp left something (``:115-123``,
the reference's "much slower" Python loop).  Warp and blend are one kernel (``k_warp_global``,
``csrc/warp_global.cu``), bit-exact with OpenCV's 8-bit fixed-point bilinear warp -- the INTER_LINEAR path with
coordinates in 1/32 pixel and 15-bit weights (``INTER_BITS = 5``, ``INTER_REMAP_COEF_BITS = 15``) that
``cv.warpPerspective`` takes for ``CV_8UC3``; the golden vectors (``tests/golden/ref_image_warping.npz``) were
produced with opencv-python 4.13.0, and OpenCV 3.x / 4.x releases share that path (a build that routes 8-bit images
through a different bilinear kernel would differ by +-1 in some pixels).  The O(1) host arithmetic
(corner projection, 3x3 inverse) restates ``cv.perspectiveTransform`` / ``cv::invert`` in numpy float64.
No CPU fallback.
"""
from __future__ import annotations

import ctypes
import math

import numpy as np

from . import _runtime as rt

__all__ = ["image_warping", "warp_perspective", "warping_canvas", "invert3x3", "match_descriptors", "coarse_matching",
           "sift_describe", "equalize_hist", "keypoint_pairs", "keypoint_pairs_batch", "find_homography_ransac",
           "find_homography_ransac_batch", "blend_layers", "feather_blend", "multiband_blend", "exposure_gains",
           "channel_gains"]


def invert3x3(m) -> np.ndarray:
    """Closed-form 3x3 inverse in the operation order of ``cv::invert`` (what ``cv.warpPerspective`` applies to
    its matrix); a singular matrix gives zeros like OpenCV."""
    m = np.asarray(m, dtype=np.float64)
    (a00, a01, a02), (a10, a11, a12), (a20, a21, a22) = m
    d = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20)
    if d == 0:
        return np.zeros((3, 3))
    d = 1.0 / d
    return np.array([[(a11 * a22 - a12 * a21) * d, (a02 * a21 - a01 * a22) * d, (a01 * a12 - a02 * a11) * d],
                     [(a12 * a20 - a10 * a22) * d, (a00 * a22 - a02 * a20) * d, (a02 * a10 - a00 * a12) * d],
                     [(a10 * a21 - a11 * a20) * d, (a01 * a20 - a00 * a21) * d, (a00 * a11 - a01 * a10) * d]])


def warping_canvas(base_shape, warp_shape, H):
    """``(canvas_w, canvas_h, t_x, t_y, Ht.dot(H))`` of pyviz/utils.py:99-112: the four corners of the image to
    warp go through ``H`` (``cv.perspectiveTransform``: float64 inside, float32 out), the canvas is their bounding
    box united with the base image, ``np.int32(min - 0.5)`` / ``np.int32(max + 0.5)``."""
    h1, w1 = base_shape[:2]
    h2, w2 = warp_shape[:2]
    m = np.asarray(H, dtype=np.float64)
    pts2 = np.array([[0, 0], [0, h2], [w2, h2], [w2, 0]], dtype=np.float32).astype(np.float64)
    z = m[2, 0] * pts2[:, 0] + m[2, 1] * pts2[:, 1] + m[2, 2]
    z = np.where(z != 0, 1.0 / np.where(z != 0, z, 1.0), 0.0)
    pts2_ = np.stack([(m[0, 0] * pts2[:, 0] + m[0, 1] * pts2[:, 1] + m[0, 2]) * z,
                      (m[1, 0] * pts2[:, 0] + m[1, 1] * pts2[:, 1] + m[1, 2]) * z], axis=1).astype(np.float32)
    pts = np.concatenate([np.array([[0, 0], [0, h1], [w1, h1], [w1, 0]], dtype=np.float32), pts2_], axis=0)
    xmin, ymin = np.int32(pts.min(axis=0) - 0.5)
    xmax, ymax = np.int32(pts.max(axis=0) + 0.5)
    tx, ty = int(-xmin), int(-ymin)
    ht = np.array([[1, 0, tx], [0, 1, ty], [0, 0, 1]])
    return int(xmax - xmin), int(ymax - ymin), tx, ty, ht.dot(np.asarray(H))


def _device_image(torch, device, img):
    if isinstance(img, np.ndarray):
        if img.ndim != 3 or img.shape[2] != 3:
            raise ValueError("expected an [H, W, 3] image")
        return rt.to_device(torch, device, img.astype(np.uint8, copy=False))
    return img.contiguous()


def warp_perspective(src, M, dsize, base=None, offset=(0, 0), mode=0, device=None, out=None):
    """``cv.warpPerspective(src, M, dsize)`` for ``uint8 [h, w, 3]`` images (bilinear, constant border 0), optionally
    fused with the paste (``mode=1``) or mean blend (``mode=2``) of ``base`` at ``offset`` on the canvas.  numpy in ->
    numpy out; CUDA tensors in -> the canvas stays on the device."""
    on_device = not isinstance(src, np.ndarray)
    torch, device = rt.torch_cuda(src.device if on_device else device)
    lib = rt.load_library()
    width, height = int(dsize[0]), int(dsize[1])
    src_dev = _device_image(torch, device, src)
    base_dev = _device_image(torch, device, base) if base is not None else None
    if out is None:
        out = torch.empty((height, width, 3), dtype=torch.uint8, device=device)
    minv = np.ascontiguousarray(invert3x3(M), dtype=np.float64)
    bh, bw = (base_dev.shape[0], base_dev.shape[1]) if base_dev is not None else (0, 0)
    with torch.cuda.device(device):
        rt.check(lib.apap_warp_perspective(
            src_dev.data_ptr(), src_dev.shape[0], src_dev.shape[1], minv.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            out.data_ptr(), height, width, base_dev.data_ptr() if base_dev is not None else None, bh, bw,
            int(offset[0]), int(offset[1]), int(mode), rt.stream_ptr(torch, device)), "apap_warp_perspective")
    return out if on_device else rt.to_host(torch, out)


def image_warping(img_base, img2warp, H, direct_blend=True, device=None):
    """Warp ``img2warp`` by the homography ``H`` onto a canvas that also holds ``img_base`` (pyviz/utils.py:93-127).

    ``direct_blend=True``: the base image covers the warped one; ``False``: the mean of the two where the warp is
    non-empty (any channel > 0), the base pixel elsewhere -- the ghosting view of the reference."""
    cw, ch, tx, ty, m = warping_canvas(img_base.shape, img2warp.shape, H)
    return warp_perspective(img2warp, m, (cw, ch), base=img_base, offset=(tx, ty), mode=1 if direct_blend else 2,
                            device=device)


def blend_layers(layers, origins, size, device=None, gains=None):
    """Mean blend of placed layers (``k_blend_layers``), the panorama blend of ``driver.stitch_panorama``.

    ``layers`` are ``uint8 [h, w, 3]`` images, ``origins`` their top-left canvas positions ``[(x0, y0), ...]`` (may be
    negative; a layer may stick out of the canvas and is clipped) and ``size = (width, height)`` the canvas.  Per
    pixel, with ``n`` the number of layers that are non-empty there (any channel > 0) and ``s`` their per-channel
    integer sum, the result is ``floor(s / n)``, 0 where ``n = 0`` -- for two equal layers at one origin exactly
    ``uniform_blend``, and independent of the layer order.  1 to 256 layers.

    ``gains`` (one finite float per layer, e.g. from ``exposure_gains``): layer k's bytes ``v`` become
    ``saturate(rint(v g_k))`` before they are summed, as ``cv.detail.GainCompensator.apply`` does; ``n`` still counts
    the layers non-empty before compensation.  Shape ``(n, 3)`` (e.g. from ``channel_gains``): byte ``v`` of channel
    ``c`` becomes ``saturate(rint(v g_kc))``, as ``cv.detail.ChannelsCompensator.apply`` does.  ``None`` leaves the
    bytes as they are.

    All numpy in -> numpy out (uploaded to ``device``); all CUDA tensors (one device) in -> a tensor on that device.
    Tensor layers are read in place when their pixels are packed (strides ``(pitch, 3, 1)``), so crops of a larger
    image need no copy.  No CPU fallback."""
    layers, origins, width, height, on_device, device = _check_layers("blend_layers", layers, origins, size,
                                                                       rt.BLEND_MAX_LAYERS, device)
    lut = None if gains is None else _gain_table("blend_layers", gains, len(layers))
    return _blend("apap_blend_layers", (), None, layers, origins, width, height, on_device, device, lut)


def feather_blend(layers, origins, size, sharpness=0.02, device=None, gains=None):
    """Feather blend of placed layers (``k_feather_rows``, ``k_feather_cols``, ``k_feather_blend``), bit for bit what
    ``cv.detail.FeatherBlender(sharpness)`` gives after ``prepare((0, 0, W, H))``, ``feed(P_k.astype(int16), mask_k,
    (0, 0))`` for every layer in the order given, and ``blend()``, converted to uint8 (``stitch_panorama(...,
    blend="feather")``).

    ``layers``, ``origins`` and ``size = (W, H)`` as for ``blend_layers``.  ``P_k`` is layer k pasted into a zero
    ``H x W`` canvas (clipped) and ``mask_k`` its non-empty pixels (any channel > 0).  Each layer's weight rises as
    ``min(D s, 1)`` (float32) with ``D`` the L1 distance to its nearest empty pixel -- pixels of the canvas outside the
    layer count as empty, the canvas border does not -- so seams between layers fade over about ``1 / s`` pixels.
    The weighted sum is kept as OpenCV keeps it (truncated int16 terms, float32 weights summed in layer order), so the
    last bits depend on the layer order.  Where one layer alone has weight 1 the result is ``v - 1`` for ``v >= 1``
    (``trunc(v / 1.00001)``): that is OpenCV's result, kept on purpose.

    1 to 128 layers (OpenCV's int16 accumulator holds 128 x 255).  ``sharpness`` must be a finite float32 of at least
    ``FLT_MIN`` (about 1.18e-38); below about 1.5e-5 the canvas must also have ``W + H <= 65536`` (distances are stored
    in 16 bits).  ``ValueError`` before any launch otherwise.  Inputs and outputs as ``blend_layers``.

    ``gains`` as for ``blend_layers``: the blender is fed the compensated ``P_k`` with the raw ``mask_k``, as OpenCV's
    stitching pipeline feeds it after ``GainCompensator.apply``; the distances, and so the weights, are unchanged.
    No CPU fallback."""
    layers, origins, width, height, on_device, device = _check_layers("feather_blend", layers, origins, size,
                                                                       rt.FEATHER_MAX_LAYERS, device)
    s = _feather_sharpness("feather_blend", sharpness)
    lut = None if gains is None else _gain_table("feather_blend", gains, len(layers))
    _feather_distance_cap(s, width, height)
    return _blend("apap_feather_blend", (s,), ("apap_feather_workspace_bytes", ()), layers, origins, width, height,
                  on_device, device, lut)


def multiband_blend(layers, origins, size, bands=5, device=None, gains=None):
    """Multi-band blend of placed layers (``k_mb_down``, ``k_mb_band``), bit for bit what
    ``cv.detail_MultiBandBlender(0, bands, cv.CV_16S)`` gives after ``prepare((0, 0, W, H))``, ``feed(P_k.astype(int16),
    mask_k, (0, 0))`` for every layer and ``blend()``, converted to uint8 with saturation (``stitch_panorama(...,
    blend="multiband")``).  ``P_k`` and ``mask_k`` as for ``feather_blend``.

    Each layer is split into Laplacian bands, and band ``i`` is blended with the mask blurred down to that band's
    scale: low frequencies mix over a wide seam, edges switch over a few pixels.  ``bands`` is any int >= 0; OpenCV
    caps it at ``ceil(log2(max(W, H)))``.  The weights are OpenCV's int16 ones (``weight_type=CV_16S``), so the blend
    is integer arithmetic throughout and does not depend on the layer order or the CPU; to compare with OpenCV, build
    its blender with ``cv.CV_16S``.  The default float32 weights (``cv.detail.MultiBandBlender()``) give a different
    blend, by tens of levels at some pixels, and are not what this computes.

    1 to 127 layers (128 would wrap OpenCV's int16 weight sums).  ``bands`` that is not an int, a bool or negative,
    too many layers and a canvas taller than 524 280 rows raise ``ValueError`` before any launch.  ``gains`` as for
    ``feather_blend``: the pyramids are built from the compensated bytes, the masks from the raw ones.  Inputs,
    outputs and the device rules as ``blend_layers`` (tensor crops are read in place).  No CPU fallback."""
    layers, origins, width, height, on_device, device = _check_layers("multiband_blend", layers, origins, size,
                                                                       rt.MULTIBAND_MAX_LAYERS, device)
    bands = _multiband_bands("multiband_blend", bands)
    if height > rt.MULTIBAND_MAX_HEIGHT:
        raise ValueError(f"multiband_blend: the canvas height must be <= {rt.MULTIBAND_MAX_HEIGHT}, got {height}")
    lut = None if gains is None else _gain_table("multiband_blend", gains, len(layers))
    return _blend("apap_multiband_blend", (bands,), ("apap_multiband_workspace_bytes", (bands,)), layers, origins,
                  width, height, on_device, device, lut)


def _multiband_bands(what, bands):
    """``bands`` as an int >= 0, or ``ValueError`` (a bool, a non-integer or a negative value)."""
    if isinstance(bands, (bool, np.bool_)) or not isinstance(bands, (int, np.integer)):
        raise ValueError(f"{what}: bands must be an int >= 0, got {bands!r}")
    if bands < 0:
        raise ValueError(f"{what}: bands must be >= 0, got {bands}")
    return min(int(bands), 1 << 20)                     # far above the cap of any canvas


def exposure_gains(layers, origins, size, device=None) -> np.ndarray:
    """Exposure-compensation gains of placed layers, float64 ``[n]``: what ``cv.detail.GainCompensator()`` (one feed,
    no similarity mask) returns from ``getMatGains()`` after ``feed([(0, 0)] * n, [P_k], [mask_k])``, with ``P_k``
    and ``mask_k`` as for ``feather_blend``.  Pass them as ``gains=`` to ``blend_layers``, ``feather_blend`` or
    ``multiband_blend``.

    The pass over every layer pixel runs on the GPU (``k_gain_stats``): per pair of layers the count of pixels both
    cover and, exactly, the sums of ``norm(P_i) = sqrt(b^2 + g^2 + r^2)`` over them -- the sums are the correctly
    rounded ``math.fsum`` of the norms, so the result does not depend on the schedule.  The small linear system is
    OpenCV's (``alpha = 0.01``, ``beta = 100``, layers that meet no other get gain 1), built in its loop order and
    solved with ``cv.solve`` on the host, as an OpenCV build without Eigen solves it.

    1 to 256 layers; ``layers``, ``origins``, ``size`` and the device rules as for ``blend_layers`` (tensor crops are
    read in place).  One launch and one download.  No CPU fallback."""
    stats, n = _overlap_stats("exposure_gains", "apap_gain_stats", layers, origins, size, device)
    return solve_gains(*gain_stats_ints(stats, n))


def channel_gains(layers, origins, size, device=None) -> np.ndarray:
    """Per-channel exposure-compensation gains of placed layers, float64 ``[n, 3]``: what
    ``cv.detail.ChannelsCompensator()`` returns from ``getMatGains()`` (the first three entries per layer) after
    ``feed([(0, 0)] * n, [P_k], [mask_k])``, with ``P_k`` and ``mask_k`` as for ``feather_blend``; column ``c`` belongs
    to channel ``c`` of the layers.  Pass them as ``gains=`` to ``blend_layers``, ``feather_blend`` or
    ``multiband_blend``.  Where ``exposure_gains`` evens out brightness only, these also even out a colour cast.

    OpenCV solves ``GainCompensator``'s system once per channel, with ``I_c(i, j)`` the mean of channel ``c`` of
    ``P_i`` over ``mask_i & mask_j`` (the masks and counts are ``exposure_gains``').  The per-pair channel sums are
    byte sums, counted exactly on the GPU (``k_gain_stats<true>``); below ``2^53`` they are exact in double too, so
    the result does not depend on the schedule.  ``solve_gains`` then runs once per channel.

    1 to 256 layers; ``layers``, ``origins``, ``size`` and the device rules as for ``blend_layers`` (tensor crops are
    read in place).  One launch and one download.  No CPU fallback."""
    stats, n = _overlap_stats("channel_gains", "apap_channel_stats", layers, origins, size, device)
    w = stats.view(np.uint64).reshape(4, n, n)
    count = [[int(v) for v in row] for row in w[0]]
    # solve_gains reads sums scaled by 2^52 (exposure_gains' fixed point); a byte sum below 2^53 scales exactly
    return np.stack([solve_gains(count, [[int(v) << 52 for v in row] for row in w[1 + c]]) for c in range(3)], axis=1)


def _overlap_stats(what, entry, layers, origins, size, device):
    """``(stats, n)``: the uint64 ``[4][n][n]`` words of ``entry`` (``apap_gain_stats`` or ``apap_channel_stats``) for
    placed layers checked as ``what``, as a host int64 array; one launch and one download."""
    layers, origins, width, height, on_device, device = _check_layers(what, layers, origins, size,
                                                                       rt.GAIN_MAX_LAYERS, device)
    torch, device, lib, devs, desc_p = _placed_layers(layers, origins, on_device, device)
    n = len(devs)
    nbytes = ctypes.c_size_t()
    rt.check(lib.apap_gain_stats_bytes(n, ctypes.byref(nbytes)), "apap_gain_stats_bytes")
    stats = torch.empty(nbytes.value // 8, dtype=torch.int64, device=device)
    with torch.cuda.device(device):
        rt.check(getattr(lib, entry)(desc_p, n, height, width, stats.data_ptr(), stats.numel() * 8,
                                     rt.stream_ptr(torch, device)), entry)
    return rt.to_host(torch, stats), n


def gain_stats_ints(stats, n):
    """``apap_gain_stats``' uint64 ``[4][n][n]`` as Python ints: ``(count, sums)`` with ``count[i][j]`` for ``i <= j``
    and ``sums[i][j] = word1 + word2 2^32 + word3 2^64`` (the sum of ``sqrt(q) 2^52`` over the intersection)."""
    w = np.asarray(stats).view(np.uint64).reshape(4, n, n)
    count = [[int(v) for v in row] for row in w[0]]
    sums = [[int(a) + (int(b) << 32) + (int(c) << 64) for a, b, c in zip(*rows)] for rows in zip(w[1], w[2], w[3])]
    return count, sums


def solve_gains(count, sums):
    """``GainCompensator::singleFeed``'s system from the statistics: ``N(i, j) = max(1, count)``, ``I(i, j) =
    round(sums[i][j]) 2^-52 / N(i, j)`` for pairs that meet, ``A`` and ``b`` in OpenCV's loop order over the layers
    that meet another, ``cv.solve`` (LU in double); gain 1 for the rest."""
    import cv2 as cv

    alpha, beta = 0.01, 100.0
    n = len(count)
    N = [[1] * n for _ in range(n)]
    inten = [[0.0] * n for _ in range(n)]
    skip = [True] * n
    for i in range(n):
        for j in range(i, n):
            c = count[i][j]
            N[i][j] = N[j][i] = max(1, c)
            if c == 0:
                continue
            if i != j:
                skip[i] = skip[j] = False
            inten[i][j] = float(sums[i][j]) * 2.0 ** -52 / N[i][j]
            inten[j][i] = float(sums[j][i]) * 2.0 ** -52 / N[i][j]
    keep = [i for i in range(n) if not skip[i]]
    gains = np.ones(n)
    if not keep:
        return gains
    A = np.zeros((len(keep), len(keep)))
    b = np.zeros((len(keep), 1))
    for ki, i in enumerate(keep):
        for kj, j in enumerate(keep):
            nij = float(N[i][j])
            b[ki, 0] += beta * nij
            A[ki, ki] += beta * nij
            if j != i:
                A[ki, ki] += 2 * alpha * inten[i][j] * inten[i][j] * nij
                A[ki, kj] -= 2 * alpha * inten[i][j] * inten[j][i] * nij
    _, sol = cv.solve(A, b)
    gains[keep] = sol[:, 0]
    return gains


def _gain_table(what, gains, n):
    """The gain tables of the blends' ``gains=``: ``gains`` of shape ``(n,)`` give ``uint8 [n, 256]``, row k mapping a
    byte ``v`` to ``saturate(rint(v g_k))`` in float64 (ties to even), what ``GainCompensator.apply`` gives; shape
    ``(n, 3)`` gives ``uint8 [n, 3, 256]``, row ``[k, c]`` for ``g_kc``, what ``ChannelsCompensator.apply`` gives.
    ``ValueError`` for any other shape or a value that is not finite."""
    try:
        g = np.asarray(gains, dtype=np.float64)
    except (TypeError, ValueError):
        raise ValueError(f"{what}: gains must be {n} finite numbers") from None
    if g.shape not in ((n,), (n, 3)) or not np.isfinite(g).all():
        raise ValueError(f"{what}: gains must be {n} finite numbers (one per layer) or [{n}, 3] (one per layer and "
                         f"channel), got shape {g.shape}")
    return np.clip(np.rint(np.arange(256, dtype=np.float64) * g[..., None]), 0, 255).astype(np.uint8)


def _feather_sharpness(what, sharpness):
    """``sharpness`` as the float32 OpenCV's blender keeps, or ``ValueError``: it must be finite and at least
    ``FLT_MIN``.  Below that (a subnormal), OpenCV gives a layer with no empty pixel the weight
    ``min(fl(FLT_MAX s), 1)``, which can be < 1, and the kernels give it 1."""
    with np.errstate(over="ignore"):
        s = float(np.float32(sharpness))
    if not (math.isfinite(s) and s >= np.finfo(np.float32).tiny):
        raise ValueError(f"{what}: sharpness must be finite and >= FLT_MIN (a normal float32), got {sharpness}")
    return s


def _feather_distance_cap(s, width, height):
    """``ValueError`` unless the feather kernels can store the distances of sharpness ``s`` (a checked float32) on a
    ``width x height`` canvas (``apap_feather_distance_cap``, host only)."""
    lib = rt.load_library()
    cap = ctypes.c_int()
    rc = lib.apap_feather_distance_cap(s, height, width, ctypes.byref(cap))
    if rc == rt.E_TOOBIG:
        raise ValueError(f"feather_blend: sharpness {s} needs distances beyond 16 bits on a {width} x {height} canvas "
                         "(a larger sharpness or W + H <= 65536)")
    if rc != 0:
        raise ValueError(f"feather_blend: {lib.apap_last_error().decode('utf-8', 'replace')}")


def _check_layers(what, layers, origins, size, max_layers, device):
    """The argument checks of the placed-layer functions, the three blends and ``exposure_gains`` (``ValueError``
    named after ``what``).  Returns ``(layers, origins, width, height, on_device, device)``; ``device`` is the layers'
    own for tensors."""
    layers = list(layers)
    origins = [tuple(o) for o in origins]
    if not 1 <= len(layers) <= max_layers:
        raise ValueError(f"{what}: 1 to {max_layers} layers, got {len(layers)}")
    if len(origins) != len(layers) or any(len(o) != 2 for o in origins):
        raise ValueError(f"{what}: one (x0, y0) origin per layer ({len(layers)} layers, {len(origins)} origins)")
    width, height = (int(v) for v in size)
    if width <= 0 or height <= 0:
        raise ValueError(f"{what}: the canvas size must be positive, got {tuple(size)}")
    numpy_in = [isinstance(img, np.ndarray) for img in layers]
    if any(numpy_in) and not all(numpy_in):
        raise ValueError(f"{what}: layers must be all numpy arrays or all CUDA tensors")
    on_device = not numpy_in[0]
    for k, img in enumerate(layers):
        if on_device and not getattr(img, "is_cuda", False):
            raise ValueError(f"{what}: layer {k} is neither a numpy array nor a CUDA tensor")
        if len(img.shape) != 3 or img.shape[2] != 3 or img.shape[0] < 1 or img.shape[1] < 1:
            raise ValueError(f"{what}: layer {k} must be [h, w, 3], got {tuple(img.shape)}")
        if (img.dtype != np.uint8) if not on_device else (str(img.dtype) != "torch.uint8"):
            raise ValueError(f"{what}: layer {k} must be uint8, got {img.dtype}")
    if on_device:
        devs = {img.device for img in layers}
        if len(devs) != 1:
            raise ValueError(f"{what}: all layers must be on one device, got {sorted(map(str, devs))}")
        device = layers[0].device
    return layers, origins, width, height, on_device, device


def _layer_descs(torch, device, layers, origins, on_device):
    """The layers on the device -- tensors in place when their pixels are packed (strides ``(pitch, 3, 1)``), numpy
    uploaded -- and their C ABI descriptors ``int64 [n, 6] = {address, h, w, row pitch, x0, y0}``."""
    if on_device:
        devs = [img if img.stride(2) == 1 and img.stride(1) == 3 and (img.shape[0] == 1 or img.stride(0) >= 3 * img.shape[1])
                else img.contiguous() for img in layers]
    else:
        devs = [rt.to_device(torch, device, img) for img in layers]
    desc = np.array([[img.data_ptr(), img.shape[0], img.shape[1], img.stride(0), x0, y0]
                     for img, (x0, y0) in zip(devs, origins)], dtype=np.int64)
    return devs, desc


def _placed_layers(layers, origins, on_device, device):
    """``(torch, device, lib, devs, desc_p)`` for a placed-layer call whose arguments are checked: the layers on the
    device (``_layer_descs``) and a ctypes pointer to their descriptors, which keeps the descriptor array alive."""
    torch, device = rt.torch_cuda(device)
    lib = rt.load_library()
    devs, desc = _layer_descs(torch, device, layers, origins, on_device)
    return torch, device, lib, devs, desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))


def _blend(entry, params, workspace, layers, origins, width, height, on_device, device, lut):
    """A placed-layer blend after its checks: the layers described (``_placed_layers``), the workspace (``None``: the
    blender needs none; else ``(query, its scalars)``), the canvas, and one call of ``entry`` -- or, with the gain
    table ``lut`` uploaded when it is not ``None``, of ``entry + "_gain"`` (``lut`` ``[n, 256]``) or ``entry +
    "_channels"`` (``[n, 3, 256]``).  The entries share one argument layout,
    ``(desc, n, h, w, *params, [lut], [ws, ws_bytes], out, out_bytes, stream)`` with ``params`` the blender's
    scalars (none, ``sharpness`` or ``bands``), and the workspace queries ``(desc, n, h, w, *scalars, &bytes)``.
    numpy layers in -> numpy out, tensors in -> a tensor on their device."""
    torch, device, lib, devs, desc_p = _placed_layers(layers, origins, on_device, device)
    head = (desc_p, len(devs), height, width)
    ws_args = lut_args = ()
    if workspace is not None:
        query, scalars = workspace
        ws_bytes = ctypes.c_size_t()
        rt.check(getattr(lib, query)(*head, *scalars, ctypes.byref(ws_bytes)), query)
        ws = torch.empty(max(ws_bytes.value, 16), dtype=torch.uint8, device=device)
        ws_args = (ws.data_ptr(), ws.numel())
    out = torch.empty((height, width, 3), dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        st = rt.stream_ptr(torch, device)
        if lut is not None:
            lut_dev = rt.to_device(torch, device, lut)
            entry, lut_args = entry + ("_channels" if lut.ndim == 3 else "_gain"), (lut_dev.data_ptr(),)
        rt.check(getattr(lib, entry)(*head, *params, *lut_args, *ws_args, out.data_ptr(), out.numel(), st), entry)
    return out if on_device else rt.to_host(torch, out)


# stitch_panorama's blend= names: (function, most layers, name of its one parameter, the parameter's validator)
_BLENDERS = {"mean": (blend_layers, rt.BLEND_MAX_LAYERS, None, None),
             "feather": (feather_blend, rt.FEATHER_MAX_LAYERS, "sharpness", _feather_sharpness),
             "multiband": (multiband_blend, rt.MULTIBAND_MAX_LAYERS, "bands", _multiband_bands)}


# ------------------------------------------------------------------ keypoint-pair producer (SURVEY 8f, row N3)
def match_descriptors(feats_query, feats_train, device=None):
    """Exact 1-nearest-neighbour match of every query descriptor in the train set on the GPU (``apap_match_nn``):
    ``(train_idx int32 [nq], distance float32 [nq])`` = what ``cv.BFMatcher(cv.NORM_L2).match(feats_query, feats_train)``
    returns as ``DMatch.trainIdx`` / ``.distance`` -- bit for bit for integer-valued descriptors such as SIFT's.
    The reference calls ``cv.FlannBasedMatcher().match`` (pyviz/utils.py:149-150), an approximate search whose result
    changes from run to run; the exact neighbour is what it approximates.  Arrays or CUDA tensors ``[n, dim]`` float32,
    ``dim`` even and <= 256."""
    torch, device = rt.torch_cuda(device if device is not None else (feats_query.device if hasattr(feats_query, "device") and
                                                                    not isinstance(feats_query, np.ndarray) else None))
    lib = rt.load_library()

    def dev(a):
        if isinstance(a, np.ndarray):
            return rt.to_device(torch, device, np.ascontiguousarray(a, dtype=np.float32))
        if a.dtype != torch.float32:
            raise TypeError("device descriptors must be float32 tensors")
        return a.contiguous()
    host_out = isinstance(feats_query, np.ndarray)
    q, t = dev(feats_query), dev(feats_train)
    if q.dim() != 2 or t.dim() != 2 or (t.shape[0] and q.shape[1] != t.shape[1]):
        raise ValueError("match_descriptors: descriptors are [n, dim] arrays of one dim")
    nq, nt, dim = int(q.shape[0]), int(t.shape[0]), int(q.shape[1])
    idx = torch.empty(nq, dtype=torch.int32, device=device)
    dist = torch.empty(nq, dtype=torch.float32, device=device)
    scratch = torch.empty(max(nq, 1), dtype=torch.int64, device=device)
    with torch.cuda.device(device):
        rt.check(lib.apap_match_nn(q.data_ptr(), t.data_ptr() if nt else None, nq, nt, dim, scratch.data_ptr(),
                                   idx.data_ptr(), dist.data_ptr(), rt.stream_ptr(torch, device)), "apap_match_nn")
    if host_out:
        return rt.to_host(torch, idx), rt.to_host(torch, dist)
    return idx, dist


SIFT_DIM = 128
_SIFT_TABLES = {}


def sift_sample_table(size, angle, h, w):
    """``(table float32 [n, 5], ori)`` of ``calcSIFTDescriptor`` (OpenCV 4.x) for keypoints of one ``size`` and ``angle`` on
    an ``h x w`` image: ``(i, j, rbin, cbin, weight)`` of every sample of the ``(2 radius + 1)^2`` window (row offset ``i``
    outer, column offset ``j`` inner) that passes the bin test, and ``ori = 360 - angle``.  float32 with OpenCV's operation
    order; the weight is ``exp`` of its float32 argument rounded once to float32 (OpenCV's own ``exp32f`` may differ from
    that in the last bit)."""
    f = np.float32
    size, angle = f(size), f(angle)
    ori = f(360.0) - angle
    if abs(ori - f(360.0)) < np.finfo(np.float32).eps:
        ori = f(0.0)
    hist_width = f(3.0) * (size * f(0.5))                              # SIFT_DESCR_SCL_FCTR * scl
    radius = int(np.rint(hist_width * f(1.4142135623730951) * f(5.0) * f(0.5)))   # * (d + 1) * 0.5
    radius = min(radius, int(np.sqrt(float(w) * w + float(h) * h)))
    rad = ori * f(np.pi / 180)
    cos_t = f(np.cos(np.float64(rad))) / hist_width
    sin_t = f(np.sin(np.float64(rad))) / hist_width
    i, j = np.meshgrid(np.arange(-radius, radius + 1, dtype=np.float32), np.arange(-radius, radius + 1, dtype=np.float32),
                       indexing="ij")
    i, j = i.ravel(), j.ravel()
    c_rot = j * cos_t - i * sin_t
    r_rot = j * sin_t + i * cos_t
    rbin = r_rot + f(2.0) - f(0.5)                                     # + d / 2 - 0.5f
    cbin = c_rot + f(2.0) - f(0.5)
    keep = (rbin > -1) & (rbin < 4) & (cbin > -1) & (cbin < 4)
    wgt = np.exp(((c_rot * c_rot + r_rot * r_rot) * f(-0.125)).astype(np.float64)).astype(np.float32)  # -1 / (d d 0.5)
    table = np.stack([i, j, rbin, cbin, wgt], axis=1)[keep]
    return np.ascontiguousarray(table, dtype=np.float32), ori


def _keypoint_args(points, size, angle):
    """``(xy float32 [K, 2] or tensor, size, angle)`` from an array / tensor of points or a list of ``cv.KeyPoint``."""
    if isinstance(points, (list, tuple)) and points and hasattr(points[0], "pt"):
        octaves = {int(kp.octave) for kp in points}
        if octaves != {0}:
            raise ValueError(f"sift_describe: keypoints of octave {sorted(octaves - {0})} are not supported (octave 0 only)")
        sizes, angles = {float(kp.size) for kp in points}, {float(kp.angle) for kp in points}
        if len(sizes) > 1:
            raise ValueError("sift_describe: keypoints of mixed sizes are not supported (one size per call)")
        if len(angles) > 1:
            raise ValueError("sift_describe: keypoints of mixed angles are not supported (one angle per call)")
        return np.array([kp.pt for kp in points], dtype=np.float32).reshape(-1, 2), sizes.pop(), angles.pop()
    if isinstance(points, (list, tuple)):
        points = np.asarray(points, dtype=np.float32).reshape(-1, 2)
    return points, size, angle


def sift_describe(image, points, size=1.0, angle=-1.0, device=None, equalize=False):
    """SIFT descriptors at given keypoints on the GPU: ``cv.SIFT.create().compute(image, [cv.KeyPoint(x, y, size,
    angle), ...])[1]`` (``apap_sift_describe``), ``float32 [K, 128]``, one row per point (a point with no sample inside
    the image gives zeros, as in OpenCV).  Every component is within +-2 of OpenCV 4.x's and almost all are equal.

    ``image``: ``uint8 [H, W, 3]`` BGR.  ``points``: ``[K, 2]`` (x, y), or a list of ``cv.KeyPoint`` of octave 0 sharing
    one size and one angle (which then replace ``size`` / ``angle``).  ``angle`` is -1 (the reference's keypoints) or in
    [0, 360).  numpy in -> numpy out; a CUDA tensor image -> the descriptors stay on its device.

    ``equalize=True`` describes the per-channel equalised image instead (the reference describes the output of
    ``visualize_equalized_hist``, pyviz/apap.py:234-236): bit for bit ``sift_describe(equalize_hist(image), ...)``, but the
    equalised image is never written -- the gray conversion reads the image through the equalisation LUT
    (``apap_equalize_hist`` + ``apap_sift_describe_lut``)."""
    points, size, angle = _keypoint_args(points, size, angle)
    if not (np.isfinite(size) and size > 0):
        raise ValueError(f"sift_describe: size must be finite and > 0, got {size}")
    if not (angle == -1.0 or 0.0 <= angle < 360.0):
        raise ValueError(f"sift_describe: angle {angle} is not supported (-1 or [0, 360))")
    on_device = not isinstance(image, np.ndarray)
    torch, device = rt.torch_cuda(image.device if on_device else device)
    lib = rt.load_library()
    if image.ndim != 3 or image.shape[2] != 3 or image.dtype != (np.uint8 if not on_device else torch.uint8):
        raise ValueError("sift_describe: expected a uint8 [H, W, 3] BGR image")
    img = _device_image(torch, device, image)
    h, w = int(img.shape[0]), int(img.shape[1])
    if isinstance(points, np.ndarray) or not hasattr(points, "device"):
        pts = rt.to_device(torch, device, np.asarray(points, dtype=np.float32).reshape(-1, 2))
    else:
        pts = points.to(device=device, dtype=torch.float32).reshape(-1, 2).contiguous()
    k = int(pts.shape[0])
    desc = torch.empty((k, SIFT_DIM), dtype=torch.float32, device=device)
    if k:
        key = (float(size), float(angle), h, w, device)
        if key not in _SIFT_TABLES:
            if len(_SIFT_TABLES) >= 64:
                _SIFT_TABLES.clear()
            table, ori = sift_sample_table(size, angle, h, w)
            _SIFT_TABLES[key] = (rt.to_device(torch, device, table), float(ori))
        table, ori = _SIFT_TABLES[key]
        base = torch.empty((h, w), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            st = rt.stream_ptr(torch, device)
            if equalize:
                hist = torch.empty(3 * 256, dtype=torch.int32, device=device)
                lut = torch.empty(3 * 256, dtype=torch.uint8, device=device)
                rt.check(lib.apap_equalize_hist(img.data_ptr(), h, w, hist.data_ptr(), lut.data_ptr(), None, st),
                         "apap_equalize_hist")
                rt.check(lib.apap_sift_describe_lut(img.data_ptr(), h, w, lut.data_ptr(), pts.data_ptr(), k, table.data_ptr(),
                                                    int(table.shape[0]), ori, base.data_ptr(), desc.data_ptr(), st),
                         "apap_sift_describe_lut")
            else:
                rt.check(lib.apap_sift_describe(img.data_ptr(), h, w, pts.data_ptr(), k, table.data_ptr(),
                                                int(table.shape[0]), ori, base.data_ptr(), desc.data_ptr(), st),
                         "apap_sift_describe")
    return desc if on_device else rt.to_host(torch, desc)


def equalize_hist(image, device=None):
    """``cv.merge([cv.equalizeHist(c) for c in cv.split(image)])`` on the GPU, bit for bit (``apap_equalize_hist``): the
    per-channel equalisation of the reference's ``visualize_equalized_hist`` (pyviz/utils.py:85-91).  ``image``: ``uint8
    [H, W, 3]``; numpy in -> numpy out, a CUDA tensor (any byte offset) in -> the result stays on its device."""
    on_device = not isinstance(image, np.ndarray)
    torch, device = rt.torch_cuda(image.device if on_device else device)
    lib = rt.load_library()
    if image.ndim != 3 or image.shape[2] != 3 or image.dtype != (np.uint8 if not on_device else torch.uint8):
        raise ValueError("equalize_hist: expected a uint8 [H, W, 3] image")
    img = _device_image(torch, device, image)
    h, w = int(img.shape[0]), int(img.shape[1])
    hist = torch.empty(3 * 256, dtype=torch.int32, device=device)
    lut = torch.empty(3 * 256, dtype=torch.uint8, device=device)
    out = torch.empty_like(img)
    with torch.cuda.device(device):
        rt.check(lib.apap_equalize_hist(img.data_ptr(), h, w, hist.data_ptr(), lut.data_ptr(), out.data_ptr(),
                                        rt.stream_ptr(torch, device)), "apap_equalize_hist")
    return out if on_device else rt.to_host(torch, out)


def coarse_matching(c_img, o_img, raw_kpts_cp, raw_kpts_op, device=None, describe="opencv"):
    """``coarse_matching`` of the reference (pyviz/utils.py:142-151) -- same arguments, same return tuple
    ``(kpts_cp, feats_cp, kpts_op, feats_op, matches)`` with ``matches`` a list of ``cv.DMatch`` (one per centre
    keypoint, in query order).  The matcher is the exact nearest neighbour on the GPU (``match_descriptors``) where the
    reference asks FLANN's randomised kd-trees for an approximation of it.

    ``describe`` picks the SIFT descriptors at the given keypoints:
      ``"opencv"`` (default): OpenCV's own ``cv.SIFT.compute`` on the host, the reference's exact bytes;
      ``"gpu"``: ``sift_describe`` -- each image is uploaded once, described on the device and matched there; every
      component is within +-2 of OpenCV's (almost all equal), and only the descriptors come back for the tuple."""
    import cv2 as cv

    kpts_cp = [cv.KeyPoint(*pt, 1) for pt in raw_kpts_cp]
    kpts_op = [cv.KeyPoint(*pt, 1) for pt in raw_kpts_op]
    if describe == "opencv":
        extractor = cv.SIFT.create(nfeatures=128)
        kpts_cp, feats_cp = extractor.compute(c_img, kpts_cp)
        kpts_op, feats_op = extractor.compute(o_img, kpts_op)
        idx, dist = match_descriptors(feats_cp, feats_op, device=device)
    elif describe == "gpu":
        torch, device = rt.torch_cuda(device)
        # the keypoints above are size 1, angle -1 (sift_describe's defaults) at the float32 points
        dev_cp = sift_describe(_device_image(torch, device, c_img), np.asarray(raw_kpts_cp, dtype=np.float32).reshape(-1, 2))
        dev_op = sift_describe(_device_image(torch, device, o_img), np.asarray(raw_kpts_op, dtype=np.float32).reshape(-1, 2))
        idx, dist = match_descriptors(dev_cp, dev_op, device=device)
        feats_cp, feats_op = rt.to_host(torch, dev_cp), rt.to_host(torch, dev_op)
        idx, dist = rt.to_host(torch, idx).tolist(), rt.to_host(torch, dist).tolist()
        kpts_cp, kpts_op = tuple(kpts_cp), tuple(kpts_op)
    else:
        raise ValueError(f"coarse_matching: describe must be 'opencv' or 'gpu', got {describe!r}")
    matches = [cv.DMatch(i, int(j), 0, float(d)) for i, (j, d) in enumerate(zip(idx, dist)) if j >= 0]
    return kpts_cp, feats_cp, kpts_op, feats_op, matches


RANSAC_MODEL_POINTS = 4


def _ransac_update_num_iters(p, ep, model_points, max_iters):
    """OpenCV's ``RANSACUpdateNumIters``: the iterations that reach confidence ``p`` at outlier ratio ``ep``."""
    p, ep = min(max(p, 0.0), 1.0), min(max(ep, 0.0), 1.0)
    num = max(1.0 - p, np.finfo(np.float64).tiny)
    denom = 1.0 - math.pow(1.0 - ep, model_points)
    if denom < np.finfo(np.float64).tiny:
        return 0
    num, denom = math.log(num), math.log(denom)
    return max_iters if denom >= 0 or -num >= max_iters * (-denom) else int(round(num / denom))   # cvRound


def _inliers(src, dst, H, thr_sq):
    """``computeError`` (float32, OpenCV's operation order, each step rounded on its own) ``<= thr_sq``."""
    hf = np.asarray(H, np.float64).ravel()[:8].astype(np.float32)
    x, y = src[:, 0], src[:, 1]
    with np.errstate(all="ignore"):                     # non-finite points: NaN errors, never inliers (as in OpenCV)
        ww = np.float32(1.0) / (hf[6] * x + hf[7] * y + np.float32(1.0))
        dx = (hf[0] * x + hf[1] * y + hf[2]) * ww - dst[:, 0]
        dy = (hf[3] * x + hf[4] * y + hf[5]) * ww - dst[:, 1]
        return dx * dx + dy * dy <= thr_sq


def find_homography_ransac(src, dst, threshold=5.0, *, confidence=0.995, max_iters=2000, device=None):
    """``cv.findHomography(src, dst, cv.RANSAC, threshold, maxIters=max_iters, confidence=confidence)`` with its
    hypothesis loop on the GPU (``apap_ransac_homography``): ``(H float64 [3, 3], mask uint8 [n, 1])``, or ``(None,
    zeros)`` when OpenCV finds no model.  ``src`` / ``dst``: ``[n, 2]`` numpy arrays or CUDA tensors (float32 as OpenCV
    converts them).

    One device call draws OpenCV's subsets and fits and scores every hypothesis exactly as OpenCV does (its RNG, its
    subset checks, ``runKernel`` with ``cv::eigen``'s Jacobi, the float32 error); one download brings back the subsets
    and counts.  The adaptive stop is applied to the counts here, the chosen hypothesis is OpenCV's own fit of its 4
    points (``cv.findHomography(4 points, 0)`` runs the same ``runKernel``), its inlier mask is computed in numpy
    float32 in OpenCV's order, and ``cv.findHomography(src[mask], dst[mask], 0)`` -- ``runKernel`` + LM on the
    inliers, which is what ``findHomography`` runs -- gives H; the returned mask is recomputed from that H.  H and
    mask are OpenCV's bit for bit, except when the best hypothesis has exactly 4 inliers: OpenCV then refits and
    LM-refines those 4 points, which ``findHomography(4 points, 0)`` does not, so H agrees to about 1e-12 relative
    (the mask is still OpenCV's).  Fewer than 4 points raise ``ValueError`` (OpenCV raises ``cv.error``)."""
    return find_homography_ransac_batch([src], [dst], threshold, confidence=confidence, max_iters=max_iters,
                                        device=device)[0]


def find_homography_ransac_batch(srcs, dsts, threshold=5.0, *, confidence=0.995, max_iters=2000, device=None):
    """``find_homography_ransac`` for several independent point sets: a list of ``(H, mask)``, element ``i`` bit for
    bit ``find_homography_ransac(srcs[i], dsts[i], ...)``.  ``srcs`` / ``dsts``: lists of ``[n_i, 2]`` numpy arrays or
    CUDA tensors.  Every set of 5 or more points goes to the device in one call (``apap_ransac_homography_batch``: the
    sets concatenated on the device, one sampler warp per set) and one download brings back all subsets and counts;
    sets of exactly 4 points are OpenCV's single fit; fewer than 4 raise ``ValueError`` naming the set.  The scan,
    fit, mask and refit run per set on the host.  The batch waits for its slowest sampler (see
    ``apap_ransac_homography_batch``)."""
    if len(srcs) != len(dsts):
        raise ValueError(f"find_homography_ransac_batch: {len(srcs)} source sets but {len(dsts)} target sets")
    if not srcs:
        return []
    first = next((s for s in srcs if not isinstance(s, np.ndarray) and hasattr(s, "device")), None)
    torch, device = rt.torch_cuda(first.device if first is not None else device)
    s_devs, d_devs, s_hosts, d_hosts = [], [], [], []
    for src, dst in zip(srcs, dsts):
        if not isinstance(src, np.ndarray) and hasattr(src, "device"):
            s_devs.append(src.to(device=device, dtype=torch.float32).reshape(-1, 2).contiguous())
            d_devs.append(dst.to(device=device, dtype=torch.float32).reshape(-1, 2).contiguous())
            s_hosts.append(None)
            d_hosts.append(None)
        else:
            s_hosts.append(np.ascontiguousarray(np.asarray(src, np.float32).reshape(-1, 2)))
            d_hosts.append(np.ascontiguousarray(np.asarray(dst, np.float32).reshape(-1, 2)))
            s_devs.append(None)
            d_devs.append(None)
    return _ransac(torch, device, s_devs, d_devs, s_hosts, d_hosts, threshold, confidence, max_iters)


def _ransac(torch, device, s_devs, d_devs, s_hosts, d_hosts, threshold, confidence, max_iters):
    """``find_homography_ransac_batch`` on float32 ``[n, 2]`` point sets.  Per set, the device points, the host copies,
    or both: a set without device points is uploaded when it is sampled, one without host copies is downloaded with
    the counts."""
    if not 0.0 < confidence < 1.0:
        raise ValueError(f"find_homography_ransac: confidence must be in (0, 1), got {confidence}")
    ns = []
    for i, (s_dev, d_dev, s_host, d_host) in enumerate(zip(s_devs, d_devs, s_hosts, d_hosts)):
        n, m = (int(s_host.shape[0]), int(d_host.shape[0])) if s_host is not None else (int(s_dev.shape[0]),
                                                                                         int(d_dev.shape[0]))
        if n < RANSAC_MODEL_POINTS or m != n:
            raise ValueError(f"find_homography_ransac: pair {i} needs at least 4 corresponding points, got {n} and {m}")
        ns.append(n)
    if threshold <= 0:
        threshold = 3.0                                 # OpenCV's defaultRANSACReprojThreshold
    max_iters = max(int(max_iters), 1)
    sampled = [i for i, n in enumerate(ns) if n > RANSAC_MODEL_POINTS]
    if max(len(sampled), 1) * max_iters > rt.RANSAC_MAX_ITERS:
        raise ValueError(f"find_homography_ransac: {len(sampled)} sets x max_iters {max_iters} must be <= "
                         f"{rt.RANSAC_MAX_ITERS}")
    for i in sampled:
        if s_devs[i] is None:
            s_devs[i], d_devs[i] = rt.to_device(torch, device, s_hosts[i]), rt.to_device(torch, device, d_hosts[i])
    down = []
    if sampled:
        lib = rt.load_library()
        b = len(sampled)
        ws_bytes = ctypes.c_size_t()
        rt.check(lib.apap_ransac_batch_workspace_bytes(b, max_iters, ctypes.byref(ws_bytes)),
                 "apap_ransac_batch_workspace_bytes")
        ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=device)
        out = torch.empty(b * (5 * max_iters + 1), dtype=torch.int32, device=device)   # subsets | counts | n_sampled
        hyps = torch.empty((b * max_iters, 9), dtype=torch.float64, device=device)
        cnt_ptr, ns_ptr = out.data_ptr() + 16 * b * max_iters, out.data_ptr() + 20 * b * max_iters
        with torch.cuda.device(device):
            st = rt.stream_ptr(torch, device)
            if b == 1:                                  # no offsets to upload
                i = sampled[0]
                rt.check(lib.apap_ransac_homography(s_devs[i].data_ptr(), d_devs[i].data_ptr(), ns[i], float(threshold),
                                                    max_iters, ws.data_ptr(), ws_bytes.value, out.data_ptr(),
                                                    hyps.data_ptr(), cnt_ptr, ns_ptr, st), "apap_ransac_homography")
            else:
                s_cat = torch.cat([s_devs[i] for i in sampled])
                d_cat = torch.cat([d_devs[i] for i in sampled])
                offsets = rt.to_device(torch, device, np.cumsum([0] + [ns[i] for i in sampled], dtype=np.int32))
                rt.check(lib.apap_ransac_homography_batch(s_cat.data_ptr(), d_cat.data_ptr(), offsets.data_ptr(), b,
                                                          max(ns[i] for i in sampled), float(threshold), max_iters,
                                                          ws.data_ptr(), ws_bytes.value, out.data_ptr(), hyps.data_ptr(),
                                                          cnt_ptr, ns_ptr, st), "apap_ransac_homography_batch")
        down.append(out)
    missing = [i for i, s in enumerate(s_hosts) if s is None]
    for i in missing:
        down += [s_devs[i], d_devs[i]]
    down = rt.to_host_many(torch, down)
    first = 1 if sampled else 0
    for k, i in enumerate(missing):
        s_hosts[i], d_hosts[i] = down[first + 2 * k], down[first + 2 * k + 1]
    records = [None] * len(ns)                          # None: 4 points, no sampling
    if sampled:
        b, rec = len(sampled), down[0]
        subsets = rec[:4 * b * max_iters].reshape(b, max_iters, 4)
        counts = rec[4 * b * max_iters:5 * b * max_iters].reshape(b, max_iters)
        for k, i in enumerate(sampled):
            records[i] = (subsets[k], counts[k], int(rec[5 * b * max_iters + k]))
    return [_ransac_tail(s_hosts[i], d_hosts[i], records[i], threshold, confidence, max_iters) for i in range(len(ns))]


def _ransac_tail(s_host, d_host, record, threshold, confidence, max_iters):
    """The host end of ``find_homography_ransac`` for one set: OpenCV's single fit for 4 points (``record`` None),
    else the adaptive-stop scan of the device's ``(subsets, counts, n_sampled)``, OpenCV's fit of the chosen subset,
    the mask and the refit."""
    import cv2 as cv

    n = int(s_host.shape[0])
    if record is None:                                  # findHomography: method 0 on the 4 points, mask all ones
        H = cv.findHomography(s_host, d_host, 0)[0]
        return H, (np.ones if H is not None else np.zeros)((n, 1), np.uint8)
    subsets, counts, n_sampled = record
    # RANSACPointSetRegistrator::run over the counts: a hypothesis is kept when it beats max(best, 3)
    niters, best, max_good, it = max_iters, -1, 0, 0
    while it < niters and it < n_sampled:
        good = int(counts[it])
        if good > max(max_good, RANSAC_MODEL_POINTS - 1):
            best, max_good = it, good
            niters = _ransac_update_num_iters(confidence, (n - good) / n, RANSAC_MODEL_POINTS, niters)
        it += 1
    if best < 0:
        return None, np.zeros((n, 1), np.uint8)
    thr_sq = np.float32(float(threshold) * float(threshold))
    sub = subsets[best]
    mask = _inliers(s_host, d_host, cv.findHomography(s_host[sub], d_host[sub], 0)[0], thr_sq)
    if int(mask.sum()) != max_good:                     # the device fit and counts are OpenCV's: never expected
        raise rt.ApapError(f"find_homography_ransac: hypothesis {best} has {max_good} inliers on the device but "
                           f"{int(mask.sum())} under OpenCV's fit of the same subset")
    H = cv.findHomography(s_host[mask], d_host[mask], 0)[0]
    return H, _inliers(s_host, d_host, H, thr_sq).astype(np.uint8).reshape(-1, 1)


def keypoint_pairs(center_img, other_img, raw_kpts_cp, raw_kpts_op, *, equalize=True, device=None, ransac="opencv"):
    """``(final_src, final_dst, H)`` of the reference's ``visualize_feature_pairs(center, other, swap=True)``
    (baseline_stitch_test.py:18-61, SURVEY 3.1) on arrays, without the ``.mat`` keypoint loading and the plots: what
    ``driver.stitch_pair`` takes.  Each image is uploaded once, equalised per channel (``equalize``: the reference
    describes ``visualize_equalized_hist``'s output, pyviz/apap.py:234-236) and described at ``float32(raw_kpts)``
    with size 1 and angle -1 on the device; the centre descriptors are matched against the other image's
    (``apap_match_nn``, exact nearest neighbour), and only the train indices come back.  Then, on the host:
    ``H, mask = cv.findHomography(centre, other, cv.RANSAC, 5.0)``, ``H = inv(H)`` and ``(other[mask], centre[mask],
    H)`` -- final_src are other-image points, final_dst centre-image points, and H maps other -> centre.  No
    ``cv.KeyPoint`` or ``cv.DMatch`` is built.

    ``equalize=False`` is for images that are already equalised (equalising twice is not the identity).  Fewer than 4
    matches, or no homography from RANSAC, raise ``ValueError``.

    ``ransac`` picks where the RANSAC runs: ``"opencv"`` (default) calls ``cv.findHomography`` on the host; ``"gpu"``
    gathers the matched points on the device from the train indices the matcher left there and runs
    ``find_homography_ransac`` on them -- the same ``(final_src, final_dst, H)`` bit for bit (see that function for
    the one case where its H is only within ~1e-12 of OpenCV's)."""
    import cv2 as cv

    if ransac not in ("opencv", "gpu"):
        raise ValueError(f"keypoint_pairs: ransac must be 'opencv' or 'gpu', got {ransac!r}")
    torch, device = rt.torch_cuda(device if device is not None else
                                  (center_img.device if not isinstance(center_img, np.ndarray) else None))
    raw_cp = np.asarray(raw_kpts_cp, dtype=np.float32).reshape(-1, 2)
    raw_op = np.asarray(raw_kpts_op, dtype=np.float32).reshape(-1, 2)
    pts_cp, pts_op = rt.to_device(torch, device, raw_cp), rt.to_device(torch, device, raw_op)
    feats_cp = sift_describe(_device_image(torch, device, center_img), pts_cp, equalize=equalize)
    feats_op = sift_describe(_device_image(torch, device, other_img), pts_op, equalize=equalize)
    idx_dev = match_descriptors(feats_cp, feats_op, device=device)[0]
    idx = rt.to_host(torch, idx_dev)
    q = np.flatnonzero(idx >= 0)
    if len(q) < 4:
        raise ValueError(f"keypoint_pairs: {len(q)} matches, a homography needs at least 4")
    centre, other = raw_cp[q], raw_op[idx[q]]
    if ransac == "gpu":
        q_dev = torch.nonzero(idx_dev >= 0).squeeze(1)
        h, mask = _ransac(torch, device, [pts_cp.index_select(0, q_dev)],
                          [pts_op.index_select(0, idx_dev.index_select(0, q_dev).long())], [centre], [other], 5.0,
                          0.995, 2000)[0]
    else:
        h, mask = cv.findHomography(centre, other, cv.RANSAC, 5.0)
    if h is None:
        raise ValueError("keypoint_pairs: RANSAC found no homography")
    mask = mask.ravel().astype(bool)
    return other[mask], centre[mask], np.linalg.inv(h)


def keypoint_pairs_batch(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, *, equalize=True, device=None,
                         ransac="opencv"):
    """``keypoint_pairs`` of one centre image against several others -- the reference's multi-image mode, where
    ``pyviz/apap.py`` runs once per image of a case against the fixed centre (run_all.sh:15,29): a list of
    ``(final_src, final_dst, H)``, element ``i`` bit for bit ``keypoint_pairs(center_img, other_imgs[i], kc_i,
    raw_kpts_ops[i], ...)`` in both ``ransac`` modes.  ``raw_kpts_cp`` is one ``[n, 2]`` array shared by all pairs
    (``kc_i = raw_kpts_cp``), or a list or tuple with one array per pair.

    The centre is uploaded, equalised and described once, at the concatenation of the pairs' centre keypoints
    (descriptors are per keypoint, so each pair's slice has its own call's bytes); each other image is uploaded and
    described once; the matches are launched back to back and all train indices come down in one copy.  With
    ``ransac="gpu"`` the matched points are gathered on the device and go through one ``find_homography_ransac_batch``;
    with ``"opencv"`` each pair calls ``cv.findHomography``.  A pair with fewer than 4 matches, or without a
    homography, raises ``ValueError`` naming its index."""
    return _keypoint_pairs_uploaded(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, equalize, device, ransac)[0]


def _keypoint_pairs_uploaded(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, equalize, device, ransac):
    """``keypoint_pairs_batch`` that also returns the images it uploaded: ``(pairs, centre [H, W, 3] uint8 device
    tensor, [other device tensors])``, for callers that warp them next (``driver.stitch_case``)."""
    import cv2 as cv

    if ransac not in ("opencv", "gpu"):
        raise ValueError(f"keypoint_pairs_batch: ransac must be 'opencv' or 'gpu', got {ransac!r}")
    k = len(other_imgs)
    shared = not isinstance(raw_kpts_cp, (list, tuple))
    if len(raw_kpts_ops) != k or (not shared and len(raw_kpts_cp) != k):
        raise ValueError(f"keypoint_pairs_batch: {k} other images need {k} keypoint sets, got {len(raw_kpts_ops)}"
                         + ("" if shared else f" and {len(raw_kpts_cp)} centre sets"))
    torch, device = rt.torch_cuda(device if device is not None else
                                  (center_img.device if not isinstance(center_img, np.ndarray) else None))
    if k == 0:
        return [], None, []
    raw_ops = [np.asarray(r, dtype=np.float32).reshape(-1, 2) for r in raw_kpts_ops]
    raw_cps = ([np.asarray(raw_kpts_cp, dtype=np.float32).reshape(-1, 2)] if shared else
               [np.asarray(r, dtype=np.float32).reshape(-1, 2) for r in raw_kpts_cp])
    cp_start = np.cumsum([0] + [len(r) for r in raw_cps])
    op_start = np.cumsum([0] + [len(r) for r in raw_ops])
    pts_cp = rt.to_device(torch, device, np.concatenate(raw_cps))
    pts_op = rt.to_device(torch, device, np.concatenate(raw_ops))
    centre_dev = _device_image(torch, device, center_img)
    feats_cp = sift_describe(centre_dev, pts_cp, equalize=equalize)
    other_devs = [_device_image(torch, device, img) for img in other_imgs]
    if shared:
        raw_cps, cp_start = raw_cps * k, np.zeros(k + 1, np.int64)
    idx_devs = []
    for i, img in enumerate(other_devs):
        feats_op = sift_describe(img, pts_op[op_start[i]:op_start[i + 1]], equalize=equalize)
        idx_devs.append(match_descriptors(feats_cp[cp_start[i]:cp_start[i] + len(raw_cps[i])], feats_op,
                                          device=device)[0])
    idxs = rt.to_host_many(torch, idx_devs)
    qs, centres, others = [], [], []
    for i, idx in enumerate(idxs):
        q = np.flatnonzero(idx >= 0)
        if len(q) < 4:
            raise ValueError(f"keypoint_pairs_batch: pair {i} has {len(q)} matches, a homography needs at least 4")
        qs.append(q)
        centres.append(raw_cps[i][q])
        others.append(raw_ops[i][idx[q]])
    if ransac == "gpu":
        rows = np.concatenate([np.concatenate([cp_start[i] + q, op_start[i] + idx[q]])
                               for i, (q, idx) in enumerate(zip(qs, idxs))]).astype(np.int64)
        rows = rt.to_device(torch, device, rows)        # per pair: centre rows, then other rows
        s_devs, d_devs, at = [], [], 0
        for q in qs:
            s_devs.append(pts_cp.index_select(0, rows[at:at + len(q)]))
            d_devs.append(pts_op.index_select(0, rows[at + len(q):at + 2 * len(q)]))
            at += 2 * len(q)
        fits = _ransac(torch, device, s_devs, d_devs, centres, others, 5.0, 0.995, 2000)
    else:
        fits = [cv.findHomography(c, o, cv.RANSAC, 5.0) for c, o in zip(centres, others)]
    pairs = []
    for i, ((h, mask), centre, other) in enumerate(zip(fits, centres, others)):
        if h is None:
            raise ValueError(f"keypoint_pairs_batch: RANSAC found no homography for pair {i}")
        mask = mask.ravel().astype(bool)
        pairs.append((other[mask], centre[mask], np.linalg.inv(h)))
    return pairs, centre_dev, other_devs
