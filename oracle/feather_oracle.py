"""The feather blend of ``utils.feather_blend`` restated in numpy: ``cv.detail.FeatherBlender(sharpness)`` after
``prepare((0, 0, W, H))``, ``feed(P_k.astype(int16), mask_k, (0, 0))`` for every layer in order and ``blend()``,
converted to uint8 (DESIGN.md section 3).

Layer ``k`` (``uint8 [h, w, 3]``) is pasted with its top-left pixel at canvas ``origins[k] = (x0, y0)`` into a zero
``H x W x 3`` canvas, clipped: ``P_k``.  ``mask_k`` is 255 where ``P_k`` is non-empty (any channel > 0).  Its weight
is ``min(D_k * s, 1)`` in float32, ``D_k`` the L1 distance to the nearest zero of ``mask_k`` (the canvas border is not
a zero; no zero at all gives ``FLT_MAX``, weight 1).  Per channel the int16 accumulator gains ``trunc(P_k * w_k)`` and
the float32 weight sum gains ``w_k``, in layer order; the result is ``trunc(acc / (wsum + 1e-5))``, 0 where
``wsum <= 1e-5``.  Where one layer alone has weight 1 this is ``v - 1`` for ``v >= 1``, as OpenCV gives it.
"""
from __future__ import annotations

import numpy as np

FLT_MAX = np.float32(np.finfo(np.float32).max)


def l1_distance(mask):
    """``cv.distanceTransform(mask, cv.DIST_L1, 3)``: float32 L1 distance of every pixel to the nearest zero of
    ``mask``, by a forward and a backward scan along the rows, then along the columns; ``FLT_MAX`` everywhere when
    ``mask`` has no zero."""
    mask = np.asarray(mask)
    h, w = mask.shape
    if (mask != 0).all():
        return np.full((h, w), FLT_MAX, np.float32)
    inf = h + w                                   # more than any distance inside the image
    d = np.ascontiguousarray(np.where(mask == 0, 0, inf).astype(np.int32).T)     # columns first, as rows
    for x in range(1, w):
        d[x] = np.minimum(d[x], d[x - 1] + 1)
    for x in range(w - 2, -1, -1):
        d[x] = np.minimum(d[x], d[x + 1] + 1)
    d = np.ascontiguousarray(d.T)
    for y in range(1, h):
        d[y] = np.minimum(d[y], d[y - 1] + 1)
    for y in range(h - 2, -1, -1):
        d[y] = np.minimum(d[y], d[y + 1] + 1)
    return d.astype(np.float32)


def paste(img, origin, size):
    """``P_k``: ``img`` with its top-left pixel at canvas ``origin = (x0, y0)`` in a zero ``size = (W, H)`` canvas."""
    width, height = int(size[0]), int(size[1])
    out = np.zeros((height, width, 3), np.uint8)
    img = np.asarray(img)
    h, w = img.shape[:2]
    x0, y0 = int(origin[0]), int(origin[1])
    cx0, cy0, cx1, cy1 = max(x0, 0), max(y0, 0), min(x0 + w, width), min(y0 + h, height)
    if cx1 > cx0 and cy1 > cy0:
        out[cy0:cy1, cx0:cx1] = img[cy0 - y0:cy1 - y0, cx0 - x0:cx1 - x0]
    return out


def feather_blend(layers, origins, size, sharpness=0.02):
    """``size = (width, height)``; returns the ``[height, width, 3]`` uint8 canvas."""
    s = np.float32(sharpness)
    width, height = int(size[0]), int(size[1])
    acc = np.zeros((height, width, 3), np.int16)
    wsum = np.zeros((height, width), np.float32)
    for img, origin in zip(layers, origins):
        p = paste(img, origin, size)
        mask = np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8)
        with np.errstate(over="ignore"):                  # FLT_MAX * s > FLT_MAX: inf, weight 1
            w = np.minimum(l1_distance(mask) * s, np.float32(1))
        acc += (p.astype(np.float32) * w[..., None]).astype(np.int16)
        wsum = wsum + w
    out = (acc.astype(np.float32) / (wsum + np.float32(1e-5))[..., None]).astype(np.int16)
    out[wsum <= np.float32(1e-5)] = 0
    return out.astype(np.uint8)
