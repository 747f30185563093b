"""The panorama blend of ``driver.stitch_panorama`` restated in numpy (the reference has no multi-image blend; the
contract is this project's, DESIGN.md section 3).

Layer ``k`` (``uint8 [h, w, 3]``) lies with its top-left pixel at canvas ``origins[k] = (x0, y0)``, clipped to the
canvas.  Per canvas pixel, ``n`` is the number of layers whose pixel there is non-empty (any channel > 0) and ``s``
their per-channel integer sum; the result is ``floor(s / n)``, 0 where ``n = 0``.  For two equal-size layers at one
origin this is ``apap_oracle.uniform_blend``: ``(a + b) >> 1`` where both are non-empty, the non-empty one otherwise.
"""
from __future__ import annotations

import numpy as np


def blend_layers(layers, origins, size):
    """``size = (width, height)``; returns the ``[height, width, 3]`` uint8 canvas."""
    width, height = int(size[0]), int(size[1])
    s = np.zeros((height, width, 3), dtype=np.int32)         # at most 255 x 256 per channel
    n = np.zeros((height, width), dtype=np.int32)
    for img, (x0, y0) in zip(layers, origins):
        img = np.asarray(img)
        h, w = img.shape[:2]
        x0, y0 = int(x0), int(y0)
        cx0, cy0 = max(x0, 0), max(y0, 0)                   # the layer's rectangle clipped to the canvas
        cx1, cy1 = min(x0 + w, width), min(y0 + h, height)
        if cx1 <= cx0 or cy1 <= cy0:
            continue
        part = img[cy0 - y0:cy1 - y0, cx0 - x0:cx1 - x0].astype(np.int32)
        s[cy0:cy1, cx0:cx1] += part
        n[cy0:cy1, cx0:cx1] += part.max(axis=-1) > 0
    return (s // np.maximum(n, 1)[..., None]).astype(np.uint8)
