"""Per-channel exposure compensation of ``utils.channel_gains`` restated in numpy: ``cv.detail.ChannelsCompensator()``
fed every layer pasted into the whole canvas, which runs ``GainCompensator::singleFeed`` once per colour channel
(DESIGN.md section 3), and the three panorama blends with the per-channel gains applied.

``P_k``, ``mask_k`` and ``N(i, j) = max(1, |mask_i & mask_j|)`` are those of ``gain_oracle``.  For channel ``c`` and
a pair that meets, ``I_c(i, j)`` is the sum of channel ``c`` of ``P_i`` over the intersection divided by ``N(i, j)``;
the rest of the system and its solve are ``gain_oracle.gains_from_stats``.  The sums are byte sums, kept as Python
ints; ``gains_from_stats`` reads sums scaled by ``2^52``, and a sum below ``2^53`` scales exactly.

Every blend treats the channels independently, given the raw masks, so channel ``c`` of a compensated composite is
channel ``c`` of the single-gain composite with gains ``g[:, c]``: the composites below reuse ``gain_oracle``'s and
``multiband_oracle``'s that way.
"""
from __future__ import annotations

import numpy as np

from oracle import gain_oracle as go
from oracle import multiband_oracle as mo


def stats(layers, origins, size):
    """``(count, sums)``: ``count[i][j] = |mask_i & mask_j|`` for ``i <= j`` (0 below the diagonal) and
    ``sums[c][i][j]`` for ``i != j`` the sum of channel ``c`` of ``P_i`` over that intersection, all Python ints."""
    width, height = int(size[0]), int(size[1])
    rects, parts, ms = [], [], []             # per layer: its rectangle clipped to the canvas, bytes and mask there
    for img, (x0, y0) in zip(layers, origins):
        img = np.asarray(img)
        h, w = img.shape[:2]
        x0, y0 = int(x0), int(y0)
        cx0, cy0, cx1, cy1 = max(x0, 0), max(y0, 0), min(x0 + w, width), min(y0 + h, height)
        part = img[max(cy0 - y0, 0):max(cy1 - y0, 0), max(cx0 - x0, 0):max(cx1 - x0, 0)]
        rects.append((cx0, cy0, cx1, cy1))
        parts.append(part)
        ms.append(part.max(axis=-1, initial=0) > 0)
    n = len(rects)
    count = [[0] * n for _ in range(n)]
    sums = [[[0] * n for _ in range(n)] for _ in range(3)]
    for i in range(n):
        for j in range(i, n):
            x0, y0 = max(rects[i][0], rects[j][0]), max(rects[i][1], rects[j][1])
            x1, y1 = min(rects[i][2], rects[j][2]), min(rects[i][3], rects[j][3])
            if x1 <= x0 or y1 <= y0:
                continue

            def crop(a, k):
                return a[y0 - rects[k][1]:y1 - rects[k][1], x0 - rects[k][0]:x1 - rects[k][0]]
            both = crop(ms[i], i) & crop(ms[j], j)
            count[i][j] = int(both.sum())
            if i != j:
                si = crop(parts[i], i)[both].sum(axis=0, dtype=np.int64)
                sj = crop(parts[j], j)[both].sum(axis=0, dtype=np.int64)
                for c in range(3):
                    sums[c][i][j], sums[c][j][i] = int(si[c]), int(sj[c])
    return count, sums


def gains_from_stats(count, sums):
    """float64 ``[n, 3]``: ``gain_oracle.gains_from_stats`` once per channel."""
    return np.stack([go.gains_from_stats(count, [[v << 52 for v in row] for row in sums[c]]) for c in range(3)],
                    axis=1)


def gains(layers, origins, size):
    """What ``ChannelsCompensator().feed([(0, 0)] * n, P, mask)`` then ``getMatGains()`` gives, float64 ``[n, 3]``."""
    return gains_from_stats(*stats(layers, origins, size))


def apply(v, g):
    """``ChannelsCompensator.apply`` on uint8 ``[..., 3]`` values: channel ``c`` is ``saturate(rint(double(v)
    g[c]))``, ties to even."""
    v = np.asarray(v)
    return np.stack([go.apply(v[..., c], g[c]) for c in range(3)], axis=-1)


def _per_channel(blend, gains_):
    g = np.asarray(gains_, dtype=np.float64)
    return np.stack([blend(g[:, c])[..., c] for c in range(3)], axis=-1)


def blend_layers(layers, origins, size, gains_):
    """The mean blend with per-channel gains ``[n, 3]``."""
    return _per_channel(lambda g: go.blend_layers(layers, origins, size, g), gains_)


def feather_blend(layers, origins, size, gains_, sharpness=0.02):
    """``FeatherBlender(sharpness)`` fed the per-channel compensated ``P_k`` with the raw ``mask_k``."""
    return _per_channel(lambda g: go.feather_blend(layers, origins, size, g, sharpness), gains_)


def multiband_blend(layers, origins, size, gains_, bands=5):
    """``MultiBandBlender(0, bands, CV_16S)`` fed the per-channel compensated ``P_k`` with the raw ``mask_k``."""
    return _per_channel(lambda g: mo.multiband_blend(layers, origins, size, bands, gains=g), gains_)
