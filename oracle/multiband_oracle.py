"""The multi-band blend of ``utils.multiband_blend`` restated in integer numpy: ``cv.detail_MultiBandBlender(0, bands,
cv.CV_16S)`` after ``prepare((0, 0, W, H))``, ``feed(P_k.astype(int16), mask_k, (0, 0))`` for every layer and
``blend()``, converted to uint8 with saturation (DESIGN.md section 3).  ``P_k`` and ``mask_k`` are those of
``feather_oracle``; with ``gains``, ``P_k`` is pasted from the compensated bytes ``saturate(rint(v g_k))`` and
``mask_k`` from the raw ones.

  - ``nb = min(bands, ceil(log2(max(W, H))))``, ``A = 2^nb``; the pyramids live on ``Wp x Hp``, ``W`` and ``H``
    rounded up to multiples of ``A``.
  - Image level 0: ``P_k`` extended to ``Wp x Hp`` by BORDER_REFLECT (the edge pixel repeats, applied again when the
    pad is wider than the image); weight level 0: 256 on ``mask_k``, else 0, and 0 in the pad.
  - ``pyr_down``: taps ``[1 4 6 4 1]`` per axis, BORDER_REFLECT_101, ``(s + 128) >> 8``; ``pyr_up``: ``out[2j] =
    s[j-1] + 6 s[j] + s[j+1]``, ``out[2j+1] = 4 (s[j] + s[j+1])`` with ``s[-1] = s[1]``, ``s[n] = s[n-1]``, then
    ``(t + 32) >> 6``; both saturate to int16.
  - ``L_i = sat16(X_i - pyr_up(X_{i+1}))``, ``L_nb = X_nb``; ``band_i += (L_i G_i) >> 8``, ``wsum_i += G_i``;
    ``V_i = trunc((band_i << 8) / (wsum_i + 1))``; ``V_{i-1} = sat16(pyr_up(V_i) + V_{i-1})`` for ``i = nb .. 1``.
  - Output: ``V_0`` cropped to ``W x H``, 0 where ``wsum_0 <= 0``, clipped to ``[0, 255]``.

OpenCV keeps ``band`` and ``wsum`` in int16 and lets them wrap; at most 127 layers, the bound ``utils.multiband_blend``
enforces, neither can (each layer adds at most 256 to ``wsum`` and 255 / 256 of that to ``|band|``), so the sums here
are plain int32 (every value stays below 2^24).  Everything is integer arithmetic: the result does not depend on
the layer order or the CPU.
"""
from __future__ import annotations

import numpy as np

from oracle.feather_oracle import paste

MAX_LAYERS = 127


def num_bands(bands, width, height):
    """``min(bands, ceil(log(max(W, H)) / log(2)))``, as ``MultiBandBlender::prepare`` caps it."""
    return min(int(bands), (max(int(width), int(height)) - 1).bit_length())


def _sat16(a):
    return np.clip(a, -32768, 32767)


def _reflect101(idx, n):
    idx = np.abs(idx)
    return np.where(idx >= n, 2 * n - 2 - idx, idx)


def pyr_down(x):
    """``cv.pyrDown`` of an int16 ``[h, w(, c)]`` array (any size), as int32."""
    x = np.asarray(x, np.int32)
    taps = (1, 4, 6, 4, 1)
    for axis in (0, 1):
        n = x.shape[axis]
        centre = 2 * np.arange((n + 1) // 2)
        x = sum(t * np.take(x, _reflect101(centre + d, n), axis=axis) for t, d in zip(taps, range(-2, 3)))
    return _sat16((x + 128) >> 8)


def _up_axis(s, axis):
    n = s.shape[axis]
    j = np.arange(n)
    prev = np.take(s, np.where(j == 0, min(1, n - 1), j - 1), axis=axis)
    nxt = np.take(s, np.minimum(j + 1, n - 1), axis=axis)
    even = prev + 6 * s + nxt
    odd = 4 * (s + nxt)
    out = np.stack([even, odd], axis=axis + 1)
    return out.reshape(s.shape[:axis] + (2 * n,) + s.shape[axis + 1:])


def pyr_up(s):
    """``cv.pyrUp`` of an int16 ``[h, w(, c)]`` array to ``[2h, 2w(, c)]``, as int32."""
    t = _up_axis(_up_axis(np.asarray(s, np.int32), 0), 1)
    return _sat16((t + 32) >> 6)


def _reflect_pad(p, hp, wp):
    """BORDER_REFLECT of ``p`` to ``hp x wp`` on the bottom and right: period ``2 n``, the edge pixel repeated."""
    def idx(m, n):
        i = np.arange(m) % (2 * n)
        return np.where(i >= n, 2 * n - 1 - i, i)
    return p[idx(hp, p.shape[0])][:, idx(wp, p.shape[1])]


def layer_pyramids(p, mask, nb, hp, wp):
    """``(X, G)``: the int32 image pyramid ``X[0..nb]`` of ``P_k`` and weight pyramid ``G[0..nb]`` of ``mask_k``."""
    x = [_reflect_pad(np.asarray(p, np.int32), hp, wp)]
    g0 = np.zeros((hp, wp), np.int32)
    g0[:mask.shape[0], :mask.shape[1]] = np.where(mask, 256, 0)
    g = [g0]
    for _ in range(nb):
        x.append(pyr_down(x[-1]))
        g.append(pyr_down(g[-1]))
    return x, g


def padded_size(bands, width, height):
    """``(nb, Wp, Hp)``."""
    nb = num_bands(bands, width, height)
    a = 1 << nb
    return nb, -(-int(width) // a) * a, -(-int(height) // a) * a


def accumulate(layers, origins, size, bands=5, gains=None):
    """``(band, wsum)``: every level's sums over the given layers (``gains`` one float per layer or ``None``).  The
    sums of disjoint sets of layers add up to those of their union, so they may be computed in pieces."""
    nb, wp, hp = padded_size(bands, *size)
    band = [np.zeros((hp >> i, wp >> i, 3), np.int32) for i in range(nb + 1)]
    wsum = [np.zeros((hp >> i, wp >> i), np.int32) for i in range(nb + 1)]
    for k, (img, origin) in enumerate(zip(layers, origins)):
        raw = paste(img, origin, size)
        mask = raw.max(axis=-1) > 0
        p = raw
        if gains is not None:
            lut = np.clip(np.rint(np.arange(256, dtype=np.float64) * float(gains[k])), 0, 255).astype(np.uint8)
            p = lut[raw]
        x, g = layer_pyramids(p, mask, nb, hp, wp)
        for i in range(nb + 1):
            lap = x[i] if i == nb else _sat16(x[i] - pyr_up(x[i + 1]))
            band[i] += (lap * g[i][..., None]) >> 8
            wsum[i] += g[i]
    return band, wsum


def finish(band, wsum, size):
    """The uint8 canvas from all layers' ``(band, wsum)``: normalise, collapse, crop, mask and clip."""
    width, height = int(size[0]), int(size[1])
    nb = len(band) - 1
    v = [None] * (nb + 1)
    for i in range(nb + 1):
        num = band[i] << 8
        den = (wsum[i] + 1)[..., None]
        v[i] = np.sign(num) * (np.abs(num) // den)          # C division: truncation toward zero
    for i in range(nb, 0, -1):
        v[i - 1] = _sat16(pyr_up(v[i]) + v[i - 1])
    out = v[0][:height, :width]
    out = np.where((wsum[0][:height, :width] > 0)[..., None], out, 0)
    return np.clip(out, 0, 255).astype(np.uint8)


def multiband_blend(layers, origins, size, bands=5, gains=None):
    """``size = (width, height)``; returns the ``[height, width, 3]`` uint8 canvas.  ``gains``: one float per layer
    or ``None``."""
    return finish(*accumulate(layers, origins, size, bands, gains), size)
