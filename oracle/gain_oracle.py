"""Exposure compensation of ``utils.exposure_gains`` restated in numpy: ``cv.detail.GainCompensator()`` (one feed,
similarity threshold 1) fed every layer pasted into the whole canvas, as OpenCV 4.x ``GainCompensator::singleFeed``
computes it (DESIGN.md section 3), and the two panorama blends with the gains applied.

``P_k`` is layer k pasted into a zero ``H x W x 3`` canvas (clipped), ``mask_k`` its non-empty pixels (any channel
> 0).  ``N(i, j) = max(1, |mask_i & mask_j|)``; for a pair that meets (count > 0, i != j) ``I(i, j)`` is the sum of
``norm(P_i) = sqrt(b^2 + g^2 + r^2)`` over the intersection divided by ``N(i, j)``, and both images count as not
skipped.  ``A`` and ``b`` are built over the images that are not skipped in OpenCV's loop order (``alpha = 0.01``,
``beta = 100``) and solved by ``cv.solve`` (LU in double); skipped images get gain 1.

The norm sums are exact: ``sqrt(q) 2^52`` is an integer below ``2^61`` for every ``q >= 1``, so they are summed as
Python ints and rounded once -- ``math.fsum`` of the norms, bit for bit.
"""
from __future__ import annotations

import numpy as np

from oracle import feather_oracle as fo

ALPHA = 0.01
BETA = 100.0


def _pasted(layers, origins, size):
    ps = [fo.paste(img, o, size) for img, o in zip(layers, origins)]
    return ps, [p.max(axis=-1) > 0 for p in ps]


def _scaled_norms(p):
    """``sqrt(b^2 + g^2 + r^2) 2^52`` per pixel as int64 (exact integers below 2^61)."""
    q = (p.astype(np.int64) ** 2).sum(axis=-1)
    return (np.sqrt(q.astype(np.float64)) * 2.0 ** 52).astype(np.int64)


def _exact_sum(v):
    """Python-int sum of int64 values below 2^61, in 32-bit halves so that no numpy sum wraps."""
    v = v.astype(np.uint64)
    return (int((v >> np.uint64(32)).sum(dtype=np.uint64)) << 32) + int((v & np.uint64(0xFFFFFFFF)).sum(dtype=np.uint64))


def stats(layers, origins, size):
    """``(count, sums)``: ``count[i][j] = |mask_i & mask_j|`` for ``i <= j`` (0 below the diagonal) and ``sums[i][j]``
    for ``i != j`` the exact sum of ``sqrt(q) 2^52`` of ``P_i`` over that intersection, all Python ints."""
    width, height = int(size[0]), int(size[1])
    rects, norms, ms = [], [], []              # per layer: its rectangle clipped to the canvas, norms and mask there
    for img, (x0, y0) in zip(layers, origins):
        img = np.asarray(img)
        h, w = img.shape[:2]
        x0, y0 = int(x0), int(y0)
        cx0, cy0, cx1, cy1 = max(x0, 0), max(y0, 0), min(x0 + w, width), min(y0 + h, height)
        part = img[max(cy0 - y0, 0):max(cy1 - y0, 0), max(cx0 - x0, 0):max(cx1 - x0, 0)]
        rects.append((cx0, cy0, cx1, cy1))
        norms.append(_scaled_norms(part))
        ms.append(part.max(axis=-1, initial=0) > 0)
    n = len(rects)
    count = [[0] * n for _ in range(n)]
    sums = [[0] * n for _ in range(n)]
    for i in range(n):
        for j in range(i, n):
            x0, y0 = max(rects[i][0], rects[j][0]), max(rects[i][1], rects[j][1])
            x1, y1 = min(rects[i][2], rects[j][2]), min(rects[i][3], rects[j][3])
            if x1 <= x0 or y1 <= y0:
                continue                       # outside each other: nothing in common

            def crop(a, k):
                return a[y0 - rects[k][1]:y1 - rects[k][1], x0 - rects[k][0]:x1 - rects[k][0]]
            both = crop(ms[i], i) & crop(ms[j], j)
            count[i][j] = int(both.sum())
            if i != j:
                sums[i][j] = _exact_sum(crop(norms[i], i)[both])
                sums[j][i] = _exact_sum(crop(norms[j], j)[both])
    return count, sums


def gains_from_stats(count, sums):
    """OpenCV's ``A``, ``b`` and ``cv.solve`` from the exact statistics; float64 ``[n]``."""
    import cv2 as cv

    n = len(count)
    N = np.ones((n, n), np.int64)
    inten = np.zeros((n, n))
    skip = [True] * n
    for i in range(n):
        for j in range(i, n):
            c = count[i][j]
            N[i, j] = N[j, i] = max(1, c)
            if c == 0:
                continue
            if i != j:
                skip[i] = skip[j] = False
            inten[i, j] = float(sums[i][j]) * 2.0 ** -52 / int(N[i, j])
            inten[j, i] = float(sums[j][i]) * 2.0 ** -52 / int(N[i, j])
    keep = [i for i in range(n) if not skip[i]]
    gains = np.ones(n)
    if not keep:
        return gains
    m = len(keep)
    A = np.zeros((m, m))
    b = np.zeros((m, 1))
    for ki, i in enumerate(keep):
        for kj, j in enumerate(keep):
            nij = float(N[i, j])
            b[ki, 0] += BETA * nij
            A[ki, ki] += BETA * nij
            if j != i:
                A[ki, ki] += 2 * ALPHA * inten[i, j] * inten[i, j] * nij
                A[ki, kj] -= 2 * ALPHA * inten[i, j] * inten[j, i] * nij
    _, sol = cv.solve(A, b)
    gains[keep] = sol[:, 0]
    return gains


def gains(layers, origins, size):
    """What ``GainCompensator().feed([(0, 0)] * n, P, mask)`` then ``getMatGains()`` gives, float64 ``[n]``."""
    return gains_from_stats(*stats(layers, origins, size))


def apply(v, g):
    """``GainCompensator.apply`` on uint8 values: ``saturate_cast<uchar>(rint(double(v) g))``, ties to even."""
    return np.clip(np.rint(np.asarray(v, dtype=np.float64) * float(g)), 0, 255).astype(np.uint8)


def compensated(layers, origins, size, gains_):
    """``(P_k with gain k applied, mask_k of the raw P_k)`` per layer."""
    ps, ms = _pasted(layers, origins, size)
    return [apply(p, g) for p, g in zip(ps, gains_)], ms


def blend_layers(layers, origins, size, gains_):
    """The mean blend with gains: per pixel ``floor(s / n)``, ``n`` the layers non-empty there before compensation,
    ``s`` the per-channel sum of their compensated bytes; 0 where ``n = 0``."""
    width, height = int(size[0]), int(size[1])
    s = np.zeros((height, width, 3), np.int32)
    cnt = np.zeros((height, width), np.int32)
    for p, m in zip(*compensated(layers, origins, size, gains_)):
        s += p
        cnt += m
    return (s // np.maximum(cnt, 1)[..., None]).astype(np.uint8)


def feather_blend(layers, origins, size, gains_, sharpness=0.02):
    """``FeatherBlender(sharpness)`` fed the compensated ``P_k`` with the raw ``mask_k`` (``feather_oracle``'s
    arithmetic: weights from the raw masks' distances, truncated int16 terms, float32 weight sum in layer order)."""
    s = np.float32(sharpness)
    width, height = int(size[0]), int(size[1])
    acc = np.zeros((height, width, 3), np.int16)
    wsum = np.zeros((height, width), np.float32)
    for p, m in zip(*compensated(layers, origins, size, gains_)):
        with np.errstate(over="ignore"):
            w = np.minimum(fo.l1_distance(np.where(m, 255, 0).astype(np.uint8)) * s, np.float32(1))
        acc += (p.astype(np.float32) * w[..., None]).astype(np.int16)
        wsum = wsum + w
    out = (acc.astype(np.float32) / (wsum + np.float32(1e-5))[..., None]).astype(np.int16)
    out[wsum <= np.float32(1e-5)] = 0
    return out.astype(np.uint8)
