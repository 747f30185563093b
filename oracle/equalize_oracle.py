"""numpy restatement of the per-channel histogram equalisation of the reference's ``visualize_equalized_hist``
(pyviz/utils.py:85-91): ``cv.merge([cv.equalizeHist(c) for c in cv.split(img)])``, OpenCV 4.x ``equalizeHist`` step by
step -- integer histogram, first non-zero bin ``i0``, ``dst.setTo(i0)`` when that bin holds every pixel, else
``scale = 255.f / (float)(total - hist[i0])`` and ``lut[i] = saturate_cast<uchar>((float)sum * scale)`` for ``i > i0``
with ``sum`` the running sum of ``hist[i0 + 1 .. i]``.  float32 arithmetic in that order, ``np.rint`` for ``cvRound``
(half to even).  Test infrastructure only: the package never imports it."""
from __future__ import annotations

import numpy as np


def histograms(img: np.ndarray) -> np.ndarray:
    """``int64 [3, 256]``: the histogram of every channel of a ``uint8 [H, W, 3]`` image."""
    return np.stack([np.bincount(img[..., c].ravel(), minlength=256) for c in range(3)])


def channel_lut(hist: np.ndarray) -> np.ndarray:
    """``uint8 [256]``: OpenCV's equalisation LUT of one channel's histogram (entries below the first non-zero bin,
    which no pixel reads, are 0)."""
    hist = np.asarray(hist, dtype=np.int64)
    total = int(hist.sum())
    i0 = int(np.flatnonzero(hist)[0])
    if hist[i0] == total:
        return np.full(256, i0, np.uint8)
    scale = np.float32(255.0) / np.float32(total - hist[i0])
    run = np.cumsum(hist) - np.cumsum(hist)[i0]                      # sum of hist[i0 + 1 .. i]
    v = np.rint(run.astype(np.float32) * scale)
    lut = np.clip(v, 0, 255).astype(np.uint8)
    lut[:i0 + 1] = 0
    return lut


def luts(img: np.ndarray) -> np.ndarray:
    """``uint8 [3, 256]``: the LUT of every channel (B, G, R)."""
    return np.stack([channel_lut(h) for h in histograms(img)])


def equalize(img: np.ndarray) -> np.ndarray:
    """The per-channel equalised image, ``uint8 [H, W, 3]``."""
    lut = luts(img)
    return np.stack([lut[c][img[..., c]] for c in range(3)], axis=-1)
