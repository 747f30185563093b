"""Float64 reference of the moving-DLT kernels K1 (Gram partial sums) and K2 (eigensolve + de-normalisation) --
TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``apap_oracle.local_homography_gram64`` checks the whole path from the raw points; this module checks the two
kernels one at a time, from exactly what each one reads:

  * ``partials64``: K1's ``partials[k_splits][24][cells]``, split by split, in float64 from the float32 row table and
    the float32 scaled anchors (``apap_gram_partials``).  The split ranges restate ``apap_gram_plan``.
  * ``abs_sums64`` + ``gate``: the scale ``A`` of every partial entry (the same sums over ``|w2 P_t|``) and the
    per-entry bound an FP32 kernel must meet.  The bound is ``(K + 2 ln2 T_c) 2^-24 A``.  ``K`` is the number of
    keypoints one FP32 accumulator spans before its sum leaves FP32 (the classical ``n u`` of a chain of n roundings):
    a 1024-keypoint split on FFMA2, a 256-keypoint segment on the tensor cores, whose truncating MMAs, segment drains
    and 3xTF32 split all fit inside it.  ``2 ln2 T_c`` is the relative error of ``2^-t`` when ``t`` carries a relative
    error of two float32 roundings (``T_c``: the largest ``t`` of the cell below the clamp).  On a B200 (1000 W) the
    largest ``|err| / gate`` over tests/test_gram_reference.py is 0.18 (tcgen05) and 0.17 (FFMA2); a lost 8-keypoint
    block exceeds the gate at least tenfold on every case there (checked on the CPU).
  * ``eig64``: K2 from the partial planes (``apap_eig_denorm``): float64 combine in split order, ``np.linalg.eigh``,
    ``T2inv h T1 / [2, 2]`` rounded to float32.
"""
from __future__ import annotations

import math

import numpy as np

from cvx_proj_b200.apap import expand_gram

KP_CHUNK = 128            # APAP_KP_CHUNK: keypoints per chunk of the plan
KP_BLOCK = 8              # APAP_KP_BLOCK: keypoints per k-block of the tensor-core table
SEGMENT = 256             # keypoints per tensor-core accumulation segment (kSegKb k-blocks)
CELL_PAD = 512            # cells_padded is a multiple of this
TERMS = 24
GRAM_TCGEN05, GRAM_FFMA2 = 0, 1                   # APAP_GRAM_*
SPLIT_CAP = {GRAM_TCGEN05: 16, GRAM_FFMA2: 8}     # chunks per split at most
SPLIT_DIV = 4                                     # target number of splits
K_GATE = {GRAM_TCGEN05: 256.0, GRAM_FFMA2: 1024.0}


def plan(n_kp_padded: int, engine: int):
    """``(k_splits, chunks_per_split)`` of ``apap_gram_plan``: ``cps = min(cap, ceil(n_chunks / 4))``, at least 1."""
    n_chunks = n_kp_padded // KP_CHUNK
    cps = min(SPLIT_CAP[engine], max(1, -(-n_chunks // SPLIT_DIV)))
    return max(1, -(-n_chunks // cps)), cps


def split_ranges(n_kp_padded: int, engine: int):
    """Keypoint range ``[k0, k1)`` of every split; the last one may be shorter."""
    ks, cps = plan(n_kp_padded, engine)
    step = cps * KP_CHUNK
    return [(s * step, min(n_kp_padded, (s + 1) * step)) for s in range(ks)]


def cells_padded(cells: int) -> int:
    return -(-cells // CELL_PAD) * CELL_PAD


def weights64(rows, anchors, gamma_sq, k0, k1):
    """``t`` [cells, k] = hypot(ax - kx, ay - ky) in float64 from the float32 operands, and ``w2 = max(2^-t, gamma^2)``."""
    a = np.asarray(anchors, dtype=np.float32).astype(np.float64)
    kx = rows[k0:k1, 24].astype(np.float64)
    ky = rows[k0:k1, 26].astype(np.float64)
    t = np.hypot(a[:, 0:1] - kx[None, :], a[:, 1:2] - ky[None, :])
    return t, np.maximum(np.exp2(-t), float(np.float32(gamma_sq)))


def _per_split(rows, anchors, gamma_sq, n_kp_padded, engine, absolute, cell_chunk=4096):
    rows = np.asarray(rows, dtype=np.float32)
    assert rows.shape == (n_kp_padded, 28), rows.shape
    p = rows[:, :TERMS].astype(np.float64)
    if absolute:
        p = np.abs(p)
    ranges = split_ranges(n_kp_padded, engine)
    cells = np.asarray(anchors).shape[0]
    out = np.zeros((len(ranges), TERMS, cells))
    t_max = np.zeros(cells)
    gsq = float(np.float32(gamma_sq))
    t_clamp = -math.log2(gsq) if 0.0 < gsq < 1.0 else (0.0 if gsq >= 1.0 else math.inf)
    for c0 in range(0, cells, cell_chunk):
        a = anchors[c0:c0 + cell_chunk]
        for s, (k0, k1) in enumerate(ranges):
            t, w2 = weights64(rows, a, gamma_sq, k0, k1)
            out[s, :, c0:c0 + cell_chunk] = (w2 @ p[k0:k1]).T
            if absolute:
                t_max[c0:c0 + cell_chunk] = np.maximum(t_max[c0:c0 + cell_chunk], np.minimum(t, t_clamp).max(axis=1))
    return out, t_max


def partials64(rows, anchors, gamma_sq, n_kp_padded, engine):
    """Float64 partial sums ``[k_splits, 24, cells]``: split s holds ``sum_i w2(c, i) P_t(i)`` over its keypoint range.
    ``rows``: the float32 row table ``[n_kp_padded, 28]`` of ``build_kp_table`` (24 product terms, then s kx, s kx,
    s ky, s ky); ``anchors``: float32 ``[cells, 2]`` scaled anchors; ``gamma_sq``: the float32 clamp K1 is given."""
    return _per_split(rows, anchors, gamma_sq, n_kp_padded, engine, absolute=False)[0]


def abs_sums64(rows, anchors, gamma_sq, n_kp_padded, engine):
    """``(A, T)``: ``A [k_splits, 24, cells]`` = the sums of ``|w2 P_t|`` (the scale of every partial entry) and
    ``T [cells]`` = the largest ``t`` of the cell below the clamp (``min(t, -log2 gamma^2)``)."""
    return _per_split(rows, anchors, gamma_sq, n_kp_padded, engine, absolute=True)


def gate(A, T, engine):
    """Per-entry bound on ``|K1 - partials64|``: ``(K_engine + 2 ln2 T_c) 2^-24 A_e``."""
    return (K_GATE[engine] + 2.0 * math.log(2.0) * np.asarray(T)[None, None, :]) * 2.0 ** -24 * A


def eig64(planes, tmats, dtype=np.float32):
    """K2 in float64: sum the planes ``[k_splits, 24, cells]`` in split order, expand to the 9x9 Gram matrix, take the
    eigenvector of the smallest eigenvalue and de-normalise with ``tmats`` ([18] = T2inv then T1, row-major).
    Returns ``(H [cells, 3, 3] float32, relative spectral gap (l2 - l1) / l9 [cells], Gram [cells, 9, 9])``;
    ``dtype=np.float64`` returns H before the final rounding."""
    planes = np.asarray(planes)
    total = np.zeros(planes.shape[1:])
    for s in range(planes.shape[0]):
        total += planes[s].astype(np.float64)
    g = expand_gram(total.T)
    lam, vec = np.linalg.eigh(g)
    h = vec[:, :, 0].reshape(-1, 3, 3)
    tm = np.asarray(tmats, dtype=np.float64)
    hh = tm[:9].reshape(3, 3) @ h @ tm[9:].reshape(3, 3)
    with np.errstate(all="ignore"):
        gap = (lam[:, 1] - lam[:, 0]) / lam[:, 8]
        return (hh / hh[:, 2:3, 2:3]).astype(dtype), gap, g
