"""APAP (moving-DLT local homographies + mesh warp) on B200.

Host-side mirror of the reference class ``APAP`` in ``pyviz/apap.py`` -- same constructor,
same method names, argument meaning, return layout and side effects -- over the C ABI of
``libapap_b200.so`` (``include/apap_b200.h``).  What runs where:

  host (numpy, bit-identical to the reference, O(N) or O(cells)):
      getNormalize2DPts / getConditionerFromPts / point_normalize (pyviz/apap.py:35-100),
      the cell lookup tables (pyviz/apap.py:207,209), ``np.linalg.inv`` for the few cells whose
      GPU inverse is not certified to round like numpy's (``APAP.invert_grid``)
  GPU (hand-written sm_100a kernels, no CPU fallback):
      the keypoint tables (pyviz/apap.py:103-119), K1 weights + Gram contraction, K2 9x9 eigenvector +
      de-normalisation (pyviz/apap.py:147-168), the per-cell inverse (pyviz/apap.py:201-203), K3 mesh warp
      (pyviz/apap.py:206-215), K4 uniform_blend (pyviz/apap_utils.py:75-88), local_weight (pyviz/apap.py:150-153)

Inputs and outputs are host numpy arrays by default, exactly like the reference; passing a
CUDA ``torch`` tensor as the image keeps the result on the device (opt-in).
"""
from __future__ import annotations

import math
import os
from concurrent.futures import ThreadPoolExecutor
from typing import NamedTuple

import numpy as np

from . import _runtime as rt
from ._runtime import GRAM_TERMS, HINV_ROW, KP_BLOCK, KP_BLOCK_FLOATS, KP_CHUNK, KP_ROW, WARP_BLOCK_ROWS

__all__ = ["APAP", "LazyLocalWeight", "build_kp_table", "build_kp_blocks", "scale_anchors", "weight_scale", "expand_gram", "build_warp_tables", "warp_luts", "build_row_blocks", "cell_lookup_tables"]

_U = 2.0 ** -24          # float32 unit roundoff


# ------------------------------------------------------------------------------ host helpers
def weight_scale(sigma) -> float:
    """``s = 2 log2(e) / sigma^2``: with coordinates multiplied by s, the squared moving-DLT weight
    ``max(exp(-|v - x| / sigma^2), gamma)^2`` (pyviz/apap.py:142,150-152) is ``max(2^-|s v - s x|, gamma^2)``."""
    return 2.0 * math.log2(math.e) / (float(sigma) ** 2)


def build_kp_table(src_point: np.ndarray, dlt: np.ndarray, scale: float) -> np.ndarray:
    """Keypoint table of the Gram kernel: ``[N_padded, 28]`` float32.

    Row i = the 24 distinct non-zero sums' per-keypoint terms, then the raw keypoint the weight
    is measured from, pre-scaled by ``scale`` (``weight_scale(sigma)``) and with each coordinate
    stored twice -- ``s kx, s kx, s ky, s ky`` -- the operand layout of the kernel's packed FP32
    arithmetic (112 B per row, 16-B aligned).
    With ``m = [x, y, 1]`` (conditioned source point) and ``(x', y')`` the conditioned target,
    the Gram matrix of the two DLT rows (pyviz/apap.py:106-118) is
    ``[[S, 0, -Sx], [0, S, -Sy], [-Sx, -Sy, Sr]]`` with ``S = m m^T``, ``Sx = x' m m^T``,
    ``Sy = y' m m^T``, ``Sr = (x'^2 + y'^2) m m^T``; each symmetric 3x3 block is packed as
    ``[xx, xy, x, yy, y, 1]``.  Products are formed in float64 from the reference's float32
    DLT entries and rounded once.  Rows past N are zero (they add nothing to any sum).
    """
    n = src_point.shape[0]
    a = dlt.astype(np.float64)
    x, y = a[0::2, 0], a[0::2, 1]
    xp, yp = -a[0::2, 8], -a[1::2, 8]
    m = np.stack([x * x, x * y, x, y * y, y, np.ones_like(x)], axis=1)           # [N, 6]
    n_pad = max(KP_CHUNK, (n + KP_CHUNK - 1) // KP_CHUNK * KP_CHUNK)
    tab = np.zeros((n_pad, KP_ROW), dtype=np.float32)
    tab[:n, 0:6] = m
    tab[:n, 6:12] = xp[:, None] * m
    tab[:n, 12:18] = yp[:, None] * m
    tab[:n, 18:24] = (xp * xp + yp * yp)[:, None] * m
    scaled = src_point.astype(np.float64) * scale
    tab[:n, 24:26] = scaled[:, 0:1]
    tab[:n, 26:28] = scaled[:, 1:2]
    return tab


def build_kp_blocks(table: np.ndarray) -> np.ndarray:
    """Host restatement of ``apap_kp_blocks`` (the product packs the blocks on the device, same bits --
    tests): keypoint table of the tensor-core Gram kernel from the row table of ``build_kp_table``:
    ``[N_padded / 8, 528]`` float32, one block per 8 keypoints = one K step of the TF32 MMA.

    Block layout: the 8 x 64 tile ``[Ph | Pl]`` (512 floats), then ``s kx[8], s ky[8]``.
    ``P = Ph + Pl`` exactly, ``Ph`` = P rounded to TF32 (10 mantissa bits, ties away -- the rounding of
    ``cvt.rna.tf32.f32``); the kernel computes ``w_hi [Ph | Pl] + w_lo Ph`` (3xTF32).  ``P`` is the
    8 x 32 matrix (keypoint k, term n; terms 24..31 are zero padding up to the MMA's N); the tile is
    stored in the K-major core-matrix layout of the MMA's shared-memory descriptor: element
    (k, column m) at float ``(k // 4) * 256 + (m // 8) * 32 + (m % 8) * 4 + k % 4``, ``m = n`` for
    ``Ph`` and ``32 + n`` for ``Pl``."""
    n_pad = table.shape[0]
    n_kb = n_pad // KP_BLOCK
    p = np.zeros((n_kb, KP_BLOCK, 32), dtype=np.float32)
    p[:, :, :GRAM_TERMS] = table[:, :GRAM_TERMS].reshape(n_kb, KP_BLOCK, GRAM_TERMS)
    hi = ((p.view(np.uint32) + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    lo = p - hi                                                       # exact in float32
    tile = np.concatenate([hi, lo], axis=2)                           # [kb, k, m = 64]
    out = np.empty((n_kb, KP_BLOCK_FLOATS), dtype=np.float32)
    # [kb, k = (j, kk), m = (r1, r0)] -> [kb, j, r1, r0, kk]
    out[:, :512] = tile.reshape(n_kb, 2, 4, 8, 8).transpose(0, 1, 3, 4, 2).reshape(n_kb, 512)
    out[:, 512:520] = table[:, 24].reshape(n_kb, KP_BLOCK)
    out[:, 520:528] = table[:, 26].reshape(n_kb, KP_BLOCK)
    return out


def scale_anchors(vertices, scale: float) -> np.ndarray:
    """``[..., 2]`` float64 cell anchors (``get_vertice``) -> ``[cells, 2]`` float32, pre-scaled."""
    return (np.asarray(vertices, dtype=np.float64).reshape(-1, 2) * scale).astype(np.float32)


_SYM3 = np.array([[0, 1, 2], [1, 3, 4], [2, 4, 5]])


def expand_gram(sums: np.ndarray) -> np.ndarray:
    """``[..., 24]`` packed sums -> ``[..., 9, 9]`` Gram matrix (host helper for tests)."""
    s = np.asarray(sums, dtype=np.float64)
    g = np.zeros(s.shape[:-1] + (9, 9))
    blk = lambda k: s[..., k * 6 + _SYM3]                                          # noqa: E731
    g[..., 0:3, 0:3] = blk(0)
    g[..., 3:6, 3:6] = blk(0)
    g[..., 0:3, 6:9] = -blk(1)
    g[..., 6:9, 0:3] = -blk(1)
    g[..., 3:6, 6:9] = -blk(2)
    g[..., 6:9, 3:6] = -blk(2)
    g[..., 6:9, 6:9] = blk(3)
    return g


def cell_lookup_tables(mesh: np.ndarray, final_w: int, final_h: int, grid_rows: int, grid_cols: int):
    """``(col_cell[final_w], row_cell[final_h])`` uint16: the cell the reference picks per pixel.

    ``np.where(k < edges)[0][0] - 1`` (pyviz/apap.py:207,209,210) == ``searchsorted(edges, k,
    'right') - 1``; an index of -1 wraps to the last cell like the reference's negative
    indexing; a pixel at or beyond the last edge makes the reference raise IndexError, so do we.
    """
    mesh_w, mesh_h = mesh
    if grid_rows > 65535 or grid_cols > 65535:
        raise ValueError("the warp tables hold cell indices in 16 bits: at most 65535 grid rows and columns "
                         f"(got {grid_rows} x {grid_cols})")
    out = []
    for edges, extent, ncell in ((mesh_w, final_w, grid_cols), (mesh_h, final_h, grid_rows)):
        edges = np.asarray(edges)
        idx = np.searchsorted(edges, np.arange(extent), side="right")
        if extent and idx.max(initial=0) >= edges.shape[0]:
            raise IndexError("index 0 is out of bounds for axis 0 with size 0")   # the reference's np.where(...)[0][0]
        idx = idx - 1
        if extent and (idx.max(initial=0) >= ncell):
            raise IndexError(f"index {int(idx.max())} is out of bounds for axis with size {ncell}")
        out.append(np.mod(idx, ncell).astype(np.uint16))
    return out[0], out[1]


_MAGIC_BITS = 0x4B400000        # float32 bits of 1.5 * 2**23 (kMagic of csrc/warp_blend.cu)

_POOL = None


def _map_row_chunks(fn, n_rows: int, min_rows: int = 16):
    """``fn(r0, r1)`` over contiguous chunks of ``range(n_rows)`` on a small thread pool (numpy
    releases the GIL inside its ufuncs and LAPACK calls); returns the results in order."""
    global _POOL
    workers = min(8, os.cpu_count() or 1, max(1, n_rows // min_rows))
    if workers <= 1:
        return [fn(0, n_rows)]
    if _POOL is None:
        _POOL = ThreadPoolExecutor(max_workers=8, thread_name_prefix="apap-host")
    edges = [n_rows * k // workers for k in range(workers + 1)]
    return list(_POOL.map(lambda k: fn(edges[k], edges[k + 1]), range(workers)))


def invert_grid_inplace(local_homography: np.ndarray) -> None:
    """The per-cell ``np.linalg.inv`` of ``local_warp`` (pyviz/apap.py:201-203), stored back into the
    caller's array: one stacked call = the same LAPACK routine per 3x3 block as the reference's loop
    (bit-identical, tests/test_oracle_golden.py).  Not threaded: numpy's gufunc holds the GIL here
    (measured on the GPU box: 11 ms serial vs 28 ms on the pool at 40 000 cells).  ``APAP.invert_grid`` is what
    the product calls: the GPU inverse for the cells it can certify, this routine's numpy call for the rest."""
    local_homography[...] = np.linalg.inv(local_homography)


def invert_grid_certified(grid: np.ndarray):
    """Host restatement of ``apap_invert_grid`` (tests): float64 partial-pivoting inverse of every float32 3x3 cell,
    rounded to float32, and the certificate that the rounding equals numpy's (``np.linalg.inv`` = LAPACK ``dgesv``
    on the float64 promotion + one rounding).  Both float64 results lie within ``E = c u |X| (P^T |L||U|) |X|`` of
    the exact inverse (componentwise forward error of a GEPP solve, ``c = 64`` for ``3n = 9``), so an entry ``x``
    with no float32 rounding boundary inside ``[x - 2E, x + 2E]`` rounds the same way in both.  Flagged (left to
    numpy): entries near a boundary, (near-)ties in the pivot search, zero / tiny / huge / non-finite entries,
    singular cells.  Returns ``(inverse float32 [cells, 3, 3], flags bool [cells])``."""
    a = np.asarray(grid, dtype=np.float32).reshape(-1, 3, 3).astype(np.float64)
    n = a.shape[0]
    lu = a.copy()
    perm = np.tile(np.arange(3), (n, 1))
    flag = np.zeros(n, dtype=bool)
    rows = np.arange(n)
    with np.errstate(all="ignore"):
        for k in range(2):
            col = np.abs(lu[:, k:, k])
            piv = k + np.argmax(col, axis=1)                     # first maximum, like idamax
            best = col[rows, piv - k]
            near = col >= (best * (1.0 - 1e-9))[:, None]
            flag |= near.sum(axis=1) > 1
            flag |= ~(best > 0.0) | ~np.isfinite(best)
            swap = lu[rows, piv].copy()
            lu[rows, piv] = lu[:, k]
            lu[:, k] = swap
            pk = perm[rows, piv].copy()
            perm[rows, piv] = perm[:, k]
            perm[:, k] = pk
            pivot = np.where(flag & (lu[:, k, k] == 0.0), 1.0, lu[:, k, k])
            for i in range(k + 1, 3):
                l = lu[:, i, k] / pivot
                lu[:, i, k] = l
                for j in range(k + 1, 3):
                    lu[:, i, j] -= l * lu[:, k, j]
        bad = ~(np.abs(lu[:, 2, 2]) > 0.0) | ~np.isfinite(lu[:, 2, 2])
        flag |= bad
        lu[bad, 2, 2] = 1.0
        x = np.empty((n, 3, 3))
        for j in range(3):
            b = (perm == j).astype(np.float64)
            y0 = b[:, 0]
            y1 = b[:, 1] - lu[:, 1, 0] * y0
            y2 = b[:, 2] - lu[:, 2, 0] * y0 - lu[:, 2, 1] * y1
            x2 = y2 / lu[:, 2, 2]
            x1 = (y1 - lu[:, 1, 2] * x2) / lu[:, 1, 1]
            x0 = (y0 - lu[:, 0, 1] * x1 - lu[:, 0, 2] * x2) / lu[:, 0, 0]
            x[:, 0, j], x[:, 1, j], x[:, 2, j] = x0, x1, x2
        lower = np.abs(np.tril(lu, -1)) + np.eye(3)
        upper = np.abs(np.triu(lu))
        m = lower @ upper                                         # |L||U| of P A
        w = np.empty_like(m)
        w[rows[:, None], perm] = m                                # rows back in A's order
        ax = np.abs(x)
        e = 2.0 * 64.0 * 2.0 ** -53 * (ax @ (w @ ax))
        f = x.astype(np.float32)
        lo = 0.5 * (f.astype(np.float64) + np.nextafter(f, np.float32(-np.inf)).astype(np.float64))
        hi = 0.5 * (f.astype(np.float64) + np.nextafter(f, np.float32(np.inf)).astype(np.float64))
        ok = (ax > 1e-30) & (ax < 1e30) & np.isfinite(e) & (x - e > lo) & (x + e < hi)
        flag |= ~ok.all(axis=(1, 2))
    return f, flag


def _cell_extent(lut: np.ndarray, n: int):
    """Per cell index: smallest / largest pixel coordinate mapped to it (lo > hi = unused)."""
    lo = np.full(n, np.iinfo(np.int64).max, dtype=np.int64)
    hi = np.full(n, np.iinfo(np.int64).min, dtype=np.int64)
    k = np.arange(lut.shape[0], dtype=np.int64)
    np.minimum.at(lo, lut, k)
    np.maximum.at(hi, lut, k)
    return lo, hi


def warp_luts(col_cell: np.ndarray, row_cell: np.ndarray, grid_rows: int, grid_cols: int):
    """The O(canvas edge) lookup inputs of the warp: ``(col_lut[W, 2] u32, row_first[grid_rows] i64,
    col_extent[grid_cols, 2] i32, row_extent[grid_rows, 2] i32)``.  ``col_lut[j] = (cell column, float32
    bits of dx)``, ``dx = j - (first canvas column of that cell)``; an extent is the ``{first, last}`` canvas
    column / row the reference's lookup (pyviz/apap.py:207,209) maps to the cell, ``first > last`` for
    a cell no pixel maps to.  These feed ``apap_warp_tables`` (device) and ``build_row_blocks``."""
    col64, row64 = col_cell.astype(np.int64), row_cell.astype(np.int64)
    jlo, jhi = _cell_extent(col64, grid_cols)
    ilo, ihi = _cell_extent(row64, grid_rows)
    col_used, row_used = jlo <= jhi, ilo <= ihi
    col_extent = np.stack([np.where(col_used, jlo, 1), np.where(col_used, jhi, 0)], axis=1).astype(np.int32)
    row_extent = np.stack([np.where(row_used, ilo, 1), np.where(row_used, ihi, 0)], axis=1).astype(np.int32)
    col_lut = np.empty((col_cell.shape[0], 2), dtype=np.uint32)
    col_lut[:, 0] = col_cell
    col_lut[:, 1] = (np.arange(col_cell.shape[0]) - np.where(col_used, jlo, 0)[col64]).astype(np.float32).view(np.uint32)
    return col_lut, np.where(row_used, ilo, 0), col_extent, row_extent


def build_warp_tables(inv_h: np.ndarray, col_cell: np.ndarray, row_cell: np.ndarray, off_x: int, off_y: int,
                      src_w: int, src_h: int):
    """Kernel inputs of the mesh warp: ``(cell_fast[cells, 12] f32, col_lut[W, 2] u32, row_first[grid_rows] i64)``.

    Host restatement of the device kernel ``k_warp_prep`` (``apap_warp_tables``; the product path builds
    the records there, bit-identical to this function -- tests); the CPU tests of the guard band run on it.

    ``col_lut[j] = (cell column, float32 bits of dx)`` with ``dx = j - (first canvas column of that
    cell)``; ``row_first[m]`` is the first canvas row of cell row m (``dy = i - row_first``, see
    ``build_row_blocks``).  ``cell_fast`` holds, per cell, the float32 fast path of
    ``csrc/warp_blend.cu``: with ``(x0, y0)`` the cell's first pixel minus the canvas offsets, the
    reference's ``t = H^-1 [x0 + dx, y0 + dy, 1]`` (pyviz/apap.py:211-213) is rewritten as

        t_x / t_z - qbx = (A0 dx + B0 dy + C0) / (A2 dx + B2 dy + C2)        (same for y with A1 B1 C1, qby)

    where ``(qbx, qby)`` is the integer source position of the cell centre and everything is scaled
    so the denominator is ~1.  Layout: ``A0 B0 C0 A1 | B1 C1 A2 B2 | C2, int32 bits of qbx - 0x4B400000,
    of qby - 0x4B400000, 0.5 - eps``.  ``eps`` is a rigorous bound on the absolute error of the
    kernel's float32 quotient inside the cell (coefficient rounding, two fused multiply-adds per
    numerator, ``rcp.approx`` and one multiply); a quotient farther than eps from every integer
    gets the same floor and bounds decision as the reference's float64, the kernel recomputes the
    others in float64.  ``0.5 - eps = -1`` sends the whole cell to the float64 path (denominator
    changes sign or varies too much inside the cell, coordinates beyond 2^20, non-finite entries);
    ``2`` marks a cell whose four corner pixels, and therefore all its pixels, map outside the
    source image by more than half a pixel: the kernel leaves it black without any arithmetic.
    """
    gr, gc = inv_h.shape[0], inv_h.shape[1]
    h_all = inv_h.astype(np.float64).reshape(gr, gc, 9)
    col64, row64 = col_cell.astype(np.int64), row_cell.astype(np.int64)
    jlo, jhi = _cell_extent(col64, gc)
    ilo, ihi = _cell_extent(row64, gr)
    col_used, row_used = jlo <= jhi, ilo <= ihi
    jlo, jhi = np.where(col_used, jlo, 0), np.where(col_used, jhi, 0)
    ilo, ihi = np.where(row_used, ilo, 0), np.where(row_used, ihi, 0)

    col_lut = np.empty((col_cell.shape[0], 2), dtype=np.uint32)
    col_lut[:, 0] = col_cell
    col_lut[:, 1] = (np.arange(col_cell.shape[0]) - jlo[col64]).astype(np.float32).view(np.uint32)

    def chunk(r0, r1):
        h = h_all[r0:r1]
        x0 = (jlo - off_x).astype(np.float64)[None, :]
        y0 = (ilo[r0:r1] - off_y).astype(np.float64)[:, None]
        dxm = (jhi - jlo).astype(np.float64)[None, :]
        dym = (ihi[r0:r1] - ilo[r0:r1]).astype(np.float64)[:, None]
        used = col_used[None, :] & row_used[r0:r1, None]
        with np.errstate(all="ignore"):
            t0 = h[..., 0] * x0 + h[..., 1] * y0 + h[..., 2]
            t1 = h[..., 3] * x0 + h[..., 4] * y0 + h[..., 5]
            t2 = h[..., 6] * x0 + h[..., 7] * y0 + h[..., 8]
            # integer base: the source position of the cell centre
            c0 = t0 + h[..., 0] * (0.5 * dxm) + h[..., 1] * (0.5 * dym)
            c1 = t1 + h[..., 3] * (0.5 * dxm) + h[..., 4] * (0.5 * dym)
            c2 = t2 + h[..., 6] * (0.5 * dxm) + h[..., 7] * (0.5 * dym)
            bx, by = np.rint(c0 / c2), np.rint(c1 / c2)
            ok = used & np.isfinite(bx) & np.isfinite(by) & (np.abs(bx) < 2.0 ** 30) & (np.abs(by) < 2.0 ** 30) & (c2 != 0)
            bx, by = np.where(ok, bx, 0.0), np.where(ok, by, 0.0)
            s = np.where(ok, 1.0 / np.where(ok, c2, 1.0), 0.0)
            coef = np.stack([(h[..., 0] - bx * h[..., 6]) * s, (h[..., 1] - bx * h[..., 7]) * s, (t0 - bx * t2) * s,
                             (h[..., 3] - by * h[..., 6]) * s, (h[..., 4] - by * h[..., 7]) * s, (t1 - by * t2) * s,
                             h[..., 6] * s, h[..., 7] * s, t2 * s], axis=-1)
            ok &= np.isfinite(coef).all(axis=-1)
            coef = np.where(ok[..., None], coef, 0.0).astype(np.float32).astype(np.float64)   # what the kernel sees
            m = [np.abs(coef[..., 3 * k]) * dxm + np.abs(coef[..., 3 * k + 1]) * dym + np.abs(coef[..., 3 * k + 2])
                 for k in range(3)]
            corners = np.stack([coef[..., 6] * cx + coef[..., 7] * cy + coef[..., 8]
                                for cx in (0.0 * dxm, dxm) for cy in (0.0 * dym, dym)], axis=-1)
            same_sign = (corners > 0).all(axis=-1)
            d_err = 3.0 * _U * m[2]
            d_min = corners.min(axis=-1) - d_err                     # the computed denominator is at least this
            ok &= same_sign & (d_min >= 0.25)
            d_safe = np.where(ok, d_min, 1.0)
            eps = np.zeros_like(d_safe)
            for k in (0, 1):
                q = m[k] / d_safe
                e = (3.0 * _U * m[k] + q * d_err) / d_safe + q * (2.0 ** -22 + _U)
                ok &= np.isfinite(q) & (q < 2.0 ** 20)
                eps = np.maximum(eps, np.where(np.isfinite(e), e, 1.0))
            eps = 1.25 * eps + 1e-7
            ok &= eps < 0.25
            # cells that map entirely outside the source image: tx - c and ty - c are ratios of functions affine
            # in (dx, dy) with a positive denominator, so their sign over the rectangle is decided at its corners
            cx = np.stack([cxx for cxx in (0.0 * dxm, dxm) for _ in (0, 1)], axis=-1) + 0.0 * dym[..., None]
            cy = np.stack([cyy for _ in (0, 1) for cyy in (0.0 * dym, dym)], axis=-1) + 0.0 * dxm[..., None]
            dc = np.where(ok[..., None], corners, 1.0)
            qx = (coef[..., 0:1] * cx + coef[..., 1:2] * cy + coef[..., 2:3]) / dc + bx[..., None]
            qy = (coef[..., 3:4] * cx + coef[..., 4:5] * cy + coef[..., 5:6]) / dc + by[..., None]
            outside = ok & ((qx < -0.5).all(-1) | (qx > src_w + 0.5).all(-1) | (qy < -0.5).all(-1) | (qy > src_h + 0.5).all(-1))
        rec = np.zeros((r1 - r0, gc, HINV_ROW), dtype=np.float32)
        rec[..., 0:9] = np.where(ok[..., None], coef, 0.0)
        rec[..., 8] = np.where(ok, rec[..., 8], 1.0)
        bits = rec.view(np.uint32)
        bits[..., 9] = (np.where(ok, bx, 0.0).astype(np.int64) - _MAGIC_BITS).astype(np.int32).view(np.uint32)
        bits[..., 10] = (np.where(ok, by, 0.0).astype(np.int64) - _MAGIC_BITS).astype(np.int32).view(np.uint32)
        hme = np.where(ok, 0.5 - eps, -1.0)
        hme32 = hme.astype(np.float32)
        hme32 = np.where(hme32.astype(np.float64) > hme, np.nextafter(hme32, np.float32(-2)), hme32)   # round down
        rec[..., 11] = np.where(outside, np.float32(2.0), hme32)          # 2 = "every pixel of the cell is left black"
        return rec

    rec = np.concatenate(_map_row_chunks(chunk, gr), axis=0)
    return rec.reshape(gr * gc, HINV_ROW), col_lut, ilo


def build_row_blocks(row_cell: np.ndarray, row_first: np.ndarray, row0: int = 0, row1=None,
                     max_rows: int = WARP_BLOCK_ROWS) -> np.ndarray:
    """Work list of the mesh warp for the canvas rows ``[row0, row1)``: ``uint32 [n_blocks, 2]`` =
    ``(first canvas row | rows << 28, cell row | dy of the first row << 16)``, in canvas order.

    Every maximal run of ``L`` canvas rows with the same cell row (``row_cell``, pyviz/apap.py:207) is
    covered by ``ceil(L / max_rows)`` blocks that never cross a cell row, so a lane of the kernel
    needs one cell record for all the pixels of a block.  Runs of at least ``max_rows`` rows get
    FULL blocks only: their starts are spread evenly over ``[0, L - max_rows]`` and neighbouring
    blocks overlap by a row where ``L`` is not a multiple (the overlapped rows are computed twice
    and written twice with identical bytes), which keeps the kernel's hot path free of per-row
    predicates.  ``dy`` is the first row's offset from the first canvas row of its cell row
    (``row_first``, the origin of the warp records)."""
    row1 = row_cell.shape[0] if row1 is None else row1
    rc = row_cell[row0:row1].astype(np.int64)
    if rc.size == 0:
        return np.zeros((0, 2), dtype=np.uint32)
    starts = np.flatnonzero(np.r_[True, rc[1:] != rc[:-1]])
    lens = np.diff(np.r_[starts, rc.size])
    parts = -(-lens // max_rows)                                  # blocks per run
    run = np.repeat(np.arange(starts.size), parts)                 # run index of every block
    k = np.arange(run.size) - np.repeat(np.cumsum(parts) - parts, parts)     # block index inside its run
    span = np.maximum(lens[run] - max_rows, 0)                     # last admissible start of a full block
    lo = starts[run] + (k * span + (parts[run] - 1) // 2) // np.maximum(parts[run] - 1, 1)
    rows = np.minimum(lens[run], max_rows)
    first = lo + row0
    dy = first - row_first[rc[lo]]
    if first.max(initial=0) >= 1 << 28 or dy.max(initial=0) >= 1 << 16 or dy.min(initial=0) < 0:
        raise ValueError("warp: canvas taller than 2^28 rows or a cell row spanning more than 65535 canvas rows")
    blocks = np.empty((run.size, 2), dtype=np.uint32)
    blocks[:, 0] = first | (rows << 28)
    blocks[:, 1] = rc[lo] | (dy << 16)
    return blocks


class _PinnedStage:
    """A reusable pinned host buffer for packing several small arrays into ONE host->device copy.
    The copy is asynchronous; an event guards the buffer against being refilled while in flight."""

    def __init__(self):
        self.buf = None
        self.event = None

    def upload(self, torch, device, arrays):
        """Returns one uint8 device view per array (each section starts 16-byte aligned)."""
        offs, total = [], 0
        for a in arrays:
            offs.append(total)
            total = (total + a.nbytes + 15) // 16 * 16
        if self.buf is None or self.buf.numel() < total:
            self.buf = torch.empty(max(total, 1 << 20), dtype=torch.uint8, pin_memory=True)
            self.event = None
        if self.event is not None:
            self.event.synchronize()
        host = self.buf.numpy()
        for a, off in zip(arrays, offs):
            host[off:off + a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        with torch.cuda.device(device):
            dev = self.buf[:total].to(device, non_blocking=True)
            self.event = torch.cuda.Event()
            self.event.record()
        return [dev[off:off + a.nbytes] for a, off in zip(arrays, offs)]


class WarpTables(NamedTuple):
    """Device-resident inputs of ``apap_warp`` for one inverted grid and one band of canvas rows
    (see ``build_warp_tables`` / ``build_row_blocks``): cell records, LUTs, row blocks and -- when the source rows
    are 16-byte aligned -- the tile engine's per-tile records.  They depend on the grid and the geometry, not on the
    images: build once, warp any number of images."""
    cell_fast: object       # float32 [cells * 12]
    cell_hinv: object       # float32 [cells * 9]
    col_lut: object         # int32 [canvas_w * 2]
    col_extent: object      # int32 [grid_cols * 2]
    row_blocks: object      # int32 [n_blocks * 2]
    tiles: object           # uint8: the tile engine's records (``apap_warp_tiles``), None = strip kernel only
    n_blocks: int
    row0: int               # the band of canvas rows the blocks cover
    row1: int

    def exact_cells_frac(self) -> float:
        """Share of cells whose every pixel takes the float64 path (reads the records back)."""
        rec = self.cell_fast.view(-1, HINV_ROW)[:, 11]
        return float((rec < 0).float().mean().item())


class LazyLocalWeight:
    """The second return value of ``local_homography``: ``[mesh_n, pt_size, N]`` float64 weights
    (pyviz/apap.py:144,153,169).

    The reference materialises it eagerly although its driver never reads it
    (pyviz/apap.py:242); at the benchmark configurations it is 40 MB ... 34 GB, so here it is
    computed on the GPU on first access (``np.asarray(w)``, ``w[i, j]``, ``w[i]``), slice by slice.
    """

    def __init__(self, src_point, vertices, gamma, sigma, device=None):
        self._src = np.ascontiguousarray(src_point, dtype=np.float64)      # exact promotion, as in `vertices - src_point`
        self._vert = np.ascontiguousarray(vertices, dtype=np.float64)
        self._gamma = float(gamma)
        self._inv = 1.0 / (sigma ** 2)
        self._device = device
        self.shape = (vertices.shape[0], vertices.shape[1], src_point.shape[0])
        self.dtype = np.dtype(np.float64)
        self.ndim = 3

    def __len__(self):
        return self.shape[0]

    def rows(self, r0: int, r1: int) -> np.ndarray:
        """Weights of the cell rows ``[r0, r1)`` as a host array ``[r1-r0, pt_size, N]``."""
        torch, device = rt.torch_cuda(self._device)
        lib = rt.load_library()
        p, n = self.shape[1], self.shape[2]
        out = np.empty((r1 - r0, p, n), dtype=np.float64)
        if out.size == 0:
            return out
        kp = rt.to_device(torch, device, self._src)
        per_call = max(1, min(65535 // max(p, 1), max(1, (1 << 28) // max(p * n * 8, 1))))   # <= 256 MB slices
        with torch.cuda.device(device):
            for a in range(r0, r1, per_call):
                b = min(r1, a + per_call)
                anchors = rt.to_device(torch, device, self._vert[a:b].reshape(-1, 2))
                buf = torch.empty(((b - a) * p, n), dtype=torch.float64, device=device)
                rt.check(lib.apap_local_weight(anchors.data_ptr(), kp.data_ptr(), (b - a) * p, n, self._inv,
                                               self._gamma, buf.data_ptr(), rt.stream_ptr(torch, device)),
                         "apap_local_weight")
                out[a - r0:b - r0] = rt.to_host(torch, buf).reshape(b - a, p, n)
        return out

    #: ``np.asarray(w)`` and the numpy-style operations below refuse to build more than this many bytes in one piece
    #: (c3 is 25.6 GB, the 64k-keypoint sweep 34 GB); ``w.rows(r0, r1)`` and ``w[i]`` stream any grid slice by slice.
    materialize_limit = 8 << 30

    @property
    def nbytes(self):
        return int(np.prod(self.shape, dtype=np.int64)) * 8

    @property
    def size(self):
        return int(np.prod(self.shape, dtype=np.int64))

    def __array__(self, dtype=None, copy=None):
        if self.nbytes > self.materialize_limit:
            raise MemoryError(f"local_weight is {self.nbytes / 2**30:.1f} GiB as one array (limit "
                              f"{self.materialize_limit / 2**30:.0f} GiB, LazyLocalWeight.materialize_limit): "
                              "read it by cell rows with .rows(r0, r1) or w[i]")
        full = self.rows(0, self.shape[0])
        return full if dtype is None else full.astype(dtype, copy=False)

    # what a reference user does with the ndarray works here too: arithmetic, comparisons and numpy functions build
    # the array once (under the limit above) and hand over to numpy
    def __array_ufunc__(self, ufunc, method, *inputs, **kwargs):
        args = [np.asarray(a) if isinstance(a, LazyLocalWeight) else a for a in inputs]
        return getattr(ufunc, method)(*args, **kwargs)

    def __array_function__(self, func, types, args, kwargs):
        def conv(a):
            if isinstance(a, LazyLocalWeight):
                return np.asarray(a)
            if isinstance(a, (list, tuple)):
                return type(a)(conv(v) for v in a)
            return a
        return func(*conv(args), **{k: conv(v) for k, v in kwargs.items()})

    def sum(self, *a, **k):
        return np.asarray(self).sum(*a, **k)

    def mean(self, *a, **k):
        return np.asarray(self).mean(*a, **k)

    def min(self, *a, **k):
        return np.asarray(self).min(*a, **k)

    def max(self, *a, **k):
        return np.asarray(self).max(*a, **k)

    def astype(self, dtype, **k):
        return np.asarray(self).astype(dtype, **k)

    def copy(self):
        return np.asarray(self).copy()

    def __mul__(self, o): return np.multiply(self, o)
    def __rmul__(self, o): return np.multiply(o, self)
    def __add__(self, o): return np.add(self, o)
    def __radd__(self, o): return np.add(o, self)
    def __sub__(self, o): return np.subtract(self, o)
    def __rsub__(self, o): return np.subtract(o, self)
    def __truediv__(self, o): return np.true_divide(self, o)
    def __rtruediv__(self, o): return np.true_divide(o, self)
    def __pow__(self, o): return np.power(self, o)
    def __neg__(self): return np.negative(self)
    def __lt__(self, o): return np.less(self, o)
    def __le__(self, o): return np.less_equal(self, o)
    def __gt__(self, o): return np.greater(self, o)
    def __ge__(self, o): return np.greater_equal(self, o)
    def __eq__(self, o): return np.equal(self, o)
    def __ne__(self, o): return np.not_equal(self, o)
    __hash__ = None

    def __getitem__(self, key):
        if isinstance(key, tuple) and len(key) >= 1 and isinstance(key[0], (int, np.integer)):
            i = int(key[0]) % self.shape[0]
            return self.rows(i, i + 1)[0][key[1:]] if len(key) > 1 else self.rows(i, i + 1)[0]
        if isinstance(key, (int, np.integer)):
            i = int(key) % self.shape[0]
            return self.rows(i, i + 1)[0]
        if isinstance(key, slice):
            r0, r1, step = key.indices(self.shape[0])
            if step == 1:
                return self.rows(r0, r1)
        return np.asarray(self)[key]


# ------------------------------------------------------------------------------------ the class
class APAP:
    """Drop-in for the reference ``APAP`` (pyviz/apap.py:21-217)."""

    def __init__(self, gamma, sigma, final_size, offset, device=None, gram_engine="tcgen05"):
        """``final_size = [width, height]`` of the stitched canvas, ``offset = [off_x, off_y]``
        (pyviz/apap.py:22-32).  Extensions: ``device`` selects the CUDA device; ``gram_engine`` the
        kernel of the moving-DLT contraction, ``"tcgen05"`` (tensor cores, 3xTF32, default) or
        ``"ffma2"`` (FP32 SIMT)."""
        if gram_engine not in ("tcgen05", "ffma2"):
            raise ValueError("gram_engine must be 'tcgen05' or 'ffma2'")
        self.gram_engine = gram_engine
        self.gamma = gamma
        self.sigma = sigma
        self.final_width, self.final_height = final_size
        self.offset_x, self.offset_y = offset
        self.device = device
        self._lut_cache = {}

    # ---- O(N) host pieces, numerically identical to the reference ------------------------------
    @staticmethod
    def getNormalize2DPts(point):
        """Hartley normaliser: centroid to the origin, mean distance sqrt(2).
        Returns ``(t[3,3] float32, normalised points [N,2])`` (pyviz/apap.py:35-59)."""
        count = point.shape[0]
        centre = np.mean(point, axis=0)
        shifted = point - centre
        mean_dist = np.mean(np.sqrt(np.sum(np.square(shifted), axis=1)))
        scale = np.sqrt(2) / (mean_dist + 1e-8)
        t = np.array([[scale, 0, -scale * centre[0]],
                      [0, scale, -scale * centre[1]],
                      [0, 0, 1]], dtype=np.float32)
        homog = np.column_stack((np.array(point, copy=True), np.ones(count, dtype=np.float32)))
        return t, t.dot(homog.T).T[:, :2]

    @staticmethod
    def getConditionerFromPts(point):
        """Per-axis conditioner from the unbiased standard deviation (pyviz/apap.py:63-89)."""
        count = point.shape[0]
        mu_x, mu_y = np.mean(point, axis=0)
        dev = np.std(point, axis=0)
        dev = np.sqrt(dev * dev * count / (count - 1))
        dev_x, dev_y = dev
        dev_x = dev_x + (dev_x == 0)
        dev_y = dev_y + (dev_y == 0)
        kx = np.sqrt(2) / dev_x
        ky = np.sqrt(2) / dev_y
        return np.array([[kx, 0, (-kx * mu_x)],
                         [0, ky, (-ky * mu_y)],
                         [0, 0, 1]], dtype=np.float32)

    @staticmethod
    def point_normalize(nf, c):
        """``cf = nf * diag(c) + translation(c)`` in float32 (pyviz/apap.py:92-100), vectorised;
        element-wise multiply-then-add is the same two roundings as the reference's loop."""
        cf = np.zeros_like(nf)
        cf[:, 0] = nf[:, 0] * c[0, 0] + c[0, 2]
        cf[:, 1] = nf[:, 1] * c[1, 1] + c[1, 2]
        return cf

    @staticmethod
    def matrix_generate(sample_n, cf1, cf2):
        """The ``[2N, 9]`` float32 DLT matrix (pyviz/apap.py:103-119), vectorised."""
        dlt = np.zeros([sample_n * 2, 9], dtype=np.float32)
        even, odd = dlt[0::2], dlt[1::2]
        even[:, 0:2] = cf1[:sample_n]
        even[:, 2] = 1
        even[:, 6] = (-cf2[:sample_n, 0]) * cf1[:sample_n, 0]
        even[:, 7] = (-cf2[:sample_n, 0]) * cf1[:sample_n, 1]
        even[:, 8] = -cf2[:sample_n, 0]
        odd[:, 3:5] = cf1[:sample_n]
        odd[:, 5] = 1
        odd[:, 6] = (-cf2[:sample_n, 1]) * cf1[:sample_n, 0]
        odd[:, 7] = (-cf2[:sample_n, 1]) * cf1[:sample_n, 1]
        odd[:, 8] = -cf2[:sample_n, 1]
        return dlt

    @staticmethod
    def warp_coordinate_estimate(pt, homography):
        """``homography @ pt`` divided by its third component (pyviz/apap.py:172-184)."""
        target = homography @ pt
        target /= target[2]
        return target

    # ---- moving DLT ----------------------------------------------------------------------------
    def _condition(self, src_point, dst_point):
        """The O(N) host prologue of ``local_homography`` (pyviz/apap.py:129-141): normalise and condition
        both point sets with the reference's own numpy calls (their float32 reductions and the BLAS product
        are kept on the host so every bit matches).  Returns the conditioned points ``cf1, cf2``
        (``[N, 2]`` float32) and the two 3x3 de-normalisation matrices packed as ``[18]`` float64."""
        src_point = np.asarray(src_point)
        dst_point = np.asarray(dst_point)
        n1, nf1 = self.getNormalize2DPts(src_point)
        n2, nf2 = self.getNormalize2DPts(dst_point)
        c1 = self.getConditionerFromPts(nf1)
        c2 = self.getConditionerFromPts(nf2)
        cf1 = self.point_normalize(nf1, c1)
        cf2 = self.point_normalize(nf2, c2)
        # h -> inv(N2) (inv(C2) h C1) N1   (pyviz/apap.py:165-166); inverses in float32 like the reference
        t2inv = np.linalg.inv(n2).astype(np.float64) @ np.linalg.inv(c2).astype(np.float64)
        t1 = c1.astype(np.float64) @ n1.astype(np.float64)
        tmats = np.concatenate([t2inv.reshape(9), t1.reshape(9)])
        return cf1, cf2, tmats

    def _prepare(self, src_point, dst_point):
        """Host restatement of the device table build (tests, tools): ``_condition``, the DLT matrix
        (pyviz/apap.py:143-145) and the keypoint ROW table (``build_kp_table``).  The product path builds the
        same rows on the device (``kp_rows_device``) from the conditioned points."""
        src_point = np.asarray(src_point)
        cf1, cf2, tmats = self._condition(src_point, dst_point)
        dlt = self.matrix_generate(src_point.shape[0], cf1, cf2)
        table = build_kp_table(src_point.astype(np.float32, copy=False), dlt, weight_scale(self.sigma))
        return table, tmats

    def weight_bound_device(self, raw_src_dev, counts_dev, anchors_dev):
        """``apap_weight_bound``: per scene an upper bound of the pre-scaled distance of pyviz/apap.py:150-151 over all
        (cell, match) pairs -- K1 leaves the clamp of :152 out for a scene where it cannot trigger (same bits).
        ``raw_src_dev`` float32 ``[batch, n, 2]``, ``anchors_dev`` float32 ``[batch, cells, 2]`` (pre-scaled)."""
        torch, device = rt.torch_cuda(raw_src_dev.device)
        lib = rt.load_library()
        batch, n, _ = raw_src_dev.shape
        bound = torch.empty(batch, dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            rt.check(lib.apap_weight_bound(raw_src_dev.data_ptr(), counts_dev.data_ptr() if counts_dev is not None else None,
                                           batch, n, weight_scale(self.sigma), anchors_dev.data_ptr(),
                                           int(anchors_dev.shape[1]), bound.data_ptr(), rt.stream_ptr(torch, device)),
                     "apap_weight_bound")
        return bound

    def condition_device(self, raw_dev, counts_dev=None):
        """``apap_condition``: the normalisers, conditioners and conditioned points of pyviz/apap.py:129-141 on the device.
        ``raw_dev`` float32 ``[2, batch, n, 2]`` (source points, target points).  Returns ``(cond [2, batch, n, 2]
        float32, tmats [batch, 18] float64)``; float64 reductions in a fixed order instead of numpy's float32 pairwise
        sums, so H agrees with the host path (``_condition``) to ~1e-6 of the gate, not bit for bit."""
        torch, device = rt.torch_cuda(raw_dev.device)
        lib = rt.load_library()
        _, batch, n, _ = raw_dev.shape
        cond = torch.empty((2, batch, n, 2), dtype=torch.float32, device=device)
        mats = torch.empty((batch, 36), dtype=torch.float32, device=device)
        tmats = torch.empty((batch, 18), dtype=torch.float64, device=device)
        with torch.cuda.device(device):
            rt.check(lib.apap_condition(raw_dev[0].data_ptr(), raw_dev[1].data_ptr(),
                                        counts_dev.data_ptr() if counts_dev is not None else None, batch, n,
                                        cond.data_ptr(), mats.data_ptr(), tmats.data_ptr(), rt.stream_ptr(torch, device)),
                     "apap_condition")
        return cond, tmats

    def kp_rows_device(self, points_dev, counts_dev=None):
        """Keypoint ROW table ``[batch, n_pad, 28]`` built on the device by ``apap_kp_rows`` (same bits as
        ``build_kp_table``) from ``points_dev`` = float32 ``[3, batch, n, 2]`` (or a tuple of three ``[batch, n, 2]``
        tensors): conditioned source points, conditioned target points, raw source points; ``counts_dev`` int32
        ``[batch]`` = matches per scene."""
        cf1, cf2, raw = points_dev[0], points_dev[1], points_dev[2]
        torch, device = rt.torch_cuda(cf1.device)
        lib = rt.load_library()
        batch, n, _ = cf1.shape
        n_pad = max(KP_CHUNK, (n + KP_CHUNK - 1) // KP_CHUNK * KP_CHUNK)
        rows = torch.empty((batch, n_pad, KP_ROW), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            rt.check(lib.apap_kp_rows(cf1.data_ptr(), cf2.data_ptr(), raw.data_ptr(),
                                      counts_dev.data_ptr() if counts_dev is not None else None, batch, n, n_pad,
                                      weight_scale(self.sigma), rows.data_ptr(), rt.stream_ptr(torch, device)),
                     "apap_kp_rows")
        return rows

    def kp_table_device(self, rows_dev):
        """Device keypoint table of this instance's Gram engine from the uploaded row table
        ``[batch, n_pad, 28]``: the rows themselves (``ffma2``) or the block table ``[batch, n_pad / 8, 528]``
        packed by ``apap_kp_blocks`` (``tcgen05``; same bits as ``build_kp_blocks``)."""
        if self.gram_engine != "tcgen05":
            return rows_dev
        torch, device = rt.torch_cuda(rows_dev.device)
        lib = rt.load_library()
        batch, n_pad, _ = rows_dev.shape
        blocks = torch.empty((batch, n_pad // KP_BLOCK, KP_BLOCK_FLOATS), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            rt.check(lib.apap_kp_blocks(rows_dev.data_ptr(), batch, n_pad, blocks.data_ptr(),
                                        rt.stream_ptr(torch, device)), "apap_kp_blocks")
        return blocks

    def _tile_counters(self, torch, device, batch, cells):
        """Zeroed int32 scratch ``[batch, ceil(cells / 128)]`` for the overlapped K1 -> K2 launch (the library
        leaves it zero after every completed call, so it is allocated and cleared once per shape)."""
        key = (str(device), batch, (cells + 127) // 128)
        hit = getattr(self, "_counters", None)
        if hit is None or hit[0] != key:
            hit = (key, torch.zeros((batch, (cells + 127) // 128), dtype=torch.int32, device=device))
            self._counters = hit
        return hit[1]

    def local_homography_device(self, table_dev, anchors_dev, tmats_dev, batch, cells, out_h=None, partials=None,
                                sweeps=None, solver=rt.EIG_AUTO, overlap=True, t_bound=None):
        """Device-resident K1 + K2 (no host traffic): tensors in, ``[batch, cells, 9]`` float32 out.
        ``table_dev`` / ``anchors_dev`` hold pre-scaled coordinates (``build_kp_table`` or, for the
        tensor-core engine, ``build_kp_blocks``; ``scale_anchors``); the engine follows from the table's shape.
        ``overlap``: launch K2 as a programmatic dependent of K1 (it starts on finished cell tiles while K1's last
        CTAs are still running); same results either way.  ``t_bound``: float32 ``[batch]`` from ``weight_bound_device``
        (K1 skips the clamp where it cannot trigger; same results)."""
        torch, device = rt.torch_cuda(table_dev.device)
        lib = rt.load_library()
        engine = rt.GRAM_TCGEN05 if table_dev.shape[-1] == KP_BLOCK_FLOATS else rt.GRAM_FFMA2
        n_pad = table_dev.shape[-2] * (KP_BLOCK if engine == rt.GRAM_TCGEN05 else 1)
        _, _, nbytes = rt.gram_plan(cells, n_pad, engine)
        if partials is None:
            partials = torch.empty(batch * nbytes // 4, dtype=torch.float32, device=device)
        if out_h is None:
            out_h = torch.empty((batch, cells, 9), dtype=torch.float32, device=device)
        counters = (self._tile_counters(torch, device, batch, cells)
                    if overlap and engine == rt.GRAM_TCGEN05 else None)
        try:
            with torch.cuda.device(device):
                rt.check(lib.apap_local_homography(
                    table_dev.data_ptr(), anchors_dev.data_ptr(), tmats_dev.data_ptr(), batch, cells, n_pad,
                    float(np.float32(float(self.gamma) ** 2)), engine, int(solver),
                    t_bound.data_ptr() if t_bound is not None else None, partials.data_ptr(),
                    counters.data_ptr() if counters is not None else None, out_h.data_ptr(),
                    sweeps.data_ptr() if sweeps is not None else None, rt.stream_ptr(torch, device)),
                    "apap_local_homography")
        except Exception:
            self._counters = None          # a failed call may leave counts behind: never reuse that scratch
            raise
        return out_h

    def local_homography(self, src_point, dst_point, vertices):
        """Local homography per mesh cell (pyviz/apap.py:121-169).

        ``src_point``, ``dst_point``: ``[N, 2]``; ``vertices``: ``[mesh_n, pt_size, 2]`` (x, y).
        Returns ``(H[mesh_n, pt_size, 3, 3] float32, local_weight[mesh_n, pt_size, N] float64)``;
        the weights are a lazy array (see ``LazyLocalWeight``).
        """
        sample_n, _ = np.shape(src_point)
        mesh_n, pt_size, _ = np.shape(vertices)
        if sample_n == 0:
            raise ValueError("local_homography needs at least one match")
        points = np.empty((2, 1, sample_n, 2), dtype=np.float32)
        points[0, 0], points[1, 0] = src_point, dst_point
        verts = np.ascontiguousarray(vertices, dtype=np.float64).reshape(1, mesh_n * pt_size, 2)
        h = self._homography_pass(points, None, verts).reshape(mesh_n, pt_size, 3, 3)
        weight = LazyLocalWeight(np.asarray(src_point), np.asarray(vertices), self.gamma, self.sigma, self.device)
        return h, weight

    def _homography_pass(self, points, counts, verts):
        """Raw inputs up, ONE library call (``apap_local_homography_points``: anchors, conditioning, keypoint table,
        clamp bound, K1, K2), H down.  ``points`` float32 ``[2, b, n, 2]`` (source, target), ``counts`` int32 ``[b]`` or
        None, ``verts`` float64 ``[b, cells, 2]``.  Returns H ``[b, cells, 9]`` float32 (host).  The device scratch is
        kept per shape; big inputs that already sit in pinned memory go up without the staging copy."""
        torch, device = rt.torch_cuda(self.device)
        lib = rt.load_library()
        _, batch, n, _ = points.shape
        cells = verts.shape[1]
        engine = rt.GRAM_TCGEN05 if self.gram_engine == "tcgen05" else rt.GRAM_FFMA2
        key = (str(device), batch, n, cells, engine)
        ws = getattr(self, "_pass_ws", None)
        if ws is None or ws[0] != key:
            import ctypes
            need = ctypes.c_size_t()
            rt.check(lib.apap_pass_workspace_bytes(batch, n, cells, engine, ctypes.byref(need)), "apap_pass_workspace_bytes")
            ws = (key, torch.empty(int(need.value), dtype=torch.uint8, device=device))
            self._pass_ws = ws
        if not hasattr(self, "_stage"):
            self._stage = _PinnedStage()
        small = [points] + ([counts] if counts is not None else [])
        v_t = torch.from_numpy(verts)
        if v_t.is_pinned():                              # no staging copy for what is already pinned
            parts = self._stage.upload(torch, device, small)
            v_dev = v_t.to(device, non_blocking=True)
        else:
            parts = self._stage.upload(torch, device, small + [verts])
            v_dev = parts[-1]
        p_dev = parts[0]
        c_dev = parts[1] if counts is not None else None
        out_h = torch.empty((batch, cells, 9), dtype=torch.float32, device=device)
        counters = self._tile_counters(torch, device, batch, cells) if engine == rt.GRAM_TCGEN05 else None
        half = batch * n * 8                             # bytes of one point set
        try:
            with torch.cuda.device(device):
                rt.check(lib.apap_local_homography_points(
                    p_dev.data_ptr(), p_dev.data_ptr() + half, c_dev.data_ptr() if c_dev is not None else None, batch, n,
                    v_dev.data_ptr(), cells, weight_scale(self.sigma), float(np.float32(float(self.gamma) ** 2)), engine,
                    rt.EIG_AUTO, ws[1].data_ptr(), ws[1].numel(), counters.data_ptr() if counters is not None else None,
                    out_h.data_ptr(), None, rt.stream_ptr(torch, device)), "apap_local_homography_points")
        except Exception:
            self._counters = None          # a failed call may leave counts behind: never reuse that scratch
            raise
        return rt.to_host(torch, out_h)

    def local_homography_batch(self, src_points, dst_points, vertices):
        """Extension (no reference API; its multi-image mode is a shell loop, run_all.sh:15,29):
        several pairs in one launch.  ``vertices`` is one ``[mesh_n, pt_size, 2]`` array shared by
        all pairs or a list of them (same shape).  Each item equals the single-pair call when the pairs' keypoint
        counts give the same Gram split plan (equal counts always do): the plan follows the largest count, so a
        smaller pair's grid can otherwise differ from its single call in the last bits."""
        count = len(src_points)
        verts = vertices if isinstance(vertices, (list, tuple)) else [vertices] * count
        mesh_n, pt_size, _ = np.shape(verts[0])
        cells = mesh_n * pt_size
        counts = np.array([np.shape(s)[0] for s in src_points], dtype=np.int32)
        if count == 0 or counts.min() == 0:
            raise ValueError("local_homography_batch needs at least one pair and one match per pair")
        points = np.zeros((2, count, int(counts.max()), 2), dtype=np.float32)
        for k, (s, d) in enumerate(zip(src_points, dst_points)):
            points[0, k, :counts[k]], points[1, k, :counts[k]] = s, d
        stacked = np.stack([np.asarray(v, dtype=np.float64).reshape(cells, 2) for v in verts])
        h = self._homography_pass(points, counts, stacked).reshape(count, mesh_n, pt_size, 3, 3)
        return [h[k] for k in range(count)]

    # ---- mesh warp -----------------------------------------------------------------------------
    def _luts(self, mesh, grid_rows, grid_cols):
        mesh = np.asarray(mesh)
        key = (mesh.shape, mesh.tobytes(), int(self.final_width), int(self.final_height), grid_rows, grid_cols)
        hit = self._lut_cache.get(key)
        if hit is None:
            hit = cell_lookup_tables(mesh, int(self.final_width), int(self.final_height), grid_rows, grid_cols)
            self._lut_cache = {key: hit}
        return hit

    def warp_tables_device(self, inv_h, col_cell, row_cell, src_w, src_h, device=None, row0=0, row1=None, hinv_dev=None):
        """The warp kernel's inputs for an inverted grid and the canvas rows ``[row0, row1)``: one
        host->device copy (inverted grid, column LUT, row blocks, cell extents), then the per-cell
        fast-path records are built on the device (``apap_warp_tables``).  ``hinv_dev``: the inverted grid as a float32
        device tensor ``[cells * 9]`` (``inv_h`` is then only read for its shape and not uploaded)."""
        torch, device = rt.torch_cuda(device if device is not None else self.device)
        lib = rt.load_library()
        row1 = int(self.final_height) if row1 is None else row1
        gr, gc = inv_h.shape[0], inv_h.shape[1]
        key = (col_cell.tobytes(), row_cell.tobytes(), gr, gc, int(row0), int(row1))
        hit = getattr(self, "_warp_lut_cache", None)
        if hit is None or hit[0] != key:
            col_lut, row_first, col_ext, row_ext = warp_luts(col_cell, row_cell, gr, gc)
            blocks = build_row_blocks(row_cell, row_first, row0, row1)
            hit = (key, col_lut, blocks, col_ext, row_ext)
            self._warp_lut_cache = hit
        _, col_lut, blocks, col_ext, row_ext = hit
        if not hasattr(self, "_warp_stage"):
            self._warp_stage = _PinnedStage()
        if hinv_dev is None:
            hinv = np.ascontiguousarray(inv_h, dtype=np.float32).reshape(-1, 9)
            views = self._warp_stage.upload(torch, device, (hinv, col_lut, blocks, col_ext, row_ext))
            hinv_dev = views[0].view(torch.float32)
        else:
            views = [None] + self._warp_stage.upload(torch, device, (col_lut, blocks, col_ext, row_ext))
        fast = torch.empty(gr * gc * HINV_ROW, dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            rt.check(lib.apap_warp_tables(hinv_dev.data_ptr(), views[3].data_ptr(), views[4].data_ptr(), gr, gc,
                                          int(self.offset_x), int(self.offset_y), int(src_w), int(src_h),
                                          fast.data_ptr(), rt.stream_ptr(torch, device)), "apap_warp_tables")
        tiles = None
        if (int(src_w) * 3) % 16 == 0 and blocks.shape[0]:         # tile engine: 16-byte aligned source rows
            import ctypes
            need = ctypes.c_size_t()
            rt.check(lib.apap_warp_tiles_bytes(int(self.final_width), int(blocks.shape[0]), ctypes.byref(need)),
                     "apap_warp_tiles_bytes")
            tiles = torch.empty(max(int(need.value), 16), dtype=torch.uint8, device=device)
            with torch.cuda.device(device):
                rt.check(lib.apap_warp_tiles(fast.data_ptr(), hinv_dev.data_ptr(), views[1].data_ptr(), views[3].data_ptr(),
                                             views[2].data_ptr(), int(blocks.shape[0]), gc, int(self.final_width),
                                             int(self.offset_x), int(self.offset_y), int(src_h), int(src_w),
                                             tiles.data_ptr(), tiles.numel(), rt.stream_ptr(torch, device)),
                         "apap_warp_tiles")
        return WarpTables(fast, hinv_dev, views[1].view(torch.int32), views[3].view(torch.int32),
                          views[2].view(torch.int32), tiles, int(blocks.shape[0]), int(row0), int(row1))

    def warp_device(self, src_dev, tables, grid_cols, centre_dev=None, out=None, force_exact=False, multicast_ptr=None,
                    legacy=False):
        """Device-resident K3 (optionally fused with K4): writes the canvas rows ``[tables.row0,
        tables.row1)`` into ``out`` (``[row1-row0, final_width, 3]`` uint8, allocated when None).
        ``multicast_ptr``: address of canvas row ``tables.row0`` inside an NVLS multicast mapping of a panorama buffer
        that every GPU of the group holds (``sharding.SymmetricPanorama``): the band is stored into all of them by
        the kernel itself and ``out`` is not written.  ``legacy``: round 1's strip kernel instead of the tile engine
        (A/B timing and tests; same bytes).  With ``centre_dev`` the strip kernel runs either way."""
        torch, device = rt.torch_cuda(src_dev.device)
        lib = rt.load_library()
        fw = int(self.final_width)
        n_bytes = (tables.row1 - tables.row0) * fw * 3
        if multicast_ptr is None and out is None:
            out = torch.empty((tables.row1 - tables.row0, fw, 3), dtype=torch.uint8, device=device)
        ch, cw = (centre_dev.shape[0], centre_dev.shape[1]) if centre_dev is not None else (0, 0)
        with torch.cuda.device(device):
            rt.check(lib.apap_warp(
                src_dev.data_ptr(), src_dev.shape[0], src_dev.shape[1], tables.cell_fast.data_ptr(),
                tables.cell_hinv.data_ptr(), tables.col_lut.data_ptr(),
                tables.row_blocks.data_ptr(), tables.n_blocks, grid_cols, fw, int(self.offset_x), int(self.offset_y),
                tables.row0, tables.row1, centre_dev.data_ptr() if centre_dev is not None else None, ch, cw,
                int(multicast_ptr) if multicast_ptr is not None else out.data_ptr(),
                n_bytes if multicast_ptr is not None else out.numel(),
                (rt.WARP_FORCE_EXACT if force_exact else 0) | (rt.WARP_LEGACY if legacy else 0),
                1 if multicast_ptr is not None else 0,
                tables.tiles.data_ptr() if tables.tiles is not None else None,
                rt.stream_ptr(torch, device)), "apap_warp")
        return out

    def invert_grid(self, local_homography, device=None) -> int:
        """The per-cell ``np.linalg.inv`` of ``local_warp`` (pyviz/apap.py:201-203), stored back into the caller's
        array, with the same bits as numpy's.  The GPU inverts every cell in float64 (``apap_invert_grid``) and
        certifies the cells whose float32 rounding cannot differ from numpy's (LAPACK ``dgesv`` + one rounding);
        the rest -- about 1 in 10^4 on homography grids, and every singular or degenerate cell -- go through
        ``np.linalg.inv`` itself here, so errors surface exactly as in the reference (``LinAlgError``).
        Returns the number of cells numpy inverted.  Grids that are not C-contiguous float32 take numpy throughout."""
        grid = local_homography
        if not self._gpu_invertible(grid):
            invert_grid_inplace(grid)
            return int(grid.size // 9)
        torch, device = rt.torch_cuda(device if device is not None else self.device)
        _, out_pin, flag_pin, _ = self._invert_grid_async(torch, device, grid)
        torch.cuda.current_stream(device).synchronize()
        return self._invert_grid_finish(grid, out_pin, flag_pin)

    @staticmethod
    def _gpu_invertible(grid) -> bool:
        return (isinstance(grid, np.ndarray) and grid.dtype == np.float32 and grid.flags.c_contiguous
                and grid.ndim >= 2 and grid.shape[-2:] == (3, 3) and grid.size > 0)

    def _invert_grid_async(self, torch, device, grid):
        """Enqueue upload, ``apap_invert_grid`` and the copies back (pinned) without waiting: ``(inverse on the device
        float32 [cells * 9], pinned host inverse, pinned host flags, event after the flags copy)``; the host arrays are
        valid once the stream (the flags: the event) has been waited for."""
        lib = rt.load_library()
        cells = grid.size // 9
        with torch.cuda.device(device):
            g_dev = rt.to_device(torch, device, grid)
            out_dev = torch.empty(cells * 9, dtype=torch.float32, device=device)
            flag_dev = torch.empty(cells, dtype=torch.uint8, device=device)
            rt.check(lib.apap_invert_grid(g_dev.data_ptr(), cells, out_dev.data_ptr(), flag_dev.data_ptr(),
                                          rt.stream_ptr(torch, device)), "apap_invert_grid")
            out_pin = torch.empty(cells * 9, dtype=torch.float32, pin_memory=True)
            flag_pin = torch.empty(cells, dtype=torch.uint8, pin_memory=True)
            flag_pin.copy_(flag_dev, non_blocking=True)
            flags_here = torch.cuda.Event()
            flags_here.record()                          # the host may read the flags once this has passed
            out_pin.copy_(out_dev, non_blocking=True)
        return out_dev, out_pin, flag_pin, flags_here

    @staticmethod
    def _invert_grid_finish(grid, out_pin, flag_pin, redo=None, fixed=None):
        """Store the inverses into the caller's array (the cells the GPU could not certify through ``np.linalg.inv``,
        which may raise like the reference -- before anything is overwritten).  Returns the number of cells redone."""
        cells = grid.size // 9
        flat = grid.reshape(cells, 3, 3)
        if redo is None:
            redo = np.flatnonzero(flag_pin.numpy())
            fixed = np.linalg.inv(flat[redo]) if redo.size else None
        flat[...] = out_pin.numpy().reshape(cells, 3, 3)
        if redo.size:
            flat[redo] = fixed
        return int(redo.size)

    def _warp(self, ori_img, local_homography, mesh, centre_img=None, force_exact=False, interpolation="nearest"):
        if interpolation not in ("nearest", "bilinear"):
            raise ValueError("interpolation must be 'nearest' (the reference's truncating lookup) or 'bilinear'")
        if interpolation == "bilinear" and centre_img is not None:
            raise ValueError("the fused warp + blend runs in the reference's nearest mode only")
        mesh_n, pt_size, _, _ = local_homography.shape
        ori_h, ori_w, _ = ori_img.shape
        on_device = not isinstance(ori_img, np.ndarray)
        torch, device = rt.torch_cuda(ori_img.device if on_device else self.device)
        col_cell, row_cell = self._luts(mesh, mesh_n, pt_size)
        gpu_inverse = self._gpu_invertible(local_homography)
        # the grid goes up first (1.4 MB), is inverted, and its flags come back while the image copies -- asynchronous
        # from pinned memory -- are still in flight behind them: waiting for the flags costs nothing
        if gpu_inverse:
            hinv_dev, out_pin, flag_pin, flags_here = self._invert_grid_async(torch, device, local_homography)
        src_dev = ori_img.contiguous() if on_device else rt.to_device(torch, device, ori_img.astype(np.uint8, copy=False))
        centre_dev = None
        if centre_img is not None:
            centre_dev = (centre_img.contiguous() if not isinstance(centre_img, np.ndarray)
                          else rt.to_device(torch, device, centre_img.astype(np.uint8, copy=False)))

        def run(hinv_dev):
            tables = self.warp_tables_device(local_homography, col_cell, row_cell, ori_w, ori_h, device, hinv_dev=hinv_dev)
            if interpolation == "bilinear":
                return self.warp_bilinear_device(src_dev, tables, pt_size)
            return self.warp_device(src_dev, tables, pt_size, centre_dev=centre_dev, force_exact=force_exact)

        # in-place per-cell inverse, stored back in the caller's array (pyviz/apap.py:201-203)
        if not gpu_inverse:
            self.invert_grid(local_homography, device)
            out = run(None)
            return out if on_device else rt.to_host(torch, out)
        flags_here.synchronize()
        cells = mesh_n * pt_size
        redo = np.flatnonzero(flag_pin.numpy())
        fixed = None
        if redo.size:
            # the cells the certificate turned down: numpy's own inverse (raises like the reference, nothing has been
            # overwritten yet), patched into the device copy the warp reads
            fixed = np.linalg.inv(local_homography.reshape(cells, 3, 3)[redo])
            with torch.cuda.device(device):
                idx = torch.from_numpy(redo.astype(np.int64)).to(device)
                vals = torch.from_numpy(np.ascontiguousarray(fixed, dtype=np.float32).reshape(-1, 9)).to(device)
                hinv_dev.view(cells, 9).index_copy_(0, idx, vals)
        out = run(hinv_dev)
        host = None
        if not on_device:
            host = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
            host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
        self._invert_grid_finish(local_homography, out_pin, flag_pin, redo, fixed)
        return out if on_device else host.numpy()

    def warp_bilinear_device(self, src_dev, tables, grid_cols, out=None):
        """Device-resident opt-in bilinear mode (``apap_warp_bilinear``): the canvas rows ``[tables.row0, tables.row1)``."""
        torch, device = rt.torch_cuda(src_dev.device)
        lib = rt.load_library()
        fw = int(self.final_width)
        if out is None:
            out = torch.empty((tables.row1 - tables.row0, fw, 3), dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            rt.check(lib.apap_warp_bilinear(
                src_dev.data_ptr(), src_dev.shape[0], src_dev.shape[1], tables.cell_hinv.data_ptr(),
                tables.col_lut.data_ptr(), tables.row_blocks.data_ptr(), tables.n_blocks, grid_cols, fw,
                int(self.offset_x), int(self.offset_y), tables.row0, tables.row1, out.data_ptr(), out.numel(),
                rt.stream_ptr(torch, device)), "apap_warp_bilinear")
        return out

    def local_warp(self, ori_img, local_homography, mesh, progress=False, interpolation="nearest"):
        """Warp ``ori_img`` onto the canvas through the per-cell homographies (pyviz/apap.py:186-217).

        Like the reference it inverts ``local_homography`` IN PLACE (the caller's array holds the
        inverses afterwards).  ``mesh`` is the ``[2, mesh_n+1]`` edge array of ``get_mesh``.
        ``progress`` is accepted for compatibility (the reference's tqdm bar) and ignored.
        Returns the ``[final_height, final_width, 3]`` uint8 canvas, zero where nothing maps.

        ``interpolation`` (extension): ``"nearest"`` is the reference's truncating lookup (pyviz/apap.py:214-215),
        bit-exact; ``"bilinear"`` writes the same pixels (same float64 coordinates and strict bounds test) with a
        bilinear sample at the mapped position (``cv.warpPerspective``'s convention, pyviz/utils.py:114), within
        +-1 LSB of the float64 restatement ``oracle.apap_oracle.local_warp_bilinear``.
        """
        return self._warp(ori_img, local_homography, mesh, interpolation=interpolation)

    def local_warp_batch(self, ori_imgs, local_homographies, mesh, centre_imgs=None):
        """Extension (no reference API; its multi-image mode is a shell loop, run_all.sh:15,29): ``local_warp`` --
        or ``local_warp_blend`` when ``centre_imgs`` is given -- for several pairs that share the canvas and the
        mesh.  Every grid is inverted in place like the single call; each item equals the single-pair call."""
        centres = centre_imgs if centre_imgs is not None else [None] * len(ori_imgs)
        if not (len(ori_imgs) == len(local_homographies) == len(centres)):
            raise ValueError("local_warp_batch: one image, one grid (and one centre image) per pair")
        return [self._warp(img, grid, mesh, centre_img=centre) for img, grid, centre in
                zip(ori_imgs, local_homographies, centres)]

    def local_warp_blend(self, ori_img, local_homography, mesh, centre_img):
        """Extension: the reference driver's commented pipeline (pyviz/apap.py:258-261) in one
        kernel -- warp, paste ``centre_img`` at the offsets, ``uniform_blend``.  Same in-place
        inversion side effect as ``local_warp``."""
        return self._warp(ori_img, local_homography, mesh, centre_img=centre_img)
