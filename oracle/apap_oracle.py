"""CPU oracle for the APAP hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A numpy restatement of the algorithm in the reference's ``pyviz/apap.py`` and
``pyviz/apap_utils.py``.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import this module, and
only as the checker (or as the timed CPU arm) -- never as something the product path
calls.  ``cvx_proj_b200`` does not import it.

Parity pinning: the reference holds no tests, golden vectors or fixtures for this path
(SURVEY.md section 8c), and its arithmetic kernel (``cv.SVDecomp``, OpenCV >= 4.5,
un-vendored) lives outside ``/root/reference``.  The oracle is therefore pinned against
outputs of the reference itself, run in the build container by ``oracle/gen_golden.py``
(which imports ``/root/reference/pyviz/apap.py`` unmodified) and committed under
``tests/golden/``; ``tests/test_oracle_golden.py`` replays them.

Every function cites the reference lines it restates (paths relative to
``/root/reference/``).
"""
from __future__ import annotations

import numpy as np

try:  # OpenCV is what the reference calls for the SVD; numpy is the stand-in if absent
    import cv2 as _cv
except Exception:  # pragma: no cover
    _cv = None


# --------------------------------------------------------------------------- grid utils
def get_mesh(size, mesh_size, start=0):
    """pyviz/apap_utils.py:10-21 -- ``[2, mesh_size]`` float64 cell edges (x row, y row)."""
    w, h = size
    return np.stack([np.linspace(start, w, mesh_size), np.linspace(start, h, mesh_size)], axis=0)


def get_vertice(size, mesh_size, offsets):
    """pyviz/apap_utils.py:23-38 -- anchors ``linspace(0,w,m) + w/(2m)`` minus offsets."""
    w, h = size
    nx = np.linspace(0, w, mesh_size) + w / (mesh_size * 2)
    ny = np.linspace(0, h, mesh_size) + h / (mesh_size * 2)
    gx, gy = np.meshgrid(nx, ny)
    return np.stack([gx, gy], axis=-1) - np.array(offsets)


def final_size(src_shape, dst_shape, project_H):
    """pyviz/apap_utils.py:40-73 -- canvas ``(w, h, off_x, off_y)``; shapes are (h, w, c)."""
    h, w = src_shape[0], src_shape[1]
    corners = []
    for pt in (np.float32([0, 0, 1]), np.float32([0, h, 1]), np.float32([w, 0, 1]), np.float32([w, h, 1])):
        vec = np.matmul(project_H, pt)
        corners.append([vec[0] / vec[2], vec[1] / vec[2]])
    corners = np.array(corners).astype(int)          # np.int in the reference (:59)
    h, w = dst_shape[0], dst_shape[1]
    max_x = max(np.max(corners[:, 0]), w)
    max_y = max(np.max(corners[:, 1]), h)
    min_x = min(np.min(corners[:, 0]), 0)
    min_y = min(np.min(corners[:, 1]), 0)
    return (max_x - min_x, max_y - min_y,
            -min_x if min_x < 0 else 0, -min_y if min_y < 0 else 0)


def uniform_blend(img1, img2):
    """pyviz/apap_utils.py:75-88 restated in integers.

    ``(a+b) * 0.5`` truncated where both pixels are non-black (channel mean > 0 <=> any
    channel > 0), ``a + b`` elsewhere.  Where at most one pixel is non-black the other
    is all-zero, so the sum never exceeds 255 and the float64 path of the reference and
    this integer path agree bit for bit.
    """
    a = img1.astype(np.uint16)
    b = img2.astype(np.uint16)
    both = (img1.max(axis=-1) > 0) & (img2.max(axis=-1) > 0)
    s = a + b
    return np.where(both[..., None], s >> 1, s).astype(np.uint8)


def uniform_blend_float(img1, img2):
    """pyviz/apap_utils.py:75-88 step by step in float64 (used to validate the integer form)."""
    g = (np.mean(img1, axis=-1) > 0) & (np.mean(img2, axis=-1) > 0)
    res = img1.astype(np.float64) + img2.astype(np.float64)
    mask = np.tile(np.expand_dims(g * 0.5, axis=-1), [1, 1, 3])
    mask[mask == 0] = 1
    return (res * mask).astype(np.uint8)


# ---------------------------------------------------------------- normalisers (host O(N))
def normalize_2d_pts(point):
    """pyviz/apap.py:35-59 -- Hartley normaliser ``(t[3,3] f32, pts[N,2] f32)``."""
    n = point.shape[0]
    c = np.mean(point, axis=0)
    pt = point - c
    pt_mean = np.mean(np.sqrt(np.sum(np.square(pt), axis=1)))
    scale = np.sqrt(2) / (pt_mean + 1e-8)
    t = np.array([[scale, 0, -scale * c[0]],
                  [0, scale, -scale * c[1]],
                  [0, 0, 1]], dtype=np.float32)
    homog = np.column_stack((point.copy(), np.ones(n, dtype=np.float32)))
    return t, t.dot(homog.T).T[:, :2]


def conditioner_from_pts(point):
    """pyviz/apap.py:63-89 -- per-axis unbiased-std conditioner ``T[3,3] f32``."""
    n = point.shape[0]
    mean_x, mean_y = np.mean(point, axis=0)
    std = np.std(point, axis=0)
    std = np.sqrt(std * std * n / (n - 1))
    std_x, std_y = std
    std_x = std_x + (std_x == 0)
    std_y = std_y + (std_y == 0)
    nx = np.sqrt(2) / std_x
    ny = np.sqrt(2) / std_y
    return np.array([[nx, 0, -nx * mean_x], [0, ny, -ny * mean_y], [0, 0, 1]], dtype=np.float32)


def point_normalize(nf, c):
    """pyviz/apap.py:92-100 -- diagonal scale + translation, float32, vectorised."""
    cf = np.zeros_like(nf)
    cf[:, 0] = nf[:, 0] * c[0, 0] + c[0, 2]
    cf[:, 1] = nf[:, 1] * c[1, 1] + c[1, 2]
    return cf


def matrix_generate(n, cf1, cf2):
    """pyviz/apap.py:103-119 -- the ``[2N, 9]`` float32 DLT matrix, vectorised."""
    a = np.zeros((2 * n, 9), dtype=np.float32)
    x, y = cf1[:, 0], cf1[:, 1]
    xp, yp = cf2[:, 0], cf2[:, 1]
    a[0::2, 0] = x
    a[0::2, 1] = y
    a[0::2, 2] = 1
    a[0::2, 6] = (-xp) * x
    a[0::2, 7] = (-xp) * y
    a[0::2, 8] = -xp
    a[1::2, 3] = x
    a[1::2, 4] = y
    a[1::2, 5] = 1
    a[1::2, 6] = (-yp) * x
    a[1::2, 7] = (-yp) * y
    a[1::2, 8] = -yp
    return a


def _prepare(src_point, dst_point):
    """pyviz/apap.py:133-145 -- normalisers, conditioners and the DLT matrix."""
    n1, nf1 = normalize_2d_pts(src_point)
    n2, nf2 = normalize_2d_pts(dst_point)
    c1 = conditioner_from_pts(nf1)
    c2 = conditioner_from_pts(nf2)
    cf1 = point_normalize(nf1, c1)
    cf2 = point_normalize(nf2, c2)
    aa = matrix_generate(src_point.shape[0], cf1, cf2)
    return n1, n2, c1, c2, aa


def cell_weights(vertex, src_point, gamma, sigma):
    """pyviz/apap.py:142,150-152 -- ``max(exp(-|v - x_i| / sigma^2), gamma)``, float64 [N]."""
    inv = 1.0 / (sigma ** 2)
    d = np.tile(vertex, (src_point.shape[0], 1)) - src_point
    w = np.exp(-(np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2) * inv))
    w[w < gamma] = gamma
    return w


def local_weight(src_point, vertices, gamma, sigma):
    """Second output of ``local_homography`` (pyviz/apap.py:144,153,169): ``[m, p, N]`` f64."""
    m, p, _ = vertices.shape
    out = np.empty((m, p, src_point.shape[0]))
    for i in range(m):
        for j in range(p):
            out[i, j] = cell_weights(vertices[i, j], src_point, gamma, sigma)
    return out


def _svd_smallest(a):
    """pyviz/apap.py:160-161 -- last row of V^T of the (float64) weighted DLT matrix."""
    if _cv is not None:
        _, _, vt = _cv.SVDecomp(a)
    else:  # pragma: no cover
        _, _, vt = np.linalg.svd(a, full_matrices=False)
    return vt[-1, :]


def _denormalise(h, n1, n2, c1, c2):
    """pyviz/apap.py:164-167."""
    h = h.reshape(3, 3)
    h = np.linalg.inv(c2).dot(h).dot(c1)
    h = np.linalg.inv(n2).dot(h).dot(n1)
    return h / h[2, 2]


def local_homography_svd(src_point, dst_point, vertices, gamma, sigma, cells=None):
    """pyviz/apap.py:121-169, cell by cell exactly as the reference runs it.

    Returns ``H[m, p, 3, 3]`` float32.  ``cells`` (optional iterable of ``(i, j)``) limits
    the loop to a subset, leaving the other entries zero -- used for bounded CPU timing
    and for spot checks at sizes where the full loop takes hours.
    """
    m, p, _ = vertices.shape
    n1, n2, c1, c2, aa = _prepare(src_point, dst_point)
    out = np.zeros((m, p, 3, 3), dtype=np.float32)
    it = cells if cells is not None else ((i, j) for i in range(m) for j in range(p))
    for i, j in it:
        w = cell_weights(vertices[i, j], src_point, gamma, sigma)
        a = np.expand_dims(np.repeat(w, 2), -1) * aa
        out[i, j] = _denormalise(_svd_smallest(a), n1, n2, c1, c2)
    return out


def local_homography_gram64(src_point, dst_point, vertices, gamma, sigma, chunk=2048, dtype=np.float32):
    """Fast float64 cross-check of pyviz/apap.py:147-168 for large grids.

    ``(WA)^T (WA) = A^T W^2 A``: the smallest right singular vector of the row-weighted
    matrix is the eigenvector of the smallest eigenvalue of ``sum_i w_i^2 (a_2i a_2i^T +
    a_2i+1 a_2i+1^T)``.  Float64 throughout; validated against ``local_homography_svd``
    in tests (agreement ~1e-7 on the size-normalised metric) -- it is a checker for
    sizes the per-cell SVD loop cannot finish, not a restatement of the SVD itself.
    ``dtype=np.float64`` returns H before the final rounding (comparisons finer than a float32 ulp).
    """
    m, p, _ = vertices.shape
    n1, n2, c1, c2, aa = _prepare(src_point, dst_point)
    n = src_point.shape[0]
    a64 = aa.astype(np.float64)
    # per-keypoint 9x9 outer-product sums, flattened: [N, 81]
    outer = (a64[0::2, :, None] * a64[0::2, None, :] + a64[1::2, :, None] * a64[1::2, None, :]).reshape(n, 81)
    verts = vertices.reshape(-1, 2).astype(np.float64)
    inv = 1.0 / (sigma ** 2)
    t2 = np.linalg.inv(n2).astype(np.float64) @ np.linalg.inv(c2).astype(np.float64)
    t1 = c1.astype(np.float64) @ n1.astype(np.float64)
    src64 = src_point.astype(np.float64)
    out = np.empty((m * p, 3, 3), dtype=dtype)
    for s in range(0, m * p, chunk):
        v = verts[s:s + chunk]
        d = np.sqrt((v[:, None, 0] - src64[None, :, 0]) ** 2 + (v[:, None, 1] - src64[None, :, 1]) ** 2)
        w = np.maximum(np.exp(-(d * inv)), gamma)
        g = ((w * w) @ outer).reshape(-1, 9, 9)
        _, vecs = np.linalg.eigh(g)
        h = vecs[:, :, 0].reshape(-1, 3, 3)
        h = t2 @ h @ t1
        out[s:s + chunk] = (h / h[:, 2:3, 2:3]).astype(dtype)
    return out.reshape(m, p, 3, 3)


# --------------------------------------------------------------------------------- warp
def invert_grid(local_h):
    """pyviz/apap.py:201-203 -- per-cell ``np.linalg.inv`` stored back as float32.

    The stacked call runs the same LAPACK routine per 3x3 block as the reference's
    loop; ``tests/test_oracle_golden.py`` checks it is bit-identical to the loop.
    """
    return np.linalg.inv(local_h).astype(np.float32)


def cell_lookup(edges, extent):
    """pyviz/apap.py:207,209 -- ``np.where(k < edges)[0][0] - 1`` for k in range(extent)."""
    return (np.searchsorted(edges, np.arange(extent), side="right") - 1).astype(np.int64)


def local_warp(ori_img, inv_h, mesh, final_wh, offset):
    """pyviz/apap.py:196-215 with the double pixel loop vectorised per canvas.

    ``inv_h`` is the already inverted float32 grid (what the reference holds after
    :201-203).  Coordinates are float64 (``float32 H @ int64 p`` promotes, :182-183);
    the gather truncates toward zero and the bounds are strict (:214-215).
    """
    mesh_w, mesh_h = mesh
    fw, fh = int(final_wh[0]), int(final_wh[1])
    ox, oy = offset
    oh, ow = ori_img.shape[0], ori_img.shape[1]
    col = cell_lookup(mesh_w, fw)
    row = cell_lookup(mesh_h, fh)
    out = np.zeros((fh, fw, 3), dtype=np.uint8)
    x = (np.arange(fw) - ox).astype(np.float64)
    band = max(1, (1 << 22) // max(fw, 1))
    for i0 in range(0, fh, band):
        i1 = min(fh, i0 + band)
        h = inv_h[row[i0:i1, None], col[None, :]].astype(np.float64)      # [b, fw, 3, 3]
        y = (np.arange(i0, i1) - oy).astype(np.float64)[:, None]
        xx = np.broadcast_to(x[None, :], (i1 - i0, fw))
        t0 = h[..., 0, 0] * xx + h[..., 0, 1] * y + h[..., 0, 2]
        t1 = h[..., 1, 0] * xx + h[..., 1, 1] * y + h[..., 1, 2]
        t2 = h[..., 2, 0] * xx + h[..., 2, 1] * y + h[..., 2, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            tx = t0 / t2
            ty = t1 / t2
        ok = (0 < tx) & (tx < ow) & (0 < ty) & (ty < oh)
        sx = np.where(ok, tx, 0).astype(np.int64)
        sy = np.where(ok, ty, 0).astype(np.int64)
        blk = out[i0:i1]
        blk[ok] = ori_img[sy[ok], sx[ok]]
    return out


def local_warp_bilinear(ori_img, inv_h, mesh, final_wh, offset):
    """Float64 restatement of the OPT-IN bilinear mode of the mesh warp (no reference counterpart: the reference's
    ``local_warp`` truncates, pyviz/apap.py:214-215; BASELINE.json's north_star asks for "bilinear sample ... within
    +-1 LSB").  Everything up to the bounds test is ``local_warp`` above (pyviz/apap.py:196-213: cell lookup, float64
    coordinates from the float32 inverted grid, strict ``0 < t < size``); the written pixels get the bilinear sample at
    ``(tx, ty)`` with the convention of the reference's only bilinear sampler, ``cv.warpPerspective`` (pyviz/utils.py:114):
    pixel centres at integer coordinates, taps ``floor`` and ``floor + 1`` clamped to the image, rounded half up."""
    mesh_w, mesh_h = mesh
    fw, fh = int(final_wh[0]), int(final_wh[1])
    ox, oy = offset
    oh, ow = ori_img.shape[0], ori_img.shape[1]
    col = cell_lookup(mesh_w, fw)
    row = cell_lookup(mesh_h, fh)
    out = np.zeros((fh, fw, 3), dtype=np.uint8)
    x = (np.arange(fw) - ox).astype(np.float64)
    img = ori_img.astype(np.float64)
    band = max(1, (1 << 21) // max(fw, 1))
    for i0 in range(0, fh, band):
        i1 = min(fh, i0 + band)
        h = inv_h[row[i0:i1, None], col[None, :]].astype(np.float64)
        y = (np.arange(i0, i1) - oy).astype(np.float64)[:, None]
        xx = np.broadcast_to(x[None, :], (i1 - i0, fw))
        t0 = h[..., 0, 0] * xx + h[..., 0, 1] * y + h[..., 0, 2]
        t1 = h[..., 1, 0] * xx + h[..., 1, 1] * y + h[..., 1, 2]
        t2 = h[..., 2, 0] * xx + h[..., 2, 1] * y + h[..., 2, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            tx = t0 / t2
            ty = t1 / t2
        ok = (0 < tx) & (tx < ow) & (0 < ty) & (ty < oh)
        tx, ty = tx[ok], ty[ok]
        x0, y0 = np.floor(tx).astype(np.int64), np.floor(ty).astype(np.int64)
        x1, y1 = np.minimum(x0 + 1, ow - 1), np.minimum(y0 + 1, oh - 1)
        fx, fy = (tx - x0)[:, None], (ty - y0)[:, None]
        val = ((1 - fx) * (1 - fy) * img[y0, x0] + fx * (1 - fy) * img[y0, x1] +
               (1 - fx) * fy * img[y1, x0] + fx * fy * img[y1, x1])
        blk = out[i0:i1]
        blk[ok] = np.minimum(np.floor(val + 0.5), 255).astype(np.uint8)
    return out


def local_warp_loop(ori_img, inv_h, mesh, final_wh, offset):
    """pyviz/apap.py:206-215 pixel by pixel (pure Python; small canvases only)."""
    mesh_w, mesh_h = mesh
    fw, fh = int(final_wh[0]), int(final_wh[1])
    ox, oy = offset
    oh, ow = ori_img.shape[0], ori_img.shape[1]
    out = np.zeros((fh, fw, 3), dtype=np.uint8)
    for i in range(fh):
        m = np.where(i < mesh_h)[0][0]
        for j in range(fw):
            n = np.where(j < mesh_w)[0][0]
            t = inv_h[m - 1, n - 1] @ np.array([j - ox, i - oy, 1])
            t /= t[2]
            if 0 < t[0] < ow and 0 < t[1] < oh:
                out[i, j] = ori_img[int(t[1]), int(t[0])]
    return out


def paste_centre(canvas_like, centre_img, offset):
    """pyviz/apap.py:259-260 -- centre image pasted on an empty canvas at the offsets."""
    ox, oy = offset
    out = np.zeros_like(canvas_like)
    ch, cw = centre_img.shape[0], centre_img.shape[1]
    out[oy:oy + ch, ox:ox + cw] = centre_img
    return out


def mat_layout(local_h):
    """pyviz/apap.py:250-265 -- the ``.mat`` product: per-cell inverse, ``/[2,2]``,
    transposed (column-major 3x3), float64, ``[cells, 9]``."""
    g = local_h.copy()
    m, p = g.shape[:2]
    for i in range(m):
        for j in range(p):
            g[i, j] = np.linalg.inv(g[i, j].copy())
            g[i, j] /= g[i, j, -1, -1]
    return g.transpose(0, 1, 3, 2).astype(np.float64).reshape(-1, 9)


# ------------------------------------------------------------------------------ metrics
def h_error_normalised(h, h_ref, extent):
    """SURVEY.md section 8c gate: per-cell ``max|S2 (H - Href) S1^-1| / max|S2 Href S1^-1|``
    with ``S = diag(1/L, 1/L, 1)``, ``L = extent``.  Returns the ``[cells]`` array."""
    length = float(extent)
    s2 = np.array([1.0 / length, 1.0 / length, 1.0])[:, None]
    s1i = np.array([length, length, 1.0])[None, :]
    h = h.reshape(-1, 3, 3).astype(np.float64)
    r = h_ref.reshape(-1, 3, 3).astype(np.float64)
    num = np.abs((h - r) * s2 * s1i).max(axis=(1, 2))
    den = np.abs(r * s2 * s1i).max(axis=(1, 2))
    return num / den


def h_error_raw(h, h_ref):
    """Largest element-wise relative error (entries with |Href| < 1e-12 skipped)."""
    h = h.reshape(-1, 9).astype(np.float64)
    r = h_ref.reshape(-1, 9).astype(np.float64)
    keep = np.abs(r) >= 1e-12
    return float((np.abs(h - r)[keep] / np.abs(r)[keep]).max())
