"""numpy / Python restatement of OpenCV 4.x ``cv.findHomography(src, dst, cv.RANSAC, threshold, maxIters=...,
confidence=...)`` (calib3d/src/fundam.cpp, calib3d/src/ptsetreg.cpp): the RNG, the subset drawing, the subset checks,
the minimal-set kernel, the float32 reprojection error and the adaptive loop.  The final Levenberg-Marquardt
refinement is not restated: OpenCV's own ``cv.findHomography(src[best], dst[best], 0)`` produces it (runKernel + LM on
the given points), which is what ``findHomography`` runs on the best hypothesis's inliers.

Test infrastructure only (the package does not import it): tests/test_ransac.py holds it equal to the live OpenCV, and
the GPU kernels (csrc/ransac.cu) equal to its per-hypothesis record.
"""
from __future__ import annotations

import math

import numpy as np

MODEL_POINTS = 4
MAX_ATTEMPTS = 10000              # getSubset(..., 10000) in RANSACPointSetRegistrator::run
RNG_COEFF = 4164903690            # CV_RNG_COEFF
FLT_EPSILON = float(np.finfo(np.float32).eps)
DBL_EPSILON = float(np.finfo(np.float64).eps)
DBL_MIN = float(np.finfo(np.float64).tiny)
_M64 = (1 << 64) - 1
_F = np.float32


class RNG:
    """``cv::RNG``: multiply-with-carry on a 64-bit state; ``RANSACPointSetRegistrator::run`` seeds it with
    ``(uint64)-1``."""

    def __init__(self, state=_M64):
        self.state = state

    def next(self):
        self.state = ((self.state & 0xFFFFFFFF) * RNG_COEFF + (self.state >> 32)) & _M64
        return self.state & 0xFFFFFFFF

    def uniform(self, a, b):
        """``RNG::uniform(int a, int b)``: ``(unsigned)next() % (b - a) + a``."""
        return a if a == b else self.next() % (b - a) + a


def have_collinear_points(p):
    """``haveCollinearPoints(m, 4)``: the last point against the line through every pair of the earlier ones.  The
    differences are float32 (``Point2f`` arithmetic) widened to double; the cross product and the bound are double."""
    i = len(p) - 1
    for j in range(i):
        dx1 = float(_F(p[j, 0]) - _F(p[i, 0]))
        dy1 = float(_F(p[j, 1]) - _F(p[i, 1]))
        for k in range(j):
            dx2 = float(_F(p[k, 0]) - _F(p[i, 0]))
            dy2 = float(_F(p[k, 1]) - _F(p[i, 1]))
            if abs(dx2 * dy1 - dy2 * dx1) <= FLT_EPSILON * (abs(dx1) + abs(dy1) + abs(dx2) + abs(dy2)):
                return True
    return False


def _det3(p, t):
    """``determinant(Matx33d(x0, y0, 1, x1, y1, 1, x2, y2, 1))`` in ``Matx_DetOp<double, 3>``'s order."""
    (x0, y0), (x1, y1), (x2, y2) = (tuple(map(float, p[i])) for i in t)
    return x0 * (y1 * 1.0 - y2 * 1.0) - y0 * (x1 * 1.0 - x2 * 1.0) + 1.0 * (x1 * y2 - x2 * y1)


_TRIANGLES = ((0, 1, 2), (1, 2, 3), (0, 2, 3), (0, 1, 3))


def check_subset(ms1, ms2):
    """``HomographyEstimatorCallback::checkSubset``: no collinear points in either set, and the four triangles have
    the same orientation in both sets (0 or 4 of the determinant products negative)."""
    if have_collinear_points(ms1) or have_collinear_points(ms2):
        return False
    negative = sum(_det3(ms1, t) * _det3(ms2, t) < 0 for t in _TRIANGLES)
    return negative in (0, 4)


def get_subset(rng, src, dst, max_attempts=MAX_ATTEMPTS):
    """``RANSACPointSetRegistrator::getSubset``: per attempt, 4 indices drawn with ``uniform(0, n)`` (a drawn index
    already in the attempt is drawn again); the first attempt that passes ``check_subset`` is returned, ``None`` after
    ``max_attempts`` failures."""
    n = len(src)
    for _ in range(max_attempts):
        idx = []
        for _ in range(MODEL_POINTS):
            j = rng.uniform(0, n)
            while j in idx:
                j = rng.uniform(0, n)
            idx.append(j)
        if check_subset(src[idx], dst[idx]):
            return idx
    return None


def run_kernel(M, m):
    """``HomographyEstimatorCallback::runKernel`` on the points ``M -> m``: float64 [3, 3] with H22 = 1, or ``None``
    (a mean absolute deviation below DBL_EPSILON: 0 models).  Every step is OpenCV's, the eigen-solver included, so the
    result is OpenCV's bit for bit."""
    M = np.asarray(M, np.float32)
    m = np.asarray(m, np.float32)
    count = len(M)
    cmx = cmy = cMx = cMy = 0.0
    for i in range(count):
        cmx += float(m[i, 0]); cmy += float(m[i, 1])
        cMx += float(M[i, 0]); cMy += float(M[i, 1])
    cmx /= count; cmy /= count; cMx /= count; cMy /= count
    smx = smy = sMx = sMy = 0.0
    for i in range(count):
        smx += abs(float(m[i, 0]) - cmx); smy += abs(float(m[i, 1]) - cmy)
        sMx += abs(float(M[i, 0]) - cMx); sMy += abs(float(M[i, 1]) - cMy)
    if abs(smx) < DBL_EPSILON or abs(smy) < DBL_EPSILON or abs(sMx) < DBL_EPSILON or abs(sMy) < DBL_EPSILON:
        return None
    smx = count / smx; smy = count / smy
    sMx = count / sMx; sMy = count / sMy
    inv_hnorm = np.array([[1.0 / smx, 0, cmx], [0, 1.0 / smy, cmy], [0, 0, 1]])
    hnorm2 = np.array([[sMx, 0, -cMx * sMx], [0, sMy, -cMy * sMy], [0, 0, 1]])
    ltl = np.zeros((9, 9))
    for i in range(count):
        x, y = (float(m[i, 0]) - cmx) * smx, (float(m[i, 1]) - cmy) * smy
        X, Y = (float(M[i, 0]) - cMx) * sMx, (float(M[i, 1]) - cMy) * sMy
        lx = (X, Y, 1.0, 0.0, 0.0, 0.0, -x * X, -x * Y, -x)
        ly = (0.0, 0.0, 0.0, X, Y, 1.0, -y * X, -y * Y, -y)
        for j in range(9):
            for k in range(j, 9):
                ltl[j, k] += lx[j] * lx[k] + ly[j] * ly[k]
    _, v = jacobi(ltl)                                         # cv::eigen of the symmetric LtL
    h0 = v[8].reshape(3, 3)
    return _scale(_mat3(_mat3(inv_hnorm, h0), hnorm2))


def _div(a, b):
    """IEEE double division (C's ``a / b``: inf or NaN where Python would raise)."""
    with np.errstate(all="ignore"):
        return float(np.float64(a) / np.float64(b))


def _hypot(a, b):
    """``hypot`` of OpenCV's lapack.cpp (not ``std::hypot``)."""
    a, b = abs(a), abs(b)
    if a > b:
        b = _div(b, a)
        return a * math.sqrt(1 + b * b)
    if b > 0:
        a = _div(a, b)
        return b * math.sqrt(1 + a * a)
    return 0.0


def jacobi(a):
    """``cv::eigen`` of a symmetric float64 matrix = ``JacobiImpl_`` (OpenCV 4.x core/src/lapack.cpp): cyclic Jacobi
    with the largest off-diagonal element as pivot (found through per-row / per-column maxima of the upper triangle),
    at most 30 n^2 rotations, stop at |pivot| <= DBL_EPSILON, eigenvalues sorted descending by selection sort.
    Returns ``(w [n], v [n, n])`` with the eigenvectors as rows.  Only the upper triangle of ``a`` is read."""
    A = [[float(x) for x in row] for row in np.asarray(a, np.float64)]
    n = len(A)
    V = [[1.0 if i == j else 0.0 for j in range(n)] for i in range(n)]
    W = [A[k][k] for k in range(n)]
    ind_r, ind_c = [0] * n, [0] * n

    def row_max(k):
        m, mv = k + 1, abs(A[k][k + 1])
        for i in range(k + 2, n):
            if mv < abs(A[k][i]):
                mv, m = abs(A[k][i]), i
        ind_r[k] = m

    def col_max(k):
        m, mv = 0, abs(A[0][k])
        for i in range(1, k):
            if mv < abs(A[i][k]):
                mv, m = abs(A[i][k]), i
        ind_c[k] = m

    for k in range(n):
        if k < n - 1:
            row_max(k)
        if k > 0:
            col_max(k)
    for _ in range(n * n * 30):
        k, mv = 0, abs(A[0][ind_r[0]])
        for i in range(1, n - 1):
            if mv < abs(A[i][ind_r[i]]):
                mv, k = abs(A[i][ind_r[i]]), i
        l = ind_r[k]
        for i in range(1, n):
            if mv < abs(A[ind_c[i]][i]):
                mv, k, l = abs(A[ind_c[i]][i]), ind_c[i], i
        p = A[k][l]
        if abs(p) <= DBL_EPSILON:
            break
        y = (W[l] - W[k]) * 0.5
        t = abs(y) + _hypot(p, y)
        s = _hypot(p, t)
        c = _div(t, s)
        s = _div(p, s)
        t = _div(p, t) * p
        if y < 0:
            s, t = -s, -t
        A[k][l] = 0.0
        W[k] -= t
        W[l] += t

        def rot(a0, b0):
            return a0 * c - b0 * s, a0 * s + b0 * c
        for i in range(k):
            A[i][k], A[i][l] = rot(A[i][k], A[i][l])
        for i in range(k + 1, l):
            A[k][i], A[i][l] = rot(A[k][i], A[i][l])
        for i in range(l + 1, n):
            A[k][i], A[l][i] = rot(A[k][i], A[l][i])
        for i in range(n):
            V[k][i], V[l][i] = rot(V[k][i], V[l][i])
        for idx in (k, l):
            if idx < n - 1:
                row_max(idx)
            if idx > 0:
                col_max(idx)
    for k in range(n - 1):
        m = k
        for i in range(k + 1, n):
            if W[m] < W[i]:
                m = i
        if k != m:
            W[m], W[k] = W[k], W[m]
            V[m], V[k] = V[k], V[m]
    return np.array(W), np.array(V)


def _mat3(a, b):
    """3x3 product with the k-sum in order (what OpenCV's gemm does for these sizes)."""
    out = np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            out[i, j] = (a[i, 0] * b[0, j] + a[i, 1] * b[1, j]) + a[i, 2] * b[2, j]
    return out


def _scale(h):
    """``_H0.convertTo(_model, CV_64F, 1. / H22)``."""
    return h * (1.0 / h[2, 2])


def compute_error(src, dst, H):
    """``HomographyEstimatorCallback::computeError``: float32 [n] squared reprojection errors with ``Hf = (float)H``
    and every operation rounded on its own."""
    hf = np.asarray(H, np.float64).ravel()[:8].astype(np.float32)
    x, y = src[:, 0].astype(np.float32), src[:, 1].astype(np.float32)
    ww = _F(1.0) / (hf[6] * x + hf[7] * y + _F(1.0))
    dx = (hf[0] * x + hf[1] * y + hf[2]) * ww - dst[:, 0].astype(np.float32)
    dy = (hf[3] * x + hf[4] * y + hf[5]) * ww - dst[:, 1].astype(np.float32)
    return dx * dx + dy * dy


def inlier_mask(src, dst, H, threshold):
    """``findInliers``: error <= ``(float)(threshold * threshold)``."""
    return compute_error(src, dst, H) <= _F(float(threshold) * float(threshold))


def update_num_iters(p, ep, model_points, max_iters):
    """``RANSACUpdateNumIters``."""
    p = min(max(p, 0.0), 1.0)
    ep = min(max(ep, 0.0), 1.0)
    num = max(1.0 - p, DBL_MIN)
    denom = 1.0 - math.pow(1.0 - ep, model_points)
    if denom < DBL_MIN:
        return 0
    num = math.log(num)
    denom = math.log(denom)
    if denom >= 0 or -num >= max_iters * (-denom):
        return max_iters
    return int(round(num / denom))                             # cvRound: half to even, like Python's round


def hypotheses(src, dst, threshold):
    """The hypotheses of the loop in draw order, without its stop: ``(subset, H or None, count)`` per iteration, count
    -1 for 0 models; ends when ``getSubset`` fails."""
    rng = RNG()
    while True:
        idx = get_subset(rng, src, dst)
        if idx is None:
            return
        H = run_kernel(src[idx], dst[idx])
        yield idx, H, (-1 if H is None else int(inlier_mask(src, dst, H, threshold).sum()))


def record(src, dst, threshold, max_iters):
    """The first ``max_iters`` hypotheses (fewer when the attempt limit ends the sequence): ``(subsets int32 [k, 4],
    valid bool [k], counts int32 [k], H float64 [k, 3, 3] (NaN where invalid))``."""
    src, dst = _f32(src), _f32(dst)
    rows = []
    for item in hypotheses(src, dst, threshold):
        rows.append(item)
        if len(rows) == max_iters:
            break
    subsets = np.array([r[0] for r in rows], np.int32).reshape(-1, 4)
    valid = np.array([r[1] is not None for r in rows], bool)
    counts = np.array([r[2] for r in rows], np.int32)
    hs = np.array([r[1] if r[1] is not None else np.full((3, 3), np.nan) for r in rows]).reshape(-1, 3, 3)
    return subsets, valid, counts, hs


def scan(counts, n, confidence, max_iters):
    """The loop of ``RANSACPointSetRegistrator::run`` over per-iteration inlier counts (``len(counts)`` = the
    iterations ``getSubset`` could fill): ``(best index or -1, iterations run)``; best -1 = no model."""
    niters, best, max_good, it = max(max_iters, 1), -1, 0, 0
    while it < niters:
        if it >= len(counts):
            if it == 0:
                return -1, 0
            break
        good = int(counts[it])
        if good > max(max_good, MODEL_POINTS - 1):
            best, max_good = it, good
            niters = update_num_iters(confidence, (n - good) / n, MODEL_POINTS, niters)
        it += 1
    return best, it


def _f32(a):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(-1, 2))


def find_homography(src, dst, threshold=5.0, confidence=0.995, max_iters=2000):
    """``cv.findHomography(src, dst, cv.RANSAC, threshold, maxIters=max_iters, confidence=confidence)``:
    ``(H float64 [3, 3] or None, mask uint8 [n, 1], rec)``, rec = ``dict(subsets, valid, counts, best,
    iterations)`` of the iterations run.  Fewer than 4 points raise ``ValueError`` (OpenCV: ``cv.error``)."""
    import cv2 as cv

    src, dst = _f32(src), _f32(dst)
    n = len(src)
    if n < MODEL_POINTS or len(dst) != n:
        raise ValueError("findHomography needs at least 4 corresponding points")
    if threshold <= 0:
        threshold = 3.0                                        # defaultRANSACReprojThreshold
    if n == MODEL_POINTS:                                      # findHomography: method 0 on the 4 points, mask all ones
        H = run_kernel(src, dst)
        rec = dict(subsets=np.arange(4, dtype=np.int32)[None], valid=np.array([H is not None]),
                   counts=np.array([4 if H is not None else -1], np.int32), best=0 if H is not None else -1,
                   iterations=0)
        return H, np.ones((n, 1), np.uint8) if H is not None else np.zeros((n, 1), np.uint8), rec
    # lazily: the loop usually stops long before max_iters
    gen = hypotheses(src, dst, threshold)
    rows = []
    niters, best, max_good, it = max(max_iters, 1), -1, 0, 0
    while it < niters:
        item = next(gen, None)
        if item is None:
            if it == 0:
                best = -1
            break
        rows.append(item)
        good = item[2]
        if good > max(max_good, MODEL_POINTS - 1):
            best, max_good = it, good
            niters = update_num_iters(confidence, (n - good) / n, MODEL_POINTS, niters)
        it += 1
    rec = dict(subsets=np.array([r[0] for r in rows], np.int32).reshape(-1, 4),
               valid=np.array([r[1] is not None for r in rows], bool),
               counts=np.array([r[2] for r in rows], np.int32), best=best, iterations=it)
    if best < 0:
        return None, np.zeros((n, 1), np.uint8), rec
    mask = inlier_mask(src, dst, rows[best][1], threshold)
    H = cv.findHomography(src[mask], dst[mask], 0)[0]          # runKernel + LM on the inliers, in index order
    return H, inlier_mask(src, dst, H, threshold).astype(np.uint8).reshape(-1, 1), rec
