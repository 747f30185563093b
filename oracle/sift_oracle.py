"""TEST INFRASTRUCTURE (not shipped, never imported by cvx_proj_b200): numpy restatement of ``cv.SIFT.compute`` at
keypoints built the reference's way (pyviz/utils.py:144-147: ``cv.KeyPoint(x, y, 1)``, octave 0, angle -1), in the
operation order of the kernels of ``csrc/sift.cu`` -- so the kernels are bit-identical to it and it is within +-2 per
component (almost always equal) of OpenCV 4.x.

With provided octave-0 keypoints, ``SIFT_Impl::detectAndCompute`` sets ``firstOctave = 0``, ``actualNOctaves = 1``, and
``calcDescriptors`` reads only ``gpyr[0]``: the gray image blurred once by sigma = sqrt(1.6^2 - 0.5^2).  Per keypoint
``calcSIFTDescriptor`` accumulates 4 x 4 x 8 trilinear orientation histograms of the gradients around the rounded point.
Every step is float32, one rounding per operation, no fused multiply-add.  What OpenCV does differently (sum orders of
its SIMD blur and of the norms, FMA in its vector atan / magnitude / exp) moves a component by at most +-2.
"""
import numpy as np

D, N = 4, 8                                   # SIFT_DESCR_WIDTH, SIFT_DESCR_HIST_BINS
SIGMA, INIT_SIGMA = np.float32(1.6), np.float32(0.5)
DESCR_SCL_FCTR, DESCR_MAG_THR, INT_DESCR_FCTR = np.float32(3.0), np.float32(0.2), np.float32(512.0)
FLT_EPSILON = np.float32(np.finfo(np.float32).eps)
DBL_EPSILON_F = np.float32(np.finfo(np.float64).eps)
HIST_SLOTS = (D + 2) * (D + 2) * (N + 2)      # 360; slot -1 is a guard (see describe_base)
# slot offsets of the 8 trilinear contributions v_rco000, 001, 010, 011, 100, 101, 110, 111
SLOT_OFFSETS = (0, 1, N + 2, N + 3, (D + 2) * (N + 2), (D + 2) * (N + 2) + 1, (D + 3) * (N + 2), (D + 3) * (N + 2) + 1)
_F = np.float32
# cv::fastAtan2 coefficients (degrees)
_P1 = _F(0.9997878412794807) * _F(180 / np.pi)
_P3 = _F(-0.3258083974640975) * _F(180 / np.pi)
_P5 = _F(0.1555786518463281) * _F(180 / np.pi)
_P7 = _F(-0.04432655554792128) * _F(180 / np.pi)


def gray(bgr):
    """``cv.cvtColor(bgr, cv.COLOR_BGR2GRAY)`` for uint8: 15-bit fixed-point coefficients, rounded."""
    b = bgr.astype(np.int32)
    return ((3735 * b[..., 0] + 19235 * b[..., 1] + 9798 * b[..., 2] + (1 << 14)) >> 15).astype(np.uint8)


def blur_sigma():
    """sig_diff of createInitialImage (no upscaling): sqrtf(max(sigma^2 - init_sigma^2, 0.01f))."""
    return np.sqrt(np.maximum(SIGMA * SIGMA - INIT_SIGMA * INIT_SIGMA, _F(0.01)))


def gaussian_taps():
    """``cv.getGaussianKernel(ksize, sig, CV_32F)`` with ``ksize = cvRound(sig * 8 + 1) | 1`` (= 13): exp(-x^2 / 2 sig^2)
    in float64, normalised, rounded to float32."""
    sig = float(blur_sigma())
    ksize = int(np.rint(sig * 8 + 1)) | 1
    x = np.arange(ksize, dtype=np.float64) - (ksize - 1) * 0.5
    t = np.exp(-0.5 / (sig * sig) * x * x)
    return (t / t.sum()).astype(np.float32)


def reflect101(p, n):
    """``cv::borderInterpolate(p, n, BORDER_REFLECT_101)`` elementwise."""
    p = np.array(p, dtype=np.int64)
    if n == 1:
        return np.zeros_like(p)
    while True:
        lo, hi = p < 0, p >= n
        if not (lo.any() or hi.any()):
            return p
        p = np.where(lo, -p, np.where(hi, 2 * (n - 1) - p, p))


def base_image(bgr):
    """Gray float32 blurred by the 13 taps: horizontal pass, then vertical, reflect-101 borders; each output is
    ``((t0 x[-6] + t1 x[-5]) + t2 x[-4]) + ...`` (taps in order, no FMA)."""
    g = gray(np.asarray(bgr, dtype=np.uint8)).astype(np.float32)
    h, w = g.shape
    t = gaussian_taps()
    r = len(t) // 2
    cols = reflect101(np.arange(-r, w + r), w)
    src = g[:, cols]
    acc = t[0] * src[:, 0:w]
    for k in range(1, len(t)):
        acc = acc + t[k] * src[:, k:k + w]
    rows = reflect101(np.arange(-r, h + r), h)
    src = acc[rows, :]
    out = t[0] * src[0:h]
    for k in range(1, len(t)):
        out = out + t[k] * src[k:k + h]
    return out.astype(np.float32)


def sample_table(size, angle, h, w):
    """``(table float32 [n, 5] = (i, j, rbin, cbin, weight), ori float32)``: the samples of calcSIFTDescriptor's
    (i outer, j inner) loop that pass the bin test, in loop order -- the part that depends only on the keypoint's size and
    angle, not on its position or the image.  A literal restatement of the C++ loop."""
    size, angle = _F(size), _F(angle)
    ori = _F(360.0) - angle
    if abs(ori - _F(360.0)) < FLT_EPSILON:
        ori = _F(0.0)
    scl = size * _F(0.5)
    hist_width = DESCR_SCL_FCTR * scl
    radius = int(np.rint(hist_width * _F(1.4142135623730951) * _F(D + 1) * _F(0.5)))
    radius = min(radius, int(np.sqrt(float(w) * w + float(h) * h)))
    rad = ori * _F(np.pi / 180)
    cos_t = _F(np.cos(np.float64(rad))) / hist_width
    sin_t = _F(np.sin(np.float64(rad))) / hist_width
    exp_scale = _F(-1.0) / _F(D * D * 0.5)
    rows = []
    for i in range(-radius, radius + 1):
        for j in range(-radius, radius + 1):
            c_rot = _F(j) * cos_t - _F(i) * sin_t
            r_rot = _F(j) * sin_t + _F(i) * cos_t
            rbin = r_rot + _F(D // 2) - _F(0.5)
            cbin = c_rot + _F(D // 2) - _F(0.5)
            if -1 < rbin < D and -1 < cbin < D:
                wgt = _F(np.exp(np.float64((c_rot * c_rot + r_rot * r_rot) * exp_scale)))
                rows.append((i, j, rbin, cbin, wgt))
    return np.array(rows, dtype=np.float32).reshape(-1, 5), ori


def fast_atan2(y, x):
    """``cv::fastAtan2(y, x)`` in degrees, elementwise, multiply and add rounded separately."""
    ax, ay = np.abs(x), np.abs(y)
    ge = ax >= ay
    c = np.minimum(ax, ay) / (np.maximum(ax, ay) + DBL_EPSILON_F)
    c2 = c * c
    a = (((_P7 * c2 + _P5) * c2 + _P3) * c2 + _P1) * c
    a = np.where(ge, a, _F(90.0) - a)
    a = np.where(x < 0, _F(180.0) - a, a)
    return np.where(y < 0, _F(360.0) - a, a).astype(np.float32)


def _warp_sum_sq(v):
    """sum of v^2 over the 128 components of each row in the order of the kernel's warp reduction: lane l holds
    components l, l + 32, l + 64, l + 96 and sums their squares in that order, then xor-butterfly 16, 8, 4, 2, 1."""
    sq = v * v
    s = ((sq[:, 0:32] + sq[:, 32:64]) + sq[:, 64:96]) + sq[:, 96:128]
    while s.shape[1] > 1:
        half = s.shape[1] // 2
        s = s[:, :half] + s[:, half:]
    return s[:, 0]


def describe_base(base, pts, table, ori):
    """float32 [K, 128] descriptors of the points ``pts`` (float32 [K, 2], x y) on the blurred image ``base``."""
    base = np.asarray(base, dtype=np.float32)
    h, w = base.shape
    pts = np.asarray(pts, dtype=np.float32).reshape(-1, 2)
    k = pts.shape[0]
    px = np.rint(pts[:, 0]).astype(np.int64)                 # cvRound: half to even
    py = np.rint(pts[:, 1]).astype(np.int64)
    bpr = _F(N) / _F(360.0)
    ori = _F(ori)
    hist = np.zeros((k, 1 + HIST_SLOTS), dtype=np.float32)    # column 0 = slot -1 (written, never read)
    kk = np.arange(k)
    for i, j, rbin, cbin, wgt in table:
        r, c = py + int(i), px + int(j)
        ok = (r > 0) & (r < h - 1) & (c > 0) & (c < w - 1)
        if not ok.any():
            continue
        rs, cs = np.where(ok, r, 1), np.where(ok, c, 1)
        dx = base[rs, np.minimum(cs + 1, w - 1)] - base[rs, cs - 1]
        dy = base[np.maximum(rs - 1, 0), cs] - base[np.minimum(rs + 1, h - 1), cs]
        o = fast_atan2(dy, dx)
        mag = np.sqrt(dx * dx + dy * dy) * wgt
        obin = (o - ori) * bpr
        r0, c0 = int(np.floor(rbin)), int(np.floor(cbin))
        o0 = np.floor(obin).astype(np.int64)
        rb, cb = rbin - _F(r0), cbin - _F(c0)
        ob = obin - o0.astype(np.float32)
        o0 = np.where(o0 < 0, o0 + N, o0)
        o0 = np.where(o0 >= N, o0 - N, o0)
        v_r1 = mag * rb; v_r0 = mag - v_r1
        v_rc11 = v_r1 * cb; v_rc10 = v_r1 - v_rc11
        v_rc01 = v_r0 * cb; v_rc00 = v_r0 - v_rc01
        v_rco111 = v_rc11 * ob; v_rco110 = v_rc11 - v_rco111
        v_rco101 = v_rc10 * ob; v_rco100 = v_rc10 - v_rco101
        v_rco011 = v_rc01 * ob; v_rco010 = v_rc01 - v_rco011
        v_rco001 = v_rc00 * ob; v_rco000 = v_rc00 - v_rco001
        idx = ((r0 + 1) * (D + 2) + c0 + 1) * (N + 2) + o0 + 1        # + 1: the guard column
        sel = kk[ok]
        for off, v in zip(SLOT_OFFSETS, (v_rco000, v_rco001, v_rco010, v_rco011,
                                         v_rco100, v_rco101, v_rco110, v_rco111)):
            col = idx[ok] + off
            hist[sel, col] = hist[sel, col] + v[ok]
    hist = hist[:, 1:].reshape(k, D + 2, D + 2, N + 2)[:, 1:D + 1, 1:D + 1]
    raw = hist[..., :N].copy()
    raw[..., 0] = raw[..., 0] + hist[..., N]
    raw[..., 1] = raw[..., 1] + hist[..., N + 1]
    raw = raw.reshape(k, D * D * N)
    thr = np.sqrt(_warp_sum_sq(raw)) * DESCR_MAG_THR
    raw = np.minimum(raw, thr[:, None])
    nrm = INT_DESCR_FCTR / np.maximum(np.sqrt(_warp_sum_sq(raw)), FLT_EPSILON)
    return np.clip(np.rint(raw * nrm[:, None]), 0, 255).astype(np.float32)


def describe(bgr, pts, size=1.0, angle=-1.0):
    """``cv.SIFT.create().compute(bgr, [cv.KeyPoint(x, y, size, angle) ...])[1]`` restated."""
    bgr = np.asarray(bgr, dtype=np.uint8)
    table, ori = sample_table(size, angle, bgr.shape[0], bgr.shape[1])
    return describe_base(base_image(bgr), pts, table, ori)
