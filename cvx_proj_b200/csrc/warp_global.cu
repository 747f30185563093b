// Global-homography warp + paste / mean blend -- the reference's `image_warping` (pyviz/utils.py:93-127):
// cv.warpPerspective (bilinear, constant border 0) of the image to warp onto the canvas, then the base image
// pasted over it (:124-125) or mean-blended where the warp left something (:115-123).
//
// Bit-exact with OpenCV's 8-bit bilinear warp (un-vendored dependency; algorithm restated in
// oracle/warp_oracle.py and pinned there against the live reference): destination pixels are processed in
// blocks `bw0` wide; for x = xb + x1 of row y, X0 = (M0 xb + M1 y) + M2 in float64, W = 32 / (W0 + M6 x1),
// X = round-to-nearest-even(clamp((X0 + M0 x1) W)) -- source coordinates in 1/32 pixel -- and the four taps
// around (X >> 5, Y >> 5) are combined with the 15-bit fixed-point weights (32 - fx | fx)(32 - fy | fy) 2^5,
// (sum + 2^14) >> 15; a tap outside the source is 0.  All float64 operations are explicit _rn (no FMA
// contraction), in OpenCV's order.
//
// HBM-bound byte work: 3 B written per canvas pixel, every source pixel read at most once from HBM (the four
// taps of neighbouring pixels overlap in L1).  CTA = a 256 x 32 canvas tile, warp = a 32-pixel segment column,
// lane = canvas column.
#include "common.cuh"

namespace apap {

struct GlobalWarpParams {
  const uint8_t *src;       // [src_h][src_w][3] image to warp
  const uint8_t *base;      // [base_h][base_w][3] base image, or nullptr (warp only)
  uint8_t *dst;             // [dst_h][dst_w][3] canvas
  double m[9];              // INVERSE map: canvas (x, y, 1) -> source, row-major
  int src_h, src_w, dst_h, dst_w, base_h, base_w;
  int off_x, off_y;         // where the base image sits on the canvas
  int bw0;                  // OpenCV's block width for this canvas
  int mode;                 // 0 warp only, 1 paste the base over the warp, 2 mean blend
};

__device__ __forceinline__ double clamp_int_range(double v) {
  // std::max((double)INT_MIN, std::min((double)INT_MAX, v)) as C++ evaluates it
  const double lo = -2147483648.0, hi = 2147483647.0;
  const double a = (v < hi) ? v : hi;
  return (lo < a) ? a : lo;
}

// OpenCV's float64 arithmetic for one canvas pixel: source coordinates in 1/32 pixel, before rounding.
__device__ __forceinline__ void exact_coords(const GlobalWarpParams &p, int x, int y, double &fX, double &fY, double &wa,
                                             double &bc_ad_x, double &bc_ad_y) {
  const double xb = (double)((x / p.bw0) * p.bw0), x1 = (double)(x % p.bw0), yd = (double)y;
  const double X0 = __dadd_rn(__dadd_rn(__dmul_rn(p.m[0], xb), __dmul_rn(p.m[1], yd)), p.m[2]);
  const double Y0 = __dadd_rn(__dadd_rn(__dmul_rn(p.m[3], xb), __dmul_rn(p.m[4], yd)), p.m[5]);
  const double W0 = __dadd_rn(__dadd_rn(__dmul_rn(p.m[6], xb), __dmul_rn(p.m[7], yd)), p.m[8]);
  const double Ws = __dadd_rn(W0, __dmul_rn(p.m[6], x1));
  const double W = (Ws != 0.0) ? __ddiv_rn(32.0, Ws) : 0.0;
  fX = clamp_int_range(__dmul_rn(__dadd_rn(X0, __dmul_rn(p.m[0], x1)), W));
  fY = clamp_int_range(__dmul_rn(__dadd_rn(Y0, __dmul_rn(p.m[3], x1)), W));
  wa = Ws;
  bc_ad_x = p.m[0] * W0 - X0 * p.m[6];           // d/dx1 of the numerator/denominator pair, see SegRec
  bc_ad_y = p.m[3] * W0 - Y0 * p.m[6];
}

// Fast path.  Inside one OpenCV block the map is v(x1) = 32 (a + b x1) / (c + d x1) per coordinate, so with an
// anchor column xa:  v(xa + t) = v(xa) + K t / (Wa + d t),  K = 32 (b c - a d) / Wa,  Wa = c + d xa  (exact algebra).
// Per 32-pixel segment of a canvas row one thread evaluates the anchor (its middle column) in float64 exactly as
// OpenCV does -- 32 segments per warp instruction, so the FP64 pipe (half the FP32 rate, long dependent chains) is touched once per 32 pixels
// instead of ~50 times per pixel -- and the pixels add the small term K t / (Wa + d t), |t| <= 16, in float32.  eps
// bounds the float32 error of that term; a pixel whose sum lands within eps of a rounding boundary (x.5) is
// re-decided with the float64 formula, the others round to the same integer in both arithmetics.
struct SegRec {
  int ix, iy;               // round(v(xa)) per coordinate
  float fx, fy;             // v(xa) - round(v(xa)), in [-0.5, 0.5]
  float kx, ky;             // K per coordinate
  float wa;                 // Wa
  float eps;                // error bound of the float32 sum; < 0: every pixel of the segment takes the float64 path
};

// kTileH: canvas rows per CTA tile (even, <= 32: one thread per (row, segment) in phase 1)
constexpr int kTileW = 256, kTileH = 16, kSegs = kTileW / 32;

__device__ __forceinline__ SegRec make_segment(const GlobalWarpParams &p, int xs, int y) {
  SegRec r;
  r.ix = r.iy = 0; r.fx = r.fy = r.kx = r.ky = 0.f; r.wa = 1.f; r.eps = -1.f;
  if (p.bw0 % 32 != 0) return r;                   // a segment would straddle OpenCV blocks: float64 for all
  const int xa = xs + 16;
  double fX, fY, wa, nx, ny;
  exact_coords(p, xa, y, fX, fY, wa, nx, ny);
  if (!(fabs(wa) > 1e-300) || !isfinite(wa)) return r;
  const double kx = 32.0 * nx / wa, ky = 32.0 * ny / wa;
  const double vary = fabs(p.m[6]) * 16.0 / fabs(wa);               // relative change of the denominator over the segment
  const double kmax = fmax(fabs(kx), fabs(ky));
  if (!(vary < 0.25) || !(kmax < 4096.0) || !(fabs(fX) < 4194304.0) || !(fabs(fY) < 4194304.0)) return r;
  const double dmax = 16.0 * kmax / (1.0 - vary);                   // largest |K t / (Wa + d t)|
  // float32 error of the sum: K, Wa, d rounded (3 x 2^-24), fma for the denominator, rcp.approx (2^-23), product,
  // final fma (relative to the sum) -- 8 x 2^-24 on the small term, 2^-23 on the sum, 1.5 x safety
  const double eps = 1.5 * (dmax * 8.0 * 5.9604644775390625e-08 + (0.5 + dmax) * 1.1920928955078125e-07) + 1e-6;
  if (!(eps < 0.125)) return r;
  const double rx = rint(fX), ry = rint(fY);
  r.ix = (int)rx; r.iy = (int)ry;
  r.fx = (float)(fX - rx); r.fy = (float)(fY - ry);
  r.kx = (float)kx; r.ky = (float)ky; r.wa = (float)wa;
  r.eps = (float)eps * 1.0000002f;
  return r;
}

__global__ void __launch_bounds__(256) k_warp_global(const GlobalWarpParams p) {
  __shared__ SegRec rec[kTileH][kSegs];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int x_tile = blockIdx.x * kTileW, y_tile = blockIdx.y * kTileH;
  {                                                // phase 1: one thread per (row, segment) of the tile
    const int r = tid / kSegs, s = tid % kSegs;
    const int xs = x_tile + s * 32, y = y_tile + r;
    SegRec v;
    v.ix = v.iy = 0; v.fx = v.fy = v.kx = v.ky = 0.f; v.wa = 1.f; v.eps = -1.f;
    if (r < kTileH) {
      if (y < p.dst_h && xs < p.dst_w) v = make_segment(p, xs, y);
      rec[r][s] = v;
    }
  }
  __syncthreads();
  const int x = x_tile + warp * 32 + lane;
  const bool col_ok = x < p.dst_w;
  const float t = (float)(lane - 16);
  const float d32 = (float)p.m[6];
  const int bx = x - p.off_x;
  const bool in_base_col = p.base && (unsigned)bx < (unsigned)p.base_w;
  const int rows = min(kTileH, p.dst_h - y_tile);
  const uint32_t src_pitch = (uint32_t)p.src_w * 3u, dst_pitch = (uint32_t)p.dst_w * 3u, base_pitch = (uint32_t)p.base_w * 3u;
  uint8_t *out = p.dst + ((size_t)y_tile * p.dst_w + (col_ok ? x : 0)) * 3;
  const uint8_t *bp = p.base ? p.base + ((long long)(y_tile - p.off_y) * p.base_w + bx) * 3 : nullptr;   // valid only inside the base

  // source coordinates of this lane's pixel of tile row r, in 1/32 pixel
  auto coords = [&](int r, int &X, int &Y) {
    const SegRec sr = rec[r][warp];
    bool exact = sr.eps < 0.f;
    if (!exact) {
      const float rw = rcp_approx(fmaf(d32, t, sr.wa));
      const float sx = fmaf(sr.kx * t, rw, sr.fx), sy = fmaf(sr.ky * t, rw, sr.fy);
      const float nx = rintf(sx), ny = rintf(sy);
      exact = !(0.5f - fabsf(sx - nx) > sr.eps) || !(0.5f - fabsf(sy - ny) > sr.eps);   // NaN -> exact
      X = sr.ix + (int)nx; Y = sr.iy + (int)ny;
    }
    if (exact) {                                   // rare: OpenCV's float64 formula
      double fX, fY, wa, nx, ny;
      exact_coords(p, col_ok ? x : p.dst_w - 1, y_tile + r, fX, fY, wa, nx, ny);
      X = __double2int_rn(fX); Y = __double2int_rn(fY);
    }
  };
  // paste / mean-blend with the base image and store (o, b: this row's canvas and base pointers)
  auto finish = [&](int acc0, int acc1, int acc2, bool in_base, uint8_t *o, const uint8_t *b) {
    int r0 = (acc0 + 512) >> 10, r1 = (acc1 + 512) >> 10, r2 = (acc2 + 512) >> 10;   // (32 acc + 2^14) >> 15
    if (in_base) {                                 // paste (mode 1) / mean where the warp left something (mode 2)
      const int b0 = b[0], b1 = b[1], b2 = b[2];
      if (p.mode == 2 && (r0 | r1 | r2)) {
        r0 = (r0 + b0) >> 1; r1 = (r1 + b1) >> 1; r2 = (r2 + b2) >> 1;
      } else {
        r0 = b0; r1 = b1; r2 = b2;
      }
    }
    if (col_ok) { o[0] = (uint8_t)r0; o[1] = (uint8_t)r1; o[2] = (uint8_t)r2; }
  };
  // one row, any position (image edges, partially covered warps)
  auto slow_row = [&](int X, int Y, bool in_base, uint8_t *o, const uint8_t *b) {
    const int sx = max(-32768, min(32767, X >> 5)), sy = max(-32768, min(32767, Y >> 5));
    const int ax = X & 31, ay = Y & 31;
    int acc0 = 0, acc1 = 0, acc2 = 0;
    if (sx >= -1 && sx < p.src_w && sy >= -1 && sy < p.src_h) {
#pragma unroll
      for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const int xx = sx + dx, yy = sy + dy;
          const int w = (dx ? ax : 32 - ax) * (dy ? ay : 32 - ay);      // x 2^5 = the 15-bit weight
          if (w != 0 && (unsigned)xx < (unsigned)p.src_w && (unsigned)yy < (unsigned)p.src_h) {
            const uint8_t *q = p.src + ((size_t)yy * p.src_w + xx) * 3;
            acc0 += w * (int)__ldg(q);
            acc1 += w * (int)__ldg(q + 1);
            acc2 += w * (int)__ldg(q + 2);
          }
        }
      }
    }
    finish(acc0, acc1, acc2, in_base, o, b);
  };

  for (int r = 0; r < rows; r += 2, out += 2 * dst_pitch, bp += 2 * base_pitch) {
    // two rows per pass: both rows' 24 byte loads are in flight together on the common path
    bool has[2], in_base[2], covered[2], inside[2];
    int X[2], Y[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      has[k] = r + k < rows;
      const int by = y_tile + r + k - p.off_y;
      in_base[k] = in_base_col && (unsigned)by < (unsigned)p.base_h;
      // paste mode: the base image covers the warp here (pyviz/utils.py:125) -- nothing to warp for the whole warp
      covered[k] = has[k] && p.mode == 1 && __all_sync(0xffffffffu, in_base[k] || !col_ok);
      inside[k] = false;
      if (has[k] && !covered[k]) {
        coords(r + k, X[k], Y[k]);
        const int sx = X[k] >> 5, sy = Y[k] >> 5;
        inside[k] = __all_sync(0xffffffffu, (unsigned)sx < (unsigned)(p.src_w - 1) && (unsigned)sy < (unsigned)(p.src_h - 1));
      }
    }
    if (inside[0] && inside[1]) {
      // all four taps of every lane lie in the source, in both rows: two 6-byte runs per pixel, no predicates
      int v[2][12];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const uint8_t *q = p.src + (size_t)((uint32_t)(Y[k] >> 5) * src_pitch + (uint32_t)(X[k] >> 5) * 3u);
        const uint8_t *q1 = q + src_pitch;
#pragma unroll
        for (int e = 0; e < 6; ++e) { v[k][e] = __ldg(q + e); v[k][6 + e] = __ldg(q1 + e); }
      }
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int ax = X[k] & 31, ay = Y[k] & 31;
        const int w00 = (32 - ax) * (32 - ay), w01 = ax * (32 - ay), w10 = (32 - ax) * ay, w11 = ax * ay;
        finish(w00 * v[k][0] + w01 * v[k][3] + w10 * v[k][6] + w11 * v[k][9],
               w00 * v[k][1] + w01 * v[k][4] + w10 * v[k][7] + w11 * v[k][10],
               w00 * v[k][2] + w01 * v[k][5] + w10 * v[k][8] + w11 * v[k][11], in_base[k], out + k * dst_pitch,
               bp + k * base_pitch);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (!has[k]) continue;
        uint8_t *o = out + k * dst_pitch;
        const uint8_t *b = bp + k * base_pitch;
        if (covered[k]) {
          if (col_ok) { o[0] = b[0]; o[1] = b[1]; o[2] = b[2]; }
        } else {
          slow_row(X[k], Y[k], in_base[k], o, b);
        }
      }
    }
  }
}

int launch_warp_global(const uint8_t *src, int src_h, int src_w, const double *minv, uint8_t *dst, int dst_h, int dst_w,
                       const uint8_t *base, int base_h, int base_w, int off_x, int off_y, int mode, cudaStream_t st) {
  if (dst_h == 0 || dst_w == 0) return 0;
  if (dst_h > 65535 * kTileH) return fail(APAP_E_TOOBIG, "warp_perspective: canvas taller than 2 M rows");
  GlobalWarpParams p;
  p.src = src; p.base = base; p.dst = dst;
  for (int k = 0; k < 9; ++k) p.m[k] = minv[k];
  p.src_h = src_h; p.src_w = src_w; p.dst_h = dst_h; p.dst_w = dst_w; p.base_h = base_h; p.base_w = base_w;
  p.off_x = off_x; p.off_y = off_y; p.mode = base ? mode : 0;
  const int bh0 = dst_h < 16 ? dst_h : 16;         // WarpPerspectiveInvoker: BLOCK_SZ = 32
  int bw0 = 1024 / bh0;
  if (bw0 > dst_w) bw0 = dst_w;
  p.bw0 = bw0;
  k_warp_global<<<dim3((dst_w + kTileW - 1) / kTileW, (dst_h + kTileH - 1) / kTileH), 256, 0, st>>>(p);
  return check_cuda(cudaGetLastError(), "k_warp_global launch");
}

}  // namespace apap

using namespace apap;

extern "C" int apap_warp_perspective(const uint8_t *src, int src_h, int src_w, const double *inverse_map, uint8_t *dst,
                                     int dst_h, int dst_w, const uint8_t *base, int base_h, int base_w, int off_x,
                                     int off_y, int mode, void *stream) {
  if (!src || !inverse_map || !dst) return fail(APAP_E_BADARG, "warp_perspective: null pointer");
  if (src_h <= 0 || src_w <= 0 || dst_h < 0 || dst_w < 0 || mode < 0 || mode > 2)
    return fail(APAP_E_BADARG, "warp_perspective: bad sizes or mode");
  if (src_h > 32767 || src_w > 32767) return fail(APAP_E_TOOBIG, "warp_perspective: source larger than 32767 (OpenCV's own limit)");
  if (base && (base_h <= 0 || base_w <= 0)) return fail(APAP_E_BADARG, "warp_perspective: bad base image size");
  return launch_warp_global(src, src_h, src_w, inverse_map, dst, dst_h, dst_w, base, base_h, base_w, off_x, off_y, mode,
                            static_cast<cudaStream_t>(stream));
}
