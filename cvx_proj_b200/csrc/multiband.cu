// Multi-band blend of N placed layers (utils.multiband_blend, driver.stitch_panorama(blend="multiband")): bit for bit
// cv.detail.MultiBandBlender(0, bands, CV_16S) fed every layer pasted into the whole canvas, converted to uint8 with
// saturation (DESIGN.md section 3).  nb = min(bands, ceil(log2(max(W, H)))), the pyramids live on Wp x Hp (W, H
// rounded up to multiples of 2^nb).  Per layer k: X_0 = P_k with a BORDER_REFLECT pad, G_0 = 256 on its non-empty
// pixels (any channel > 0) and 0 elsewhere and in the pad; X_{i+1} = pyrDown(X_i), G_{i+1} = pyrDown(G_i) ([1 4 6 4 1],
// reflect-101, (s + 128) >> 8).  Per level i: L = X_i - pyrUp(X_{i+1}) (L_nb = X_nb), band_i += (L G_i) >> 8,
// wsum_i += G_i; V_i = trunc((band_i << 8) / (wsum_i + 1)); R_nb = V_nb, R_i = mb_sat16(pyrUp(R_{i+1}) + V_i); the output
// is R_0 clipped to [0, 255], 0 where wsum_0 = 0.  All integer: the result does not depend on the layer order.
//
// At most APAP_MULTIBAND_MAX_LAYERS = 127 layers: |L| <= 255 and G <= 256, so |band| <= 127 x 255 and wsum <= 127 x
// 256 both fit int16, where OpenCV keeps them; the kernels' int32 sums are then OpenCV's without emulating a wrap.
//
// Windows: layer k's pyramids are stored only on a box per level that holds every non-zero value of X_{k,i} and
// G_{k,i}.  Level 0: its clipped rectangle, extended to the pad's end on an axis where the reflected pad picks up
// some of it; level i + 1: [floor((a - 1) / 2), floor((b + 1) / 2) + 1) of level i's [a, b), clipped -- pyrDown's
// output j reads inputs 2j - 2 .. 2j + 2 only, its reflect-101 edge included.  Outside its box a level is exactly 0,
// so a read outside returns 0 and every stored value is the full-canvas one; where G_{k,i} = 0 the layer adds exactly
// (L 0) >> 8 = 0 and 0, so a pixel skips layers whose box (level 0: rectangle) misses its tile.
//
// Kernels, each a 32 x 8 pixel tile per CTA, one pixel per thread:
//   k_mb_down<kLevel0, kGains>  one launch per level i < nb for all layers (grid z = layer): X_{i+1} and G_{i+1} as
//                               int16 {b, g, r, w} on the level i + 1 box.  Level 0 is never stored: it is read from
//                               the layer bytes (the zero paste, the reflect pad, the weight from the raw bytes,
//                               kGains: the bytes through the layer's exposure-gain table lut[k][256], kChannels:
//                               through its per-channel table lut[k][3][256]).
//   k_mb_band<kLevel0, kTop, kGains>  one launch per level, nb down to 0: per pixel the layers' L, G summed in int32
//                               registers (the per-layer Laplacians never leave the SM), normalised, pyrUp(R_{i+1})
//                               added; R_i (i >= 1) is stored on the full level as int16 {b, g, r, 0}, level 0
//                               writes the cropped, masked, saturated uint8 canvas.
#include <algorithm>
#include <vector>

#include "layers.cuh"

namespace apap {

constexpr int kMbTileX = 32, kMbTileY = 8;

struct MbWin {
  short4 *p;                                      // w x h values, row pitch w; {b, g, r, weight}
  int x0, y0, w, h;                               // box on its level (w = h = 0: the layer is absent)
};

struct MbParams {
  LayerDesc layer[APAP_MULTIBAND_MAX_LAYERS];
  int4 rect[APAP_MULTIBAND_MAX_LAYERS];           // clipped rectangle [x0, x1) x [y0, y1) on the canvas
  MbWin lo[APAP_MULTIBAND_MAX_LAYERS];            // level i
  MbWin hi[APAP_MULTIBAND_MAX_LAYERS];            // level i + 1
  const uint8_t *lut;                             // [n_layers][256] (kGains), [n_layers][3][256] (kChannels)
  short4 *r_lo;                                   // R_i (k_mb_band, i >= 1), full level, row pitch lw
  const short4 *r_hi;                             // R_{i+1}, row pitch hw
  uint8_t *out;
  int n_layers, canvas_w, canvas_h, wp, hp;       // the canvas and its padded size
  int lw, lh, hw, hh;                             // sizes of levels i and i + 1
};

__device__ __forceinline__ int mb_sat16(int v) { return min(max(v, -32768), 32767); }

// BORDER_REFLECT_101 for the pyrDown taps (i in [-2, n], n >= 2): at n = 2, -2 reflects to 2 and on to 0
__device__ __forceinline__ int mb_reflect101(int i, int n) {
  i = i < 0 ? -i : i;
  return i >= n ? 2 * n - 2 - i : i;
}

// BORDER_REFLECT of the pad: period 2n, the edge pixel repeated (i >= 0)
__device__ __forceinline__ int mb_reflect_pad(int i, int n) {
  const int m = i % (2 * n);
  return m >= n ? 2 * n - 1 - m : m;
}

// level 0 of layer l at padded position (x, y): X_0 {b, g, r} and G_0 in .w
template <bool kGains, bool kChannels>
__device__ __forceinline__ int4 mb_level0(const MbParams &p, int l, int x, int y) {
  const int4 R = p.rect[l];
  const bool in_canvas = x < p.canvas_w && y < p.canvas_h;
  const int cx = mb_reflect_pad(x, p.canvas_w), cy = mb_reflect_pad(y, p.canvas_h);
  if (cx < R.x || cx >= R.z || cy < R.y || cy >= R.w) return make_int4(0, 0, 0, 0);
  const LayerDesc &L = p.layer[l];
  const uint8_t *q = L.addr + (long long)(cy - L.y0) * L.pitch + 3LL * (cx - L.x0);
  int b = __ldg(q), g = __ldg(q + 1), r = __ldg(q + 2);
  const int w = in_canvas && (b | g | r) ? 256 : 0;
  if constexpr (kGains && kChannels) {
    const uint8_t *lut = p.lut + 768 * l;
    b = __ldg(lut + b);
    g = __ldg(lut + 256 + g);
    r = __ldg(lut + 512 + r);
  } else if constexpr (kGains) {
    const uint8_t *lut = p.lut + 256 * l;
    b = __ldg(lut + b);
    g = __ldg(lut + g);
    r = __ldg(lut + r);
  }
  return make_int4(b, g, r, w);
}

// a stored box value at level position (x, y), 0 outside the box
__device__ __forceinline__ int4 mb_win_at(const MbWin &W, int x, int y) {
  x -= W.x0;
  y -= W.y0;
  if ((unsigned)x >= (unsigned)W.w || (unsigned)y >= (unsigned)W.h) return make_int4(0, 0, 0, 0);
  const short4 v = W.p[(size_t)y * (size_t)W.w + x];
  return make_int4(v.x, v.y, v.z, v.w);
}

// pyrUp taps along one axis for output o of a level of n: out[2j] = s[j-1] + 6 s[j] + s[j+1], out[2j+1] = 4 (s[j] +
// s[j+1]); s[-1] = s[1], s[n] = s[n-1]
__device__ __forceinline__ int mb_up_taps(int o, int n, int (&idx)[3], int (&wt)[3]) {
  const int j = o >> 1;
  const int nx = min(j + 1, n - 1);
  if (o & 1) {
    idx[0] = j; wt[0] = 4;
    idx[1] = nx; wt[1] = 4;
    return 2;
  }
  idx[0] = j > 0 ? j - 1 : min(1, n - 1); wt[0] = 1;
  idx[1] = j; wt[1] = 6;
  idx[2] = nx; wt[2] = 1;
  return 3;
}

// pyrUp of a stored box (0 outside it) at output (x, y): {b, g, r}, saturated
__device__ __forceinline__ int3 mb_up_win(const MbWin &W, int n_x, int n_y, int x, int y) {
  int ix[3], wx[3], iy[3], wy[3];
  const int nx = mb_up_taps(x, n_x, ix, wx), ny = mb_up_taps(y, n_y, iy, wy);
  int t0 = 0, t1 = 0, t2 = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (a >= ny) break;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      if (c >= nx) break;
      const int4 v = mb_win_at(W, ix[c], iy[a]);
      const int w = wy[a] * wx[c];
      t0 += w * v.x;
      t1 += w * v.y;
      t2 += w * v.z;
    }
  }
  return make_int3(mb_sat16((t0 + 32) >> 6), mb_sat16((t1 + 32) >> 6), mb_sat16((t2 + 32) >> 6));
}

// pyrUp of a full level (row pitch n_x) at output (x, y)
__device__ __forceinline__ int3 mb_up_full(const short4 *__restrict__ s, int n_x, int n_y, int x, int y) {
  int ix[3], wx[3], iy[3], wy[3];
  const int nx = mb_up_taps(x, n_x, ix, wx), ny = mb_up_taps(y, n_y, iy, wy);
  int t0 = 0, t1 = 0, t2 = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (a >= ny) break;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      if (c >= nx) break;
      const short4 v = s[(size_t)iy[a] * (size_t)n_x + ix[c]];
      const int w = wy[a] * wx[c];
      t0 += w * v.x;
      t1 += w * v.y;
      t2 += w * v.z;
    }
  }
  return make_int3(mb_sat16((t0 + 32) >> 6), mb_sat16((t1 + 32) >> 6), mb_sat16((t2 + 32) >> 6));
}

template <bool kLevel0, bool kGains, bool kChannels>
__global__ void __launch_bounds__(kMbTileX *kMbTileY) k_mb_down(const __grid_constant__ MbParams p) {
  const int l = blockIdx.z;
  const MbWin &D = p.hi[l];
  const int ox = blockIdx.x * kMbTileX + threadIdx.x, oy = blockIdx.y * kMbTileY + threadIdx.y;
  if (ox >= D.w || oy >= D.h) return;
  const int x = D.x0 + ox, y = D.y0 + oy;                       // level i + 1 position
  constexpr int taps[5] = {1, 4, 6, 4, 1};
  int ix[5], iy[5];
#pragma unroll
  for (int d = 0; d < 5; ++d) {
    ix[d] = mb_reflect101(2 * x + d - 2, p.lw);
    iy[d] = mb_reflect101(2 * y + d - 2, p.lh);
  }
  int s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll
  for (int a = 0; a < 5; ++a) {
#pragma unroll
    for (int c = 0; c < 5; ++c) {
      int4 v;
      if constexpr (kLevel0) v = mb_level0<kGains, kChannels>(p, l, ix[c], iy[a]);
      else v = mb_win_at(p.lo[l], ix[c], iy[a]);
      const int w = taps[a] * taps[c];
      s0 += w * v.x;
      s1 += w * v.y;
      s2 += w * v.z;
      s3 += w * v.w;
    }
  }
  D.p[(size_t)oy * (size_t)D.w + ox] = make_short4((short)mb_sat16((s0 + 128) >> 8), (short)mb_sat16((s1 + 128) >> 8),
                                                   (short)mb_sat16((s2 + 128) >> 8), (short)mb_sat16((s3 + 128) >> 8));
}

template <bool kLevel0, bool kTop, bool kGains, bool kChannels>
__global__ void __launch_bounds__(kMbTileX *kMbTileY) k_mb_band(const __grid_constant__ MbParams p) {
  const int tx0 = blockIdx.x * kMbTileX, ty0 = blockIdx.y * kMbTileY;
  const int x = tx0 + threadIdx.x, y = ty0 + threadIdx.y;
  const int n_x = kLevel0 ? p.canvas_w : p.lw, n_y = kLevel0 ? p.canvas_h : p.lh;   // pixels this level writes
  const bool active = x < n_x && y < n_y;
  int acc0 = 0, acc1 = 0, acc2 = 0, wsum = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    int bx0, by0, bx1, by1;                                     // where G_{l,i} may be non-zero
    if constexpr (kLevel0) {
      const int4 R = p.rect[l];
      bx0 = R.x; by0 = R.y; bx1 = R.z; by1 = R.w;
    } else {
      const MbWin &W = p.lo[l];
      bx0 = W.x0; by0 = W.y0; bx1 = W.x0 + W.w; by1 = W.y0 + W.h;
    }
    if (bx1 <= tx0 || bx0 >= tx0 + kMbTileX || by1 <= ty0 || by0 >= ty0 + kMbTileY) continue;   // uniform
    if (!active || x < bx0 || x >= bx1 || y < by0 || y >= by1) continue;
    int4 v;
    if constexpr (kLevel0) v = mb_level0<kGains, kChannels>(p, l, x, y);
    else v = mb_win_at(p.lo[l], x, y);
    if (v.w == 0) continue;
    if constexpr (!kTop) {
      const int3 u = mb_up_win(p.hi[l], p.hw, p.hh, x, y);
      v.x = mb_sat16(v.x - u.x);
      v.y = mb_sat16(v.y - u.y);
      v.z = mb_sat16(v.z - u.z);
    }
    acc0 += (v.x * v.w) >> 8;
    acc1 += (v.y * v.w) >> 8;
    acc2 += (v.z * v.w) >> 8;
    wsum += v.w;
  }
  if (!active) return;
  // each term has |(L G) >> 8| <= ceil(255 G / 256) <= G (the floor shift of a negative L rounds away from 0), so
  // |acc| <= wsum and |acc 256 / (wsum + 1)| < 256: the quotient fits int16, as OpenCV's (short) cast of it
  int r0 = (acc0 * 256) / (wsum + 1), r1 = (acc1 * 256) / (wsum + 1), r2 = (acc2 * 256) / (wsum + 1);
  if constexpr (!kTop) {
    const int3 u = mb_up_full(p.r_hi, p.hw, p.hh, x, y);
    r0 = mb_sat16(u.x + r0);
    r1 = mb_sat16(u.y + r1);
    r2 = mb_sat16(u.z + r2);
  }
  if constexpr (kLevel0) {
    uint8_t *o = p.out + ((size_t)y * (size_t)p.canvas_w + x) * 3;
    const bool on = wsum > 0;
    o[0] = on ? (uint8_t)min(max(r0, 0), 255) : 0;
    o[1] = on ? (uint8_t)min(max(r1, 0), 255) : 0;
    o[2] = on ? (uint8_t)min(max(r2, 0), 255) : 0;
  } else {
    p.r_lo[(size_t)y * (size_t)p.lw + x] = make_short4((short)r0, (short)r1, (short)r2, 0);
  }
}

namespace {

// Host plan: level sizes and boxes, their buffers carved from the workspace at `base` (16-byte aligned each; base =
// nullptr only sizes them).
struct MbPlan {
  int nb, wp, hp;
  std::vector<int4> rect;                         // per layer
  std::vector<MbWin> win;                         // [layer][level 0 .. nb]; level 0 is never stored (p = nullptr)
  std::vector<short4 *> r;                        // R_i, i = 1 .. nb (index i)
  size_t bytes;
};

size_t mb_align(size_t b) { return (b + 15) & ~(size_t)15; }

// level 0's box along one axis: the clipped [c0, c1) of a canvas of n padded to np, extended to np when the
// BORDER_REFLECT pad [n, np) repeats one of its pixels (the pad holds [2n - np, n) reflected, or all of [0, n) once
// np - n >= n)
void pad_extent(int c0, int c1, int n, int np, int &a, int &b) {
  a = c0;
  b = c1;
  if (np > n && (np - n >= n || c1 > 2 * n - np)) b = np;
}

// ceil(log2(v)) for v >= 1: MultiBandBlender::prepare's cap ceil(log(max(W, H)) / log(2.0)) for every v <= 2^30
int ceil_log2(int v) { return v <= 1 ? 0 : 32 - __builtin_clz((unsigned)(v - 1)); }

void mb_plan(const long long *layers, int n_layers, int canvas_h, int canvas_w, int bands, uint8_t *base, MbPlan &P) {
  P.nb = std::min(bands, ceil_log2(std::max(canvas_w, canvas_h)));
  const long long A = 1LL << P.nb;
  P.wp = (int)((canvas_w + A - 1) / A * A);
  P.hp = (int)((canvas_h + A - 1) / A * A);
  P.rect.assign(n_layers, make_int4(0, 0, 0, 0));
  P.win.assign((size_t)n_layers * (P.nb + 1), MbWin{nullptr, 0, 0, 0, 0});
  P.r.assign(P.nb + 1, nullptr);
  size_t used = 0;
  for (int l = 0; l < n_layers; ++l) {
    const LayerDesc L = layer_desc(layers + 6 * l);
    const long long x0 = std::max(0LL, (long long)L.x0), y0 = std::max(0LL, (long long)L.y0);
    const long long x1 = std::min((long long)canvas_w, (long long)L.x0 + L.w);
    const long long y1 = std::min((long long)canvas_h, (long long)L.y0 + L.h);
    if (x1 <= x0 || y1 <= y0) continue;           // outside the canvas: absent at every level
    P.rect[l] = make_int4((int)x0, (int)y0, (int)x1, (int)y1);
    int ax, bx, ay, by;
    pad_extent((int)x0, (int)x1, canvas_w, P.wp, ax, bx);
    pad_extent((int)y0, (int)y1, canvas_h, P.hp, ay, by);
    MbWin *w = &P.win[(size_t)l * (P.nb + 1)];
    w[0] = MbWin{nullptr, ax, ay, bx - ax, by - ay};
    for (int i = 1; i <= P.nb; ++i) {
      const MbWin &u = w[i - 1];
      const int a_x = std::max(0, (u.x0 - 1) >> 1), b_x = std::min(P.wp >> i, ((u.x0 + u.w + 1) >> 1) + 1);
      const int a_y = std::max(0, (u.y0 - 1) >> 1), b_y = std::min(P.hp >> i, ((u.y0 + u.h + 1) >> 1) + 1);
      w[i] = MbWin{reinterpret_cast<short4 *>(base + used), a_x, a_y, b_x - a_x, b_y - a_y};
      used += mb_align((size_t)w[i].w * (size_t)w[i].h * sizeof(short4));
    }
  }
  for (int i = 1; i <= P.nb; ++i) {
    P.r[i] = reinterpret_cast<short4 *>(base + used);
    used += mb_align((size_t)(P.wp >> i) * (size_t)(P.hp >> i) * sizeof(short4));
  }
  P.bytes = used;
}

int mb_fail(int code, const char *what, const char *err) {
  char msg[160];
  snprintf(msg, sizeof(msg), "%s: %s", what, err);
  return fail(code, msg);
}

int mb_check(const char *what, const long long *layers, int n_layers, int canvas_h, int canvas_w, int bands) {
  if (!layers) return mb_fail(APAP_E_BADARG, what, "null pointer");
  if (int rc = check_layer_count_canvas(what, n_layers, APAP_MULTIBAND_MAX_LAYERS, "APAP_MULTIBAND_MAX_LAYERS",
                                        canvas_h, canvas_w))
    return rc;
  if (int rc = check_layer_descs(what, layers, n_layers)) return rc;
  if (bands < 0) return mb_fail(APAP_E_BADARG, what, "bands must be >= 0");
  // the band kernels' grid y counts the 8-row tiles of a level
  if ((canvas_h + kMbTileY - 1) / kMbTileY > 65535) return mb_fail(APAP_E_TOOBIG, what, "canvas_h above 524280");
  return 0;
}

template <bool kGains, bool kChannels>
int mb_launch(const MbPlan &P, MbParams &p, cudaStream_t st) {
  const int nb = P.nb;
  const dim3 block(kMbTileX, kMbTileY);
  // p.lo / p.hi = the boxes of levels i / i + 1 (none above nb)
  auto bind = [&](int i) {
    for (int l = 0; l < p.n_layers; ++l) {
      p.lo[l] = P.win[(size_t)l * (nb + 1) + i];
      p.hi[l] = i < nb ? P.win[(size_t)l * (nb + 1) + i + 1] : MbWin{nullptr, 0, 0, 0, 0};
    }
    p.lw = P.wp >> i;
    p.lh = P.hp >> i;
    p.hw = i < nb ? P.wp >> (i + 1) : 0;
    p.hh = i < nb ? P.hp >> (i + 1) : 0;
  };
  for (int i = 0; i < nb; ++i) {
    bind(i);
    int mw = 0, mh = 0;
    for (int l = 0; l < p.n_layers; ++l) {
      mw = std::max(mw, p.hi[l].w);
      mh = std::max(mh, p.hi[l].h);
    }
    if (mw == 0) break;                           // every layer lies outside the canvas
    const dim3 grid((unsigned)((mw + kMbTileX - 1) / kMbTileX), (unsigned)((mh + kMbTileY - 1) / kMbTileY),
                    (unsigned)p.n_layers);
    if (i == 0) k_mb_down<true, kGains, kChannels><<<grid, block, 0, st>>>(p);
    else k_mb_down<false, false, false><<<grid, block, 0, st>>>(p);
    if (int rc = check_cuda(cudaGetLastError(), "k_mb_down launch")) return rc;
  }
  for (int i = nb; i >= 0; --i) {
    bind(i);
    p.r_lo = P.r[i];
    p.r_hi = i < nb ? P.r[i + 1] : nullptr;
    const int n_x = i == 0 ? p.canvas_w : p.lw, n_y = i == 0 ? p.canvas_h : p.lh;
    const dim3 grid((unsigned)((n_x + kMbTileX - 1) / kMbTileX), (unsigned)((n_y + kMbTileY - 1) / kMbTileY));
    if (i == 0 && nb == 0) k_mb_band<true, true, kGains, kChannels><<<grid, block, 0, st>>>(p);
    else if (i == 0) k_mb_band<true, false, kGains, kChannels><<<grid, block, 0, st>>>(p);
    else if (i == nb) k_mb_band<false, true, false, false><<<grid, block, 0, st>>>(p);
    else k_mb_band<false, false, false, false><<<grid, block, 0, st>>>(p);
    if (int rc = check_cuda(cudaGetLastError(), "k_mb_band launch")) return rc;
  }
  return 0;
}

// lut: none (nullptr), [n][256] or (channels) [n][3][256]
int multiband_blend(const char *what, const long long *layers, int n_layers, int canvas_h, int canvas_w, int bands,
                    const uint8_t *lut, bool channels, void *workspace, size_t workspace_bytes, uint8_t *out, size_t out_bytes,
                    cudaStream_t st) {
  if (!out || !workspace) return mb_fail(APAP_E_BADARG, what, "null pointer");
  if (int rc = mb_check(what, layers, n_layers, canvas_h, canvas_w, bands)) return rc;
  if (out_bytes < (size_t)canvas_h * (size_t)canvas_w * 3)
    return mb_fail(APAP_E_BADARG, what, "out is smaller than canvas_h x canvas_w x 3 bytes");
  if (reinterpret_cast<uintptr_t>(workspace) & 15u) return mb_fail(APAP_E_ALIGN, what, "workspace must be 16-byte aligned");
  MbPlan P;
  mb_plan(layers, n_layers, canvas_h, canvas_w, bands, static_cast<uint8_t *>(workspace), P);
  if (workspace_bytes < P.bytes)
    return mb_fail(APAP_E_BADARG, what, "workspace is smaller than apap_multiband_workspace_bytes");
  MbParams p;
  for (int l = 0; l < n_layers; ++l) {
    p.layer[l] = layer_desc(layers + 6 * l);
    p.rect[l] = P.rect[l];
  }
  p.lut = lut;
  p.out = out;
  p.n_layers = n_layers;
  p.canvas_w = canvas_w;
  p.canvas_h = canvas_h;
  p.wp = P.wp;
  p.hp = P.hp;
  if (lut && channels) return mb_launch<true, true>(P, p, st);
  return lut ? mb_launch<true, false>(P, p, st) : mb_launch<false, false>(P, p, st);
}

}  // namespace
}  // namespace apap

using namespace apap;

extern "C" int apap_multiband_workspace_bytes(const long long *layers, int n_layers, int canvas_h, int canvas_w,
                                              int bands, size_t *bytes) {
  if (!bytes) return mb_fail(APAP_E_BADARG, "multiband", "null pointer");
  if (int rc = mb_check("multiband", layers, n_layers, canvas_h, canvas_w, bands)) return rc;
  MbPlan P;
  mb_plan(layers, n_layers, canvas_h, canvas_w, bands, nullptr, P);
  *bytes = P.bytes;
  return 0;
}

extern "C" int apap_multiband_blend(const long long *layers, int n_layers, int canvas_h, int canvas_w, int bands,
                                    void *workspace, size_t workspace_bytes, uint8_t *out, size_t out_bytes,
                                    void *stream) {
  return multiband_blend("multiband_blend", layers, n_layers, canvas_h, canvas_w, bands, nullptr, false, workspace,
                         workspace_bytes, out, out_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int apap_multiband_blend_gain(const long long *layers, int n_layers, int canvas_h, int canvas_w, int bands,
                                         const uint8_t *lut, void *workspace, size_t workspace_bytes, uint8_t *out,
                                         size_t out_bytes, void *stream) {
  if (!lut) return fail(APAP_E_BADARG, "multiband_blend_gain: null gain table");
  return multiband_blend("multiband_blend_gain", layers, n_layers, canvas_h, canvas_w, bands, lut, false, workspace,
                         workspace_bytes, out, out_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int apap_multiband_blend_channels(const long long *layers, int n_layers, int canvas_h, int canvas_w,
                                             int bands, const uint8_t *lut, void *workspace, size_t workspace_bytes,
                                             uint8_t *out, size_t out_bytes, void *stream) {
  if (!lut) return fail(APAP_E_BADARG, "multiband_blend_channels: null gain table");
  return multiband_blend("multiband_blend_channels", layers, n_layers, canvas_h, canvas_w, bands, lut, true,
                         workspace, workspace_bytes, out, out_bytes, static_cast<cudaStream_t>(stream));
}
