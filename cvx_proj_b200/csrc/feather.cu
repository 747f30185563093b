// Feather blend of N placed layers (utils.feather_blend, driver.stitch_panorama(blend="feather")): bit for bit
// cv.detail.FeatherBlender(s) fed every layer pasted into the whole canvas (DESIGN.md section 3).  Per layer k and
// canvas pixel, D_k = the L1 distance to the nearest empty pixel of the pasted layer (any channel > 0 is non-empty;
// the canvas border is not empty), w_k = min(fl(D_k s), 1); acc += trunc(v_k w_k) per channel and wsum += w_k in
// layer order; out = trunc(acc / (wsum + 1e-5)), 0 where wsum <= 1e-5.
//
// Three kernels over one workspace of uint16 distances, one ch x cw block per layer for its rectangle clipped to the
// canvas [cx0, cx0 + cw) x [cy0, cy0 + ch):
//   k_feather_rows  one CTA per (layer, clipped row): the horizontal distance to the nearest empty pixel of the row,
//                   reading the layer bytes through layers.cuh's fetch_group (the mask is never stored).  A forward
//                   sweep over 1024-pixel tiles carries the last empty column (block max-scan), a backward sweep over
//                   the stored values the next one (block min-scan).  The pixel just left / right of the clipped row
//                   is empty when it lies inside the canvas.
//   k_feather_cols  one CTA per (layer, 32 columns), 8 row segments per column: each thread summarises its segment
//                   (the values a downward and an upward min(h, prev + 1) scan leave at its ends), the segments
//                   exchange those in shared memory, then each thread scans its segment down and up with the carries.
//   k_feather_blend one CTA per kSegPx-pixel canvas row segment, 4 pixels per thread (layers.cuh): a layer that does
//                   not cover the segment adds exactly +0.0f and 0 and is skipped (uniform test).  kGains
//                   (apap_feather_blend_gain): layer l's bytes go through its exposure-gain table lut[l][256]
//                   first; the distances, made from the raw bytes, are unchanged.
// Distances are stored as min(D, cap) (apap_feather_distance_cap): cap is either the smallest integer with
// fl(cap s) >= 1 -- float multiplication by s > 0 is monotone, so every D >= cap has weight 1 -- or, when that is
// larger, W + H - 1, more than any finite distance in the canvas, so that only a layer with no empty pixel in the
// canvas stores cap; the blend gives D = cap weight 1 in both cases, which is OpenCV's min(fl(FLT_MAX s), 1) for
// every s >= FLT_MIN (smaller, subnormal s are refused).  min-plus scans of capped values give min(D, cap)
// again.  The arithmetic is written with _rn / _rz intrinsics: a contracted FMA would change the bits.
#include <cfloat>
#include <cmath>

#include "layers.cuh"

namespace apap {

constexpr int kColThreadsX = 32;        // columns per k_feather_cols CTA
constexpr int kColSegs = 8;             // row segments per column
constexpr int kFar = 1 << 30;           // farther than any distance; kFar + a canvas extent stays below 2^31
constexpr int kNoneRight = 0x7fffffff;  // no empty column to the right (minus a column index stays >= 0)

struct FeatherRect {
  uint16_t *dist;                       // ch x cw distances, row pitch cw
  int cx0, cy0, cw, ch;                 // the layer's rectangle clipped to the canvas (cw = ch = 0: outside it)
};

struct FeatherParams {
  LayerDesc layer[APAP_FEATHER_MAX_LAYERS];
  FeatherRect rect[APAP_FEATHER_MAX_LAYERS];
  uint8_t *out;
  float s;
  int n_layers, canvas_h, canvas_w, segs_per_row, cap;
};

// exclusive block scans over the 256 threads of k_feather_rows: the max of v over lower threads / the min of v over
// higher threads, and the value over all threads; red[] holds one value per warp
__device__ __forceinline__ int prefix_max(int v, int *red, int &all) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc = max(inc, u);
  }
  if (lane == 31) red[warp] = inc;
  __syncthreads();
  int ex = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) ex = -kFar;
  all = -kFar;
#pragma unroll
  for (int k = 0; k < kLayerThreads / 32; ++k) {
    if (k < warp) ex = max(ex, red[k]);
    all = max(all, red[k]);
  }
  __syncthreads();                      // red[] is free again
  return ex;
}

__device__ __forceinline__ int suffix_min(int v, int *red, int &all) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_down_sync(0xffffffffu, inc, o);
    if (lane + o < 32) inc = min(inc, u);
  }
  if (lane == 0) red[warp] = inc;
  __syncthreads();
  int ex = __shfl_down_sync(0xffffffffu, inc, 1);
  if (lane == 31) ex = kNoneRight;
  all = kNoneRight;
#pragma unroll
  for (int k = 0; k < kLayerThreads / 32; ++k) {
    if (k > warp) ex = min(ex, red[k]);
    all = min(all, red[k]);
  }
  __syncthreads();
  return ex;
}

__global__ void __launch_bounds__(kLayerThreads) k_feather_rows(const __grid_constant__ FeatherParams p) {
  __shared__ int red[kLayerThreads / 32];
  const FeatherRect &R = p.rect[blockIdx.y];
  const int r = blockIdx.x;
  if (r >= R.ch) return;                // uniform
  const int y = R.cy0 + r, x_end = R.cx0 + R.cw;
  uint16_t *row = R.dist + (size_t)r * (size_t)R.cw;
  const int n_tiles = (R.cw + kSegPx - 1) / kSegPx;

  // forward: distance to the nearest empty column at or left of each pixel
  int last = R.cx0 > 0 ? R.cx0 - 1 : -kFar;
  for (int t = 0; t < n_tiles; ++t) {
    const int seg0 = R.cx0 + t * kSegPx;
    const int seg_px = min(kSegPx, x_end - seg0);
    const int x = seg0 + kLayerGroupPx * (int)threadIdx.x;
    const int n_px = min(kLayerGroupPx, x_end - x);
    uint32_t w[3];
    fetch_group(p.layer[blockIdx.y], y, seg0, seg_px, x, n_px, w);
    const uint32_t nz = byte_nonzero(group_or(w[0], w[1], w[2]));
    int mine = -kFar;
#pragma unroll
    for (int k = 0; k < kLayerGroupPx; ++k)
      if (k < n_px && !((nz >> (8 * k)) & 1u)) mine = x + k;
    int all;
    int l = max(last, prefix_max(mine, red, all));
    last = max(last, all);
#pragma unroll
    for (int k = 0; k < kLayerGroupPx; ++k) {
      if (k < n_px) {
        if (!((nz >> (8 * k)) & 1u)) l = x + k;
        row[x + k - R.cx0] = (uint16_t)min(x + k - l, p.cap);
      }
    }
  }
  // backward: the nearest empty column at or right of each pixel (stored 0 = empty; each thread rereads its own pixels)
  int next = x_end < p.canvas_w ? x_end : kNoneRight;
  for (int t = n_tiles - 1; t >= 0; --t) {
    const int x = R.cx0 + t * kSegPx + kLayerGroupPx * (int)threadIdx.x;
    const int n_px = min(kLayerGroupPx, x_end - x);
    int d[kLayerGroupPx];
    int mine = kNoneRight;
#pragma unroll
    for (int k = kLayerGroupPx - 1; k >= 0; --k) {
      d[k] = k < n_px ? row[x + k - R.cx0] : 1;
      if (d[k] == 0) mine = x + k;
    }
    int all;
    int n = min(next, suffix_min(mine, red, all));
    next = min(next, all);
#pragma unroll
    for (int k = kLayerGroupPx - 1; k >= 0; --k) {
      if (k < n_px) {
        if (d[k] == 0) n = x + k;
        row[x + k - R.cx0] = (uint16_t)min(d[k], n - (x + k));
      }
    }
  }
}

__global__ void __launch_bounds__(kColThreadsX * kColSegs) k_feather_cols(const __grid_constant__ FeatherParams p) {
  __shared__ int down_end[kColSegs][kColThreadsX], up_end[kColSegs][kColThreadsX];
  const FeatherRect &R = p.rect[blockIdx.y];
  const int c = blockIdx.x * kColThreadsX + threadIdx.x, seg = threadIdx.y;
  if ((int)blockIdx.x * kColThreadsX >= R.cw) return;            // uniform
  const bool active = c < R.cw;
  const int seg_rows = (R.ch + kColSegs - 1) / kColSegs;
  const int r0 = min(R.ch, seg * seg_rows), r1 = min(R.ch, r0 + seg_rows);
  uint16_t *col = R.dist + c;
  const size_t pitch = (size_t)R.cw;

  // the segment on its own: the downward scan's value at row r1 - 1 and the upward scan's at row r0
  int dn = kFar, up = kFar;
  if (active) {
#pragma unroll 8
    for (int r = r0; r < r1; ++r) {
      const int h = col[r * pitch];
      dn = min(dn + 1, h);
      up = min(up, h + (r - r0));
    }
  }
  down_end[seg][threadIdx.x] = dn;
  up_end[seg][threadIdx.x] = up;
  __syncthreads();
  if (!active || r0 >= r1) return;
  // carries: the downward scan's value at row r0 - 1 and the upward scan's at row r1 (the row just above / below the
  // clipped rectangle is empty when it lies inside the canvas)
  int din = R.cy0 > 0 ? r0 : kFar;
  int uin = R.cy0 + R.ch < p.canvas_h ? R.ch - r1 : kFar;
  for (int k = 0; k < kColSegs; ++k) {
    const int k0 = min(R.ch, k * seg_rows), k1 = min(R.ch, k0 + seg_rows);
    if (k1 <= k0) continue;
    if (k < seg) din = min(din, down_end[k][threadIdx.x] + (r0 - k1));
    if (k > seg) uin = min(uin, up_end[k][threadIdx.x] + (k0 - r1));
  }
#pragma unroll 8
  for (int r = r0; r < r1; ++r) {
    din = min(din + 1, (int)col[r * pitch]);
    col[r * pitch] = (uint16_t)min(din, p.cap);
  }
#pragma unroll 8
  for (int r = r1 - 1; r >= r0; --r) {
    uin = min(uin + 1, (int)col[r * pitch]);
    col[r * pitch] = (uint16_t)min(uin, p.cap);
  }
}

template <bool kGains>
__global__ void __launch_bounds__(kLayerThreads) k_feather_blend(const __grid_constant__ FeatherParams p,
                                                                 const uint8_t *__restrict__ lut) {
  __shared__ __align__(16) uint32_t stage[kSegBytes / 4];
  const int y = blockIdx.x / p.segs_per_row;
  const int seg0 = (blockIdx.x - y * p.segs_per_row) * kSegPx;
  const int seg_px = min(kSegPx, p.canvas_w - seg0);
  const int x = seg0 + kLayerGroupPx * (int)threadIdx.x;
  const int n_px = min(kLayerGroupPx, p.canvas_w - x);          // pixels of this thread (<= 0: none)

  int acc[3 * kLayerGroupPx];
  float wsum[kLayerGroupPx];
#pragma unroll
  for (int b = 0; b < 3 * kLayerGroupPx; ++b) acc[b] = 0;
#pragma unroll
  for (int k = 0; k < kLayerGroupPx; ++k) wsum[k] = 0.f;
  for (int l = 0; l < p.n_layers; ++l) {
    const FeatherRect &R = p.rect[l];
    const int r = y - R.cy0;
    if ((unsigned)r >= (unsigned)R.ch || seg0 + seg_px <= R.cx0 || seg0 >= R.cx0 + R.cw) continue;   // uniform
    uint32_t v[3];
    fetch_group(p.layer[l], y, seg0, seg_px, x, n_px, v);
    if constexpr (kGains) gain_group(lut + 256 * l, v);
    const uint16_t *row = R.dist + (size_t)r * (size_t)R.cw;
#pragma unroll
    for (int k = 0; k < kLayerGroupPx; ++k) {
      const int lx = x + k - R.cx0;
      float wk = 0.f;
      if (k < n_px && (unsigned)lx < (unsigned)R.cw) {
        const int d = row[lx];
        wk = d >= p.cap ? 1.f : fminf(__fmul_rn((float)d, p.s), 1.f);
      }
      wsum[k] = __fadd_rn(wsum[k], wk);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int b = 3 * k + c;
        const uint32_t byte = (v[b >> 2] >> (8 * (b & 3))) & 0xffu;
        acc[b] += __float2int_rz(__fmul_rn((float)byte, wk));
      }
    }
  }

  if (n_px > 0) {
    uint32_t o[3] = {0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < kLayerGroupPx; ++k) {
      const float den = __fadd_rn(wsum[k], 1e-5f);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int b = 3 * k + c;
        const uint32_t q = wsum[k] > 1e-5f ? (uint32_t)__float2int_rz(__fdiv_rn((float)acc[b], den)) : 0u;
        o[b >> 2] |= q << (8 * (b & 3));
      }
    }
    stage[3 * threadIdx.x] = o[0];
    stage[3 * threadIdx.x + 1] = o[1];
    stage[3 * threadIdx.x + 2] = o[2];
  }
  __syncthreads();
  store_segment(stage, p.out + ((size_t)y * (size_t)p.canvas_w + (size_t)seg0) * 3, 3 * seg_px);
}

// the layer's rectangle clipped to the canvas; cw = ch = 0 when they do not meet
void clip_rect(const LayerDesc &L, int canvas_h, int canvas_w, FeatherRect &R) {
  const long long x0 = std::max(0LL, (long long)L.x0), y0 = std::max(0LL, (long long)L.y0);
  const long long x1 = std::min((long long)canvas_w, (long long)L.x0 + L.w);
  const long long y1 = std::min((long long)canvas_h, (long long)L.y0 + L.h);
  R.dist = nullptr;
  R.cx0 = (int)x0;
  R.cy0 = (int)y0;
  R.cw = x1 > x0 && y1 > y0 ? (int)(x1 - x0) : 0;
  R.ch = R.cw ? (int)(y1 - y0) : 0;
}

size_t dist_bytes(const FeatherRect &R) { return ((size_t)R.cw * (size_t)R.ch * 2 + 15) & ~(size_t)15; }

int check_layers(const long long *layers, int n_layers, int canvas_h, int canvas_w) {
  if (!layers) return fail(APAP_E_BADARG, "feather: null pointer");
  if (int rc = check_layer_count_canvas("feather", n_layers, APAP_FEATHER_MAX_LAYERS, "APAP_FEATHER_MAX_LAYERS",
                                        canvas_h, canvas_w))
    return rc;
  return check_layer_descs("feather", layers, n_layers);
}

int distance_cap(float s, int canvas_h, int canvas_w, int *cap) {
  if (!cap) return fail(APAP_E_BADARG, "feather: null pointer");
  // below FLT_MIN (a subnormal s), fl(FLT_MAX s) < 1 can hold: OpenCV then gives a layer with no empty pixel the
  // weight min(fl(FLT_MAX s), 1) < 1, where the kernels give D = cap the weight 1
  if (!(s >= FLT_MIN) || !std::isfinite(s))
    return fail(APAP_E_BADARG, "feather: sharpness must be finite and >= FLT_MIN (a normal float)");
  if (canvas_h <= 0 || canvas_w <= 0 || canvas_w > (1 << 30) || canvas_h > (1 << 30))
    return fail(APAP_E_BADARG, "feather: canvas sizes must be in [1, 2^30]");
  // the smallest d >= 1 with fl(d s) >= 1; (double)d * s is exact for d < 2^29, so its float rounding is fl(d s)
  const double g = std::ceil(1.0 / (double)s);
  long long d = 1LL << 40;
  if (g < (double)(1 << 28)) {
    d = std::max(1LL, (long long)g);
    while (d > 1 && (float)((double)(d - 1) * s) >= 1.f) --d;
    while ((float)((double)d * s) < 1.f) ++d;
  }
  const long long limit = (long long)canvas_h + canvas_w - 1;    // more than any finite distance in the canvas
  const long long c = std::min(d, limit);
  if (c > 65535)
    return fail(APAP_E_TOOBIG, "feather: the distance cap exceeds 65535 (a larger sharpness or a smaller canvas)");
  *cap = (int)c;
  return 0;
}

}  // namespace apap

using namespace apap;

extern "C" int apap_feather_distance_cap(float sharpness, int canvas_h, int canvas_w, int *cap) {
  return distance_cap(sharpness, canvas_h, canvas_w, cap);
}

extern "C" int apap_feather_workspace_bytes(const long long *layers, int n_layers, int canvas_h, int canvas_w,
                                            size_t *bytes) {
  if (!bytes) return fail(APAP_E_BADARG, "feather: null pointer");
  if (int rc = check_layers(layers, n_layers, canvas_h, canvas_w)) return rc;
  size_t total = 0;
  for (int l = 0; l < n_layers; ++l) {
    FeatherRect R;
    clip_rect(layer_desc(layers + 6 * l), canvas_h, canvas_w, R);
    total += dist_bytes(R);
  }
  *bytes = total;
  return 0;
}

static int feather_blend(const long long *layers, int n_layers, int canvas_h, int canvas_w, float sharpness,
                         const uint8_t *lut, void *workspace, size_t workspace_bytes, uint8_t *out,
                         size_t out_bytes, cudaStream_t st) {
  if (!out || !workspace) return fail(APAP_E_BADARG, "feather_blend: null pointer");
  if (int rc = check_layers(layers, n_layers, canvas_h, canvas_w)) return rc;
  if (out_bytes < (size_t)canvas_h * (size_t)canvas_w * 3)
    return fail(APAP_E_BADARG, "feather_blend: out is smaller than canvas_h x canvas_w x 3 bytes");
  if (reinterpret_cast<uintptr_t>(workspace) & 15u)
    return fail(APAP_E_ALIGN, "feather_blend: workspace must be 16-byte aligned");
  FeatherParams p;
  if (int rc = distance_cap(sharpness, canvas_h, canvas_w, &p.cap)) return rc;
  uint8_t *ws = static_cast<uint8_t *>(workspace);
  size_t used = 0;
  int max_ch = 0, max_cw = 0;
  for (int l = 0; l < n_layers; ++l) {
    p.layer[l] = layer_desc(layers + 6 * l);
    clip_rect(p.layer[l], canvas_h, canvas_w, p.rect[l]);
    p.rect[l].dist = reinterpret_cast<uint16_t *>(ws + used);
    used += dist_bytes(p.rect[l]);
    max_ch = std::max(max_ch, p.rect[l].ch);
    max_cw = std::max(max_cw, p.rect[l].cw);
  }
  if (workspace_bytes < used)
    return fail(APAP_E_BADARG, "feather_blend: workspace is smaller than apap_feather_workspace_bytes");
  p.out = out;
  p.s = sharpness;
  p.n_layers = n_layers;
  p.canvas_h = canvas_h;
  p.canvas_w = canvas_w;
  p.segs_per_row = (canvas_w + kSegPx - 1) / kSegPx;
  const long long blocks = (long long)p.segs_per_row * canvas_h;
  if (blocks > 2147483647LL) return fail(APAP_E_TOOBIG, "feather_blend: canvas too large");
  if (max_ch > 0) {
    k_feather_rows<<<dim3((unsigned)max_ch, (unsigned)n_layers), kLayerThreads, 0, st>>>(p);
    if (int rc = check_cuda(cudaGetLastError(), "k_feather_rows launch")) return rc;
    k_feather_cols<<<dim3((unsigned)((max_cw + kColThreadsX - 1) / kColThreadsX), (unsigned)n_layers),
                     dim3(kColThreadsX, kColSegs), 0, st>>>(p);
    if (int rc = check_cuda(cudaGetLastError(), "k_feather_cols launch")) return rc;
  }
  if (lut) k_feather_blend<true><<<(unsigned)blocks, kLayerThreads, 0, st>>>(p, lut);
  else k_feather_blend<false><<<(unsigned)blocks, kLayerThreads, 0, st>>>(p, nullptr);
  return check_cuda(cudaGetLastError(), "k_feather_blend launch");
}

extern "C" int apap_feather_blend(const long long *layers, int n_layers, int canvas_h, int canvas_w, float sharpness,
                                  void *workspace, size_t workspace_bytes, uint8_t *out, size_t out_bytes,
                                  void *stream) {
  return feather_blend(layers, n_layers, canvas_h, canvas_w, sharpness, nullptr, workspace, workspace_bytes, out,
                       out_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int apap_feather_blend_gain(const long long *layers, int n_layers, int canvas_h, int canvas_w,
                                       float sharpness, const uint8_t *lut, void *workspace, size_t workspace_bytes,
                                       uint8_t *out, size_t out_bytes, void *stream) {
  if (!lut) return fail(APAP_E_BADARG, "feather_blend_gain: null gain table");
  return feather_blend(layers, n_layers, canvas_h, canvas_w, sharpness, lut, workspace, workspace_bytes, out,
                       out_bytes, static_cast<cudaStream_t>(stream));
}
