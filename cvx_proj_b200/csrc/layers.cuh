// Placed uint8 [h][w][3] layers read and a canvas row segment written by the N-layer kernels (blend_layers.cu,
// feather.cu, gain.cu).  A CTA owns a segment of kSegPx pixels of one canvas row, a thread 4 consecutive pixels
// (12 bytes).
// A layer row's 12-byte groups all share one phase modulo 4 (12 is a multiple of 4), so a thread reads its group as 3
// or 4 aligned words -- each holding at least one byte of the group -- and funnel-shifts them into place; the at most
// two groups that straddle a layer's left or right edge read byte by byte.  The segment's bytes are staged in shared
// memory and leave as aligned 16-byte stores plus a byte-wise head and tail.
#pragma once
#include <cstdio>

#include "common.cuh"

namespace apap {

constexpr int kLayerThreads = 256;
constexpr int kLayerGroupPx = 4;                         // pixels per thread
constexpr int kSegPx = kLayerThreads * kLayerGroupPx;    // canvas pixels per CTA
constexpr int kSegBytes = 3 * kSegPx;
static_assert(kSegBytes / 16 <= kLayerThreads - 32, "the last warp writes the head and tail bytes");

struct LayerDesc {
  const uint8_t *addr;     // pixel (0, 0) of the layer
  long long pitch;         // bytes from one layer row to the next
  int h, w, x0, y0;        // size and canvas position of the top-left pixel (may be negative)
};

// {device address, h, w, row pitch in bytes, x0, y0} of the C ABI
inline LayerDesc layer_desc(const long long *d) {
  LayerDesc L;
  L.addr = reinterpret_cast<const uint8_t *>(static_cast<uintptr_t>(d[0]));
  L.h = (int)d[1];
  L.w = (int)d[2];
  L.pitch = d[3];
  L.x0 = (int)d[4];
  L.y0 = (int)d[5];
  return L;
}

// Argument checks the placed-layer entry points share (apap_blend_layers*, apap_feather_*, apap_gain_stats), in two
// steps so that each entry keeps its own order of checks; every message starts with `what`.
// The layer count (1 .. max_layers, named max_name in the message) and the canvas sizes.
inline int check_layer_count_canvas(const char *what, int n_layers, int max_layers, const char *max_name, int canvas_h,
                                    int canvas_w) {
  char msg[160];
  if (n_layers < 1 || n_layers > max_layers) {
    snprintf(msg, sizeof(msg), "%s: 1 <= n_layers <= %s", what, max_name);
    return fail(APAP_E_BADARG, msg);
  }
  if (canvas_h <= 0 || canvas_w <= 0 || canvas_w > (1 << 30) || canvas_h > (1 << 30)) {
    snprintf(msg, sizeof(msg), "%s: canvas sizes must be in [1, 2^30]", what);
    return fail(APAP_E_BADARG, msg);
  }
  return 0;
}

// every descriptor {device address, h, w, row pitch in bytes, x0, y0} of the C ABI
inline int check_layer_descs(const char *what, const long long *layers, int n_layers) {
  char msg[160];
  for (int l = 0; l < n_layers; ++l) {
    const long long *d = layers + 6 * l;
    const long long h = d[1], w = d[2], pitch = d[3], x0 = d[4], y0 = d[5];
    const char *err = nullptr;
    if (!d[0]) err = "null layer address";
    else if (h < 1 || w < 1 || h > (1 << 30) || w > (1 << 30)) err = "layer sizes must be in [1, 2^30]";
    else if (h > 1 && pitch < 3 * w) err = "layer pitch is smaller than 3 x width";
    else if (x0 < -(1LL << 30) || x0 > (1LL << 30) || y0 < -(1LL << 30) || y0 > (1LL << 30))
      err = "layer origin outside [-2^30, 2^30]";
    if (err) {
      snprintf(msg, sizeof(msg), "%s: %s", what, err);
      return fail(APAP_E_BADARG, msg);
    }
  }
  return 0;
}

// one byte per pixel of a 12-byte group: the OR of its three channel bytes
__device__ __forceinline__ uint32_t group_or(uint32_t w0, uint32_t w1, uint32_t w2) {
  const uint32_t x = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);   // bytes 0, 3, 6, 9
  const uint32_t y = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);   // bytes 1, 4, 7, 10
  const uint32_t z = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);   // bytes 2, 5, 8, 11
  return x | y | z;
}

// bit 0 of every byte = that byte of v is non-zero, the other bits 0
__device__ __forceinline__ uint32_t byte_nonzero(uint32_t v) {
  return ((((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v) >> 7) & 0x01010101u;
}

// the 12 bytes of layer L under this thread's group of canvas pixels [x, x + n_px) of row y, zeros where the layer is
// absent (the row or the pixels outside the layer); [seg0, seg0 + seg_px) is the CTA's segment
__device__ __forceinline__ void fetch_group(const LayerDesc &L, int y, int seg0, int seg_px, int x, int n_px,
                                            uint32_t (&w)[3]) {
  w[0] = w[1] = w[2] = 0u;
  const int ly = y - L.y0;
  const int lx0 = seg0 - L.x0;                  // layer column of the segment's first pixel
  if ((unsigned)ly >= (unsigned)L.h || lx0 >= L.w || lx0 + seg_px <= 0) return;   // uniform
  const int lx = x - L.x0;
  if (n_px <= 0 || lx >= L.w || lx + n_px <= 0) return;
  const uint8_t *q = L.addr + (long long)ly * L.pitch + 3LL * lx;
  if (n_px == kLayerGroupPx && lx >= 0 && lx + kLayerGroupPx <= L.w) {
    const uint32_t phase = (uint32_t)reinterpret_cast<uintptr_t>(q) & 3u;   // uniform over the CTA
    const uint32_t *a = reinterpret_cast<const uint32_t *>(q - phase);
    const uint32_t a0 = __ldg(a), a1 = __ldg(a + 1), a2 = __ldg(a + 2), a3 = phase ? __ldg(a + 3) : 0u;
    w[0] = __funnelshift_r(a0, a1, 8u * phase);
    w[1] = __funnelshift_r(a1, a2, 8u * phase);
    w[2] = __funnelshift_r(a2, a3, 8u * phase);
  } else {                                      // the group straddles the layer's edge or the canvas end
#pragma unroll
    for (int k = 0; k < kLayerGroupPx; ++k) {
      if (k < n_px && (unsigned)(lx + k) < (unsigned)L.w) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int b = 3 * k + c;
          w[b >> 2] |= (uint32_t)__ldg(q + b) << (8 * (b & 3));
        }
      }
    }
  }
}

// exposure gain of one group (the blends' kGains instantiations): every byte v becomes lut[v], the layer's
// saturate(rint(v g)) table of apap_blend_layers_gain; lut[0] is 0, so absent pixels stay 0.  kChannels: lut is the
// layer's [3][256] table of apap_blend_layers_channels, and byte b of the group, channel b % 3, reads row b % 3
template <bool kChannels>
__device__ __forceinline__ void gain_group(const uint8_t *__restrict__ lut, uint32_t (&v)[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const uint32_t u = v[i];
    if constexpr (kChannels) {
      const uint8_t *t0 = lut + 256 * ((4 * i) % 3), *t1 = lut + 256 * ((4 * i + 1) % 3);
      const uint8_t *t2 = lut + 256 * ((4 * i + 2) % 3), *t3 = lut + 256 * ((4 * i + 3) % 3);
      v[i] = (uint32_t)__ldg(t0 + (u & 0xffu)) | (uint32_t)__ldg(t1 + ((u >> 8) & 0xffu)) << 8 |
             (uint32_t)__ldg(t2 + ((u >> 16) & 0xffu)) << 16 | (uint32_t)__ldg(t3 + (u >> 24)) << 24;
    } else {
      v[i] = (uint32_t)__ldg(lut + (u & 0xffu)) | (uint32_t)__ldg(lut + ((u >> 8) & 0xffu)) << 8 |
             (uint32_t)__ldg(lut + ((u >> 16) & 0xffu)) << 16 | (uint32_t)__ldg(lut + (u >> 24)) << 24;
    }
  }
}

// the segment's staged bytes [0, nb) go to dst: byte-wise head up to a 16-byte boundary, 16-byte units, byte-wise
// tail; every thread of the CTA calls it after the stage is complete.  k_blend_layers keeps the same code inline:
// calling this helper there compiles to a different schedule and register assignment (cuobjdump -sass), while the
// inline copy leaves its SASS as it was before the helper existed.
__device__ __forceinline__ void store_segment(const uint32_t (&stage)[kSegBytes / 4], uint8_t *dst, int nb) {
  const int head = min(nb, (int)((16u - ((uint32_t)reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u));
  const int units = (nb - head) >> 4;
  const int tail0 = head + 16 * units;
  const uint8_t *stage8 = reinterpret_cast<const uint8_t *>(stage);
  const int t = threadIdx.x;
  if (t < units) {
    const int off = head + 16 * t;              // a multiple of 4 plus (head & 3)
    const int sh = off & 3;
    const uint32_t *src = stage + (off >> 2);
    const uint32_t a0 = src[0], a1 = src[1], a2 = src[2], a3 = src[3], a4 = sh ? src[4] : 0u;
    reinterpret_cast<uint4 *>(dst + off)[0] =
        make_uint4(__funnelshift_r(a0, a1, 8 * sh), __funnelshift_r(a1, a2, 8 * sh), __funnelshift_r(a2, a3, 8 * sh),
                   __funnelshift_r(a3, a4, 8 * sh));
  } else if (t >= kLayerThreads - 32) {         // one warp: head and tail bytes (fewer than 16 each)
    const int k = t - (kLayerThreads - 32);
    if (k < head) dst[k] = stage8[k];
    else if (k >= 16 && tail0 + (k - 16) < nb) dst[tail0 + k - 16] = stage8[tail0 + k - 16];
  }
}

}  // namespace apap
