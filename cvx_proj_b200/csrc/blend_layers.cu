// Panorama blend of N placed layers (driver.stitch_panorama): per canvas pixel, the per-channel floor mean of the
// layers that are non-empty there (any channel > 0), 0 where none is.  For two equal layers at one origin this is
// uniform_blend (K4) bit for bit.
//
// Bandwidth-bound byte work: every canvas byte is written once and every layer byte inside the canvas is read once.
// The segment and group shape and the layer reads are layers.cuh's.  The layer loop runs over all descriptors (a
// __grid_constant__ parameter, read through the constant cache with a uniform index); the row and segment tests are
// uniform per CTA.  Sums are packed 16-bit pairs in registers (255 x 256 < 2^16), counts too.  An empty pixel adds
// zero to the sums, so only the count needs the non-empty test.  floor(s / n) is __umulhi(s, ceil(2^32 / n)) for
// n >= 2 (exact: s (m n - 2^32) < s n <= 255 x 256^2 < 2^32), s itself for n <= 1 (n = 0 means s = 0).
// The segment's bytes are staged in shared memory and leave as aligned 16-byte stores plus a byte-wise head and tail.
// kGains (apap_blend_layers_gain): layer l's bytes go through its exposure-gain table lut[l][256] before they are
// summed; the non-empty test still reads the raw bytes, and compensated bytes are <= 255, so the bound above holds.
#include "layers.cuh"

namespace apap {

struct LayerParams {
  LayerDesc layer[APAP_BLEND_MAX_LAYERS];
  uint8_t *out;
  int n_layers, canvas_h, canvas_w, segs_per_row;
};

template <bool kGains>
__global__ void __launch_bounds__(kLayerThreads) k_blend_layers(const __grid_constant__ LayerParams p,
                                                                const uint8_t *__restrict__ lut) {
  __shared__ uint32_t recip[APAP_BLEND_MAX_LAYERS + 1];
  __shared__ __align__(16) uint32_t stage[kSegBytes / 4];
  for (int i = threadIdx.x; i <= APAP_BLEND_MAX_LAYERS; i += kLayerThreads)
    recip[i] = i < 2 ? 0u : 0xffffffffu / (uint32_t)i + 1u;    // ceil(2^32 / n) = floor((2^32 - 1) / n) + 1

  const int y = blockIdx.x / p.segs_per_row;
  const int seg0 = (blockIdx.x - y * p.segs_per_row) * kSegPx;
  const int seg_px = min(kSegPx, p.canvas_w - seg0);
  const int x = seg0 + kLayerGroupPx * (int)threadIdx.x;
  const int n_px = min(kLayerGroupPx, p.canvas_w - x);          // pixels of this thread (<= 0: none)

  uint32_t s[6] = {0u, 0u, 0u, 0u, 0u, 0u};   // s[k]: sums of group bytes 2k (low half) and 2k + 1 (high half)
  uint32_t c01 = 0u, c23 = 0u;                 // non-empty counts of pixels 0, 1 and 2, 3 (16-bit halves)
  for (int l = 0; l < p.n_layers; ++l) {
    uint32_t w[3];
    fetch_group(p.layer[l], y, seg0, seg_px, x, n_px, w);
    uint32_t v[3] = {w[0], w[1], w[2]};
    if constexpr (kGains) gain_group(lut + 256 * l, v);
    s[0] += __byte_perm(v[0], 0u, 0x4140); s[1] += __byte_perm(v[0], 0u, 0x4342);
    s[2] += __byte_perm(v[1], 0u, 0x4140); s[3] += __byte_perm(v[1], 0u, 0x4342);
    s[4] += __byte_perm(v[2], 0u, 0x4140); s[5] += __byte_perm(v[2], 0u, 0x4342);
    const uint32_t nz = byte_nonzero(group_or(w[0], w[1], w[2]));
    c01 += __byte_perm(nz, 0u, 0x4140);
    c23 += __byte_perm(nz, 0u, 0x4342);
  }
  __syncthreads();                              // recip[] is written

  if (n_px > 0) {
    const uint32_t n[4] = {c01 & 0xffffu, c01 >> 16, c23 & 0xffffu, c23 >> 16};
    uint32_t o[3] = {0u, 0u, 0u};
#pragma unroll
    for (int b = 0; b < 12; ++b) {
      const uint32_t sum = (s[b >> 1] >> (16 * (b & 1))) & 0xffffu;
      const uint32_t cnt = n[b / 3];
      const uint32_t v = cnt < 2 ? sum : __umulhi(sum, recip[cnt]);
      o[b >> 2] |= v << (8 * (b & 3));
    }
    stage[3 * threadIdx.x] = o[0];
    stage[3 * threadIdx.x + 1] = o[1];
    stage[3 * threadIdx.x + 2] = o[2];
  }
  __syncthreads();

  // the segment's bytes [0, nb) go to dst: byte-wise head up to a 16-byte boundary, 16-byte units, byte-wise tail
  uint8_t *dst = p.out + ((size_t)y * (size_t)p.canvas_w + (size_t)seg0) * 3;
  const int nb = 3 * seg_px;
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

int launch_blend_layers(const long long *layers, int n_layers, int canvas_h, int canvas_w, const uint8_t *lut,
                        uint8_t *out, cudaStream_t st) {
  LayerParams p;
  for (int l = 0; l < n_layers; ++l) p.layer[l] = layer_desc(layers + 6 * l);
  p.out = out;
  p.n_layers = n_layers;
  p.canvas_h = canvas_h;
  p.canvas_w = canvas_w;
  p.segs_per_row = (canvas_w + kSegPx - 1) / kSegPx;
  const long long blocks = (long long)p.segs_per_row * canvas_h;
  if (blocks > 2147483647LL) return fail(APAP_E_TOOBIG, "blend_layers: canvas too large");
  if (lut) k_blend_layers<true><<<(unsigned)blocks, kLayerThreads, 0, st>>>(p, lut);
  else k_blend_layers<false><<<(unsigned)blocks, kLayerThreads, 0, st>>>(p, nullptr);
  return check_cuda(cudaGetLastError(), "k_blend_layers launch");
}

}  // namespace apap

using namespace apap;

namespace {

int check_blend_layers(const long long *layers, int n_layers, int canvas_h, int canvas_w, const uint8_t *out,
                       size_t out_bytes) {
  if (!layers || !out) return fail(APAP_E_BADARG, "blend_layers: null pointer");
  if (int rc = check_layer_count_canvas("blend_layers", n_layers, APAP_BLEND_MAX_LAYERS, "APAP_BLEND_MAX_LAYERS",
                                        canvas_h, canvas_w))
    return rc;
  if (out_bytes < (size_t)canvas_h * (size_t)canvas_w * 3)
    return fail(APAP_E_BADARG, "blend_layers: out is smaller than canvas_h x canvas_w x 3 bytes");
  return check_layer_descs("blend_layers", layers, n_layers);
}

}  // namespace

extern "C" int apap_blend_layers(const long long *layers, int n_layers, int canvas_h, int canvas_w, uint8_t *out,
                                 size_t out_bytes, void *stream) {
  if (int rc = check_blend_layers(layers, n_layers, canvas_h, canvas_w, out, out_bytes)) return rc;
  return launch_blend_layers(layers, n_layers, canvas_h, canvas_w, nullptr, out, static_cast<cudaStream_t>(stream));
}

extern "C" int apap_blend_layers_gain(const long long *layers, int n_layers, int canvas_h, int canvas_w,
                                      const uint8_t *lut, uint8_t *out, size_t out_bytes, void *stream) {
  if (!lut) return fail(APAP_E_BADARG, "blend_layers_gain: null gain table");
  if (int rc = check_blend_layers(layers, n_layers, canvas_h, canvas_w, out, out_bytes)) return rc;
  return launch_blend_layers(layers, n_layers, canvas_h, canvas_w, lut, out, static_cast<cudaStream_t>(stream));
}
