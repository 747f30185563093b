// Overlap statistics of cv.detail.GainCompensator (utils.exposure_gains, DESIGN.md section 3): for placed layers, per
// pair i <= j the count |mask_i & mask_j| and per pair i != j the sum over that intersection of norm(P_i) =
// sqrt(b^2 + g^2 + r^2) in double.  mask_k is "any channel > 0" of layer k, as in the panorama blends.
//
// Exact and order-free: for q >= 1, sqrt(q) (__dsqrt_rn, correctly rounded) lies in [1, 2^9), so sqrt(q) 2^52 is an
// integer below 2^61, and the kernel sums those integers exactly.  Per pixel it splits them into three 25-bit limbs;
// a thread sums at most 4 pixels per limb (< 2^27), a warp that with one redux.sync (< 2^32), the CTA the 8 warps in
// 64 bits.  The CTA total T < 2^71 (1024 pixels, each below 2^61) then goes to global memory as three 32-bit pieces
// (bits 0-31, 32-63, 64-95), each added to its own 64-bit word: at most 2^31 CTAs add less than 2^32 each, so no word
// wraps.  Integer adds commute, so any schedule gives the same words; the host reads word0 + word1 2^32 + word2 2^64.
//
// One CTA per kSegPx-pixel canvas row segment, 4 pixels per thread (layers.cuh).  The CTA first walks the layers
// whose rectangle meets the segment (uniform test) and keeps those with a non-empty pixel in it (a CTA vote), with
// every thread's 4-bit mask of each in shared memory.  Then per ordered pair (a, b) of those layers that meets in
// the segment (a second vote): the count (a <= b) and the limb sums of norm(P_a) over the intersection (a != b),
// reduced per warp, then per CTA by thread 0, which adds them to global memory (fire-and-forget reductions).
#include "layers.cuh"

namespace apap {

constexpr int kLimbBits = 25;
constexpr unsigned long long kLimbMask = (1ull << kLimbBits) - 1ull;
constexpr int kWarps = kLayerThreads / 32;

struct GainStatsParams {
  LayerDesc layer[APAP_GAIN_MAX_LAYERS];
  unsigned long long *count;            // [n][n], i <= j
  unsigned long long *sum;              // [3][n][n], i != j: 32-bit pieces of the exact sum
  int n_layers, canvas_w, segs_per_row;
};

__global__ void __launch_bounds__(kLayerThreads) k_gain_stats(const __grid_constant__ GainStatsParams p) {
  __shared__ uint8_t nib[APAP_GAIN_MAX_LAYERS / 2][kLayerThreads];   // 4-bit masks, two present layers per byte
  __shared__ short present[APAP_GAIN_MAX_LAYERS];
  __shared__ uint32_t red[kWarps][4];
  const int y = blockIdx.x / p.segs_per_row;
  const int seg0 = (blockIdx.x - y * p.segs_per_row) * kSegPx;
  const int seg_px = min(kSegPx, p.canvas_w - seg0);
  const int x = seg0 + kLayerGroupPx * (int)threadIdx.x;
  const int n_px = min(kLayerGroupPx, p.canvas_w - x);          // pixels of this thread (<= 0: none)
  const int n = p.n_layers;

  int m = 0;                                    // present layers, in layer order
  for (int l = 0; l < n; ++l) {
    const LayerDesc &L = p.layer[l];
    const int ly = y - L.y0, lx0 = seg0 - L.x0;
    if ((unsigned)ly >= (unsigned)L.h || lx0 >= L.w || lx0 + seg_px <= 0) continue;   // uniform
    uint32_t w[3];
    fetch_group(L, y, seg0, seg_px, x, n_px, w);
    const uint32_t nz = byte_nonzero(group_or(w[0], w[1], w[2]));
    const uint32_t bits = (nz | nz >> 7 | nz >> 14 | nz >> 21) & 15u;
    if (!__syncthreads_or(bits)) continue;      // uniform
    uint8_t &slot = nib[m >> 1][threadIdx.x];   // this thread's own byte
    slot = (m & 1) ? (uint8_t)(slot | bits << 4) : (uint8_t)bits;
    if (threadIdx.x == 0) present[m] = (short)l;
    ++m;
  }
  __syncthreads();                              // present[] is written

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int a = 0; a < m; ++a) {
    const int la = present[a];
    uint32_t w[3];
    fetch_group(p.layer[la], y, seg0, seg_px, x, n_px, w);
    const uint32_t ma = (nib[a >> 1][threadIdx.x] >> (4 * (a & 1))) & 15u;
    uint32_t limb[3][kLayerGroupPx];            // sqrt(q) 2^52 in 25-bit limbs, 0 where empty
#pragma unroll
    for (int k = 0; k < kLayerGroupPx; ++k) {
      uint32_t q = 0u;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int b = 3 * k + c;
        const uint32_t v = (w[b >> 2] >> (8 * (b & 3))) & 0xffu;
        q += v * v;
      }
      const unsigned long long e =
          q ? __double2ull_rn(__dmul_rn(__dsqrt_rn((double)q), 4503599627370496.0)) : 0ull;   // x 2^52, exact
      limb[0][k] = (uint32_t)(e & kLimbMask);
      limb[1][k] = (uint32_t)((e >> kLimbBits) & kLimbMask);
      limb[2][k] = (uint32_t)(e >> (2 * kLimbBits));
    }
    for (int b = 0; b < m; ++b) {
      const uint32_t inter = ma & (nib[b >> 1][threadIdx.x] >> (4 * (b & 1))) & 15u;
      if (!__syncthreads_or(inter)) continue;   // uniform; also keeps red[] until thread 0 has read it
      uint32_t s[3] = {0u, 0u, 0u};
      if (b != a) {
#pragma unroll
        for (int k = 0; k < kLayerGroupPx; ++k) {
          const uint32_t on = 0u - ((inter >> k) & 1u);
#pragma unroll
          for (int i = 0; i < 3; ++i) s[i] += limb[i][k] & on;
        }
      }
      const uint32_t r0 = __reduce_add_sync(0xffffffffu, s[0]);
      const uint32_t r1 = __reduce_add_sync(0xffffffffu, s[1]);
      const uint32_t r2 = __reduce_add_sync(0xffffffffu, s[2]);
      const uint32_t rc = __reduce_add_sync(0xffffffffu, (uint32_t)__popc(inter));
      if (lane == 0) {
        red[warp][0] = r0;
        red[warp][1] = r1;
        red[warp][2] = r2;
        red[warp][3] = rc;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned long long t[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
        for (int k = 0; k < kWarps; ++k)
#pragma unroll
          for (int i = 0; i < 4; ++i) t[i] += red[k][i];
        const int lb = present[b];
        if (a <= b) atomicAdd(p.count + (size_t)la * n + lb, t[3]);
        if (a != b) {
          const unsigned __int128 total = (unsigned __int128)t[0] + ((unsigned __int128)t[1] << kLimbBits) +
                                          ((unsigned __int128)t[2] << (2 * kLimbBits));
          const size_t plane = (size_t)n * n, at = (size_t)la * n + lb;
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const unsigned long long piece = (unsigned long long)(total >> (32 * i)) & 0xffffffffull;
            if (piece) atomicAdd(p.sum + i * plane + at, piece);
          }
        }
      }
    }
  }
}

int check_gain_layers(const long long *layers, int n_layers, int canvas_h, int canvas_w) {
  if (!layers) return fail(APAP_E_BADARG, "gain_stats: null pointer");
  if (int rc = check_layer_count_canvas("gain_stats", n_layers, APAP_GAIN_MAX_LAYERS, "APAP_GAIN_MAX_LAYERS", canvas_h,
                                        canvas_w))
    return rc;
  return check_layer_descs("gain_stats", layers, n_layers);
}

size_t gain_stats_bytes(int n_layers) { return (size_t)4 * n_layers * n_layers * sizeof(unsigned long long); }

}  // namespace apap

using namespace apap;

extern "C" int apap_gain_stats_bytes(int n_layers, size_t *bytes) {
  if (!bytes) return fail(APAP_E_BADARG, "gain_stats: null pointer");
  if (n_layers < 1 || n_layers > APAP_GAIN_MAX_LAYERS)
    return fail(APAP_E_BADARG, "gain_stats: 1 <= n_layers <= APAP_GAIN_MAX_LAYERS");
  *bytes = gain_stats_bytes(n_layers);
  return 0;
}

extern "C" int apap_gain_stats(const long long *layers, int n_layers, int canvas_h, int canvas_w, void *stats,
                               size_t stats_bytes, void *stream) {
  if (!stats) return fail(APAP_E_BADARG, "gain_stats: null pointer");
  if (int rc = check_gain_layers(layers, n_layers, canvas_h, canvas_w)) return rc;
  if (stats_bytes < gain_stats_bytes(n_layers))
    return fail(APAP_E_BADARG, "gain_stats: stats is smaller than apap_gain_stats_bytes");
  if (reinterpret_cast<uintptr_t>(stats) & 7u) return fail(APAP_E_ALIGN, "gain_stats: stats must be 8-byte aligned");
  GainStatsParams p;
  for (int l = 0; l < n_layers; ++l) p.layer[l] = layer_desc(layers + 6 * l);
  p.count = static_cast<unsigned long long *>(stats);
  p.sum = p.count + (size_t)n_layers * n_layers;
  p.n_layers = n_layers;
  p.canvas_w = canvas_w;
  p.segs_per_row = (canvas_w + kSegPx - 1) / kSegPx;
  const long long blocks = (long long)p.segs_per_row * canvas_h;
  if (blocks > 2147483647LL) return fail(APAP_E_TOOBIG, "gain_stats: canvas too large");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = check_cuda(cudaMemsetAsync(stats, 0, gain_stats_bytes(n_layers), st), "gain_stats memset")) return rc;
  k_gain_stats<<<(unsigned)blocks, kLayerThreads, 0, st>>>(p);
  return check_cuda(cudaGetLastError(), "k_gain_stats launch");
}
