// Per-channel histogram equalisation of a BGR image: cv.merge([cv.equalizeHist(c) for c in cv.split(img)]), the
// reference's visualize_equalized_hist (pyviz/utils.py:85-91, SURVEY 3.1), bit for bit.
//   k_eq_hist  : three 256-bin uint32 histograms of a uint8 [h][w][3] image, read as one run of 3 h w bytes (the
//                channel of byte k is k mod 3) in 16-byte vectors, 48 bytes (16 pixels) per thread and step.
//   k_eq_lut   : OpenCV's LUT per channel from its histogram: i0 = first non-zero bin; all i0 if hist[i0] == total
//                (dst.setTo(i0)); else lut[i0] = 0 and lut[i] = saturate_cast<uchar>((float)sum * scale) for i > i0,
//                sum = hist[i0 + 1] + ... + hist[i], scale = 255.f / (float)(total - hist[i0]).  Integer sums are
//                exact in any order, and the float steps are rounded one by one (no FMA contraction), so the LUT is
//                OpenCV's.  Entries below i0 are never read; they are written 0.
//   k_eq_apply : the equalised image through the LUT (only the standalone equalisation materialises it; SIFT
//                description reads the raw image through the LUT in k_sift_base<true>, csrc/sift.cu).
#include "common.cuh"

namespace apap {

constexpr int kEqThreads = 256;
constexpr int kEqBins = 3 * 256;
// One histogram copy per lane index, interleaved (copy l of bin b at word 32 b + l): a lane always hits its own bank,
// so a flat image costs no more than noise; warps of the CTA share the copies through shared atomics.
constexpr int kEqCopies = 32;
constexpr int kEqHistSmem = kEqBins * kEqCopies * (int)sizeof(uint32_t);     // 96 KB: two CTAs per SM

// The image as a byte run of n = 3 h w bytes: `head` bytes up to the first 16-byte aligned address, then `units`
// aligned 48-byte units (whose first byte has channel `head mod 3`), then a tail of fewer than 48 bytes.
struct EqRun {
  long long n, head, units;
};

static EqRun eq_run(const void *p, long long n) {
  EqRun r;
  r.n = n;
  r.head = (long long)((16u - (unsigned)(reinterpret_cast<uintptr_t>(p) & 15u)) & 15u);
  if (r.head > n) r.head = n;
  r.units = (n - r.head) / 48;
  return r;
}

__device__ __forceinline__ void unpack48(const uint4 *v, uint32_t (&wd)[12]) {
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    const uint4 x = __ldg(v + q);
    wd[4 * q] = x.x; wd[4 * q + 1] = x.y; wd[4 * q + 2] = x.z; wd[4 * q + 3] = x.w;
  }
}

__global__ void __launch_bounds__(kEqThreads) k_eq_hist(const uint8_t *__restrict__ bgr, EqRun run,
                                                        uint32_t *__restrict__ hist) {
  extern __shared__ __align__(16) uint32_t eq_sh[];                 // [kEqBins][kEqCopies]
  for (int i = threadIdx.x; i < kEqBins * kEqCopies / 4; i += kEqThreads)
    reinterpret_cast<uint4 *>(eq_sh)[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  uint32_t *mine = eq_sh + (threadIdx.x & 31);
  const int phase = (int)(run.head % 3);
  // word offset of channel (phase + j) mod 3 for byte j of a unit
  const int off0 = phase * 256 * kEqCopies, off1 = ((phase + 1) % 3) * 256 * kEqCopies,
            off2 = ((phase + 2) % 3) * 256 * kEqCopies;
  const uint4 *vec = reinterpret_cast<const uint4 *>(bgr + run.head);
  for (long long u = (long long)blockIdx.x * kEqThreads + threadIdx.x; u < run.units; u += (long long)gridDim.x * kEqThreads) {
    uint32_t wd[12];
    unpack48(vec + 3 * u, wd);
#pragma unroll
    for (int j = 0; j < 48; ++j) {
      const uint32_t v = (wd[j >> 2] >> (8 * (j & 3))) & 0xffu;
      const int off = j % 3 == 0 ? off0 : (j % 3 == 1 ? off1 : off2);
      atomicAdd(mine + off + (int)v * kEqCopies, 1u);
    }
  }
  if (blockIdx.x == 0) {                                            // unaligned head and the tail, byte by byte
    for (long long k = threadIdx.x; k < run.head; k += kEqThreads)
      atomicAdd(mine + ((int)(k % 3) * 256 + bgr[k]) * kEqCopies, 1u);
    for (long long k = run.head + 48 * run.units + threadIdx.x; k < run.n; k += kEqThreads)
      atomicAdd(mine + ((int)(k % 3) * 256 + bgr[k]) * kEqCopies, 1u);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < kEqBins; b += kEqThreads) {
    uint32_t s = 0;
#pragma unroll 8
    for (int l = 0; l < kEqCopies; ++l) s += eq_sh[b * kEqCopies + ((l + b) & (kEqCopies - 1))];   // rotated: no conflicts
    if (s) atomicAdd(hist + b, s);
  }
}

// grid = 3 (one CTA per channel), 256 threads (one per bin)
__global__ void __launch_bounds__(256) k_eq_lut(const uint32_t *__restrict__ hist, int total, uint8_t *__restrict__ lut) {
  __shared__ uint32_t warp_sum[8];
  __shared__ int first;
  const int c = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint32_t hv = hist[c * 256 + t];
  if (t == 0) first = 256;
  __syncthreads();
  if (hv) atomicMin(&first, t);
  uint32_t s = hv;                                                  // inclusive prefix sum (integers: exact)
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, s, d);
    if (lane >= d) s += o;
  }
  if (lane == 31) warp_sum[warp] = s;
  __syncthreads();
  for (int k = 0; k < warp; ++k) s += warp_sum[k];
  __shared__ uint32_t scan_i0;
  const int i0 = first;
  if (t == i0) scan_i0 = s;
  __syncthreads();
  const int h0 = (int)hist[c * 256 + i0];
  int q;
  if (h0 == total) {
    q = i0;                                                         // OpenCV: dst.setTo(i0)
  } else if (t <= i0) {
    q = 0;
  } else {
    const float scale = __fdiv_rn(255.f, __int2float_rn(total - h0));
    q = __float2int_rn(__fmul_rn(__int2float_rn((int)(s - scan_i0)), scale));   // cvRound: half to even
    q = min(max(q, 0), 255);
  }
  lut[c * 256 + t] = (uint8_t)q;
}

// kVec: input and output share their 16-byte phase, so both move in aligned 48-byte units; otherwise byte by byte
template <bool kVec>
__global__ void __launch_bounds__(kEqThreads) k_eq_apply(const uint8_t *__restrict__ bgr, EqRun run,
                                                         const uint8_t *__restrict__ lut, uint8_t *__restrict__ out) {
  __shared__ uint8_t lut_s[kEqBins];
  for (int i = threadIdx.x; i < kEqBins; i += kEqThreads) lut_s[i] = lut[i];
  __syncthreads();
  const long long stride = (long long)gridDim.x * kEqThreads;
  if constexpr (kVec) {
    const int phase = (int)(run.head % 3);
    const int off0 = phase * 256, off1 = ((phase + 1) % 3) * 256, off2 = ((phase + 2) % 3) * 256;
    const uint4 *vec = reinterpret_cast<const uint4 *>(bgr + run.head);
    uint4 *dst = reinterpret_cast<uint4 *>(out + run.head);
    for (long long u = (long long)blockIdx.x * kEqThreads + threadIdx.x; u < run.units; u += stride) {
      uint32_t wd[12], wo[12];
      unpack48(vec + 3 * u, wd);
#pragma unroll
      for (int q = 0; q < 12; ++q) {
        uint32_t r = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int j = 4 * q + b;
          const int off = j % 3 == 0 ? off0 : (j % 3 == 1 ? off1 : off2);
          r |= (uint32_t)lut_s[off + ((wd[q] >> (8 * b)) & 0xffu)] << (8 * b);
        }
        wo[q] = r;
      }
#pragma unroll
      for (int q = 0; q < 3; ++q) dst[3 * u + q] = make_uint4(wo[4 * q], wo[4 * q + 1], wo[4 * q + 2], wo[4 * q + 3]);
    }
    if (blockIdx.x == 0) {
      for (long long k = threadIdx.x; k < run.head; k += kEqThreads) out[k] = lut_s[(k % 3) * 256 + bgr[k]];
      for (long long k = run.head + 48 * run.units + threadIdx.x; k < run.n; k += kEqThreads)
        out[k] = lut_s[(k % 3) * 256 + bgr[k]];
    }
  } else {
    for (long long k = (long long)blockIdx.x * kEqThreads + threadIdx.x; k < run.n; k += stride)
      out[k] = lut_s[(k % 3) * 256 + bgr[k]];
  }
}

static int eq_grid(long long work) {                                // two resident CTAs per SM at most
  const long long want = (work + kEqThreads - 1) / kEqThreads;
  const long long cap = 2LL * sm_count_cached();
  return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

int launch_equalize_hist(const uint8_t *bgr, int h, int w, uint32_t *hist, uint8_t *lut, uint8_t *out, cudaStream_t st) {
  const long long n = 3LL * h * w;
  const EqRun run = eq_run(bgr, n);
  int rc = check_cuda(cudaMemsetAsync(hist, 0, kEqBins * sizeof(uint32_t), st), "equalize_hist: memset");
  if (rc) return rc;
  rc = check_cuda(cudaFuncSetAttribute(k_eq_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, kEqHistSmem),
                  "equalize_hist: cudaFuncSetAttribute");
  if (rc) return rc;
  k_eq_hist<<<eq_grid(run.units), kEqThreads, kEqHistSmem, st>>>(bgr, run, hist);
  rc = check_cuda(cudaGetLastError(), "k_eq_hist launch");
  if (rc) return rc;
  k_eq_lut<<<3, 256, 0, st>>>(hist, h * w, lut);
  rc = check_cuda(cudaGetLastError(), "k_eq_lut launch");
  if (rc || !out) return rc;
  if (((reinterpret_cast<uintptr_t>(bgr) ^ reinterpret_cast<uintptr_t>(out)) & 15u) == 0)
    k_eq_apply<true><<<eq_grid(run.units), kEqThreads, 0, st>>>(bgr, run, lut, out);
  else
    k_eq_apply<false><<<eq_grid(n / 16), kEqThreads, 0, st>>>(bgr, run, lut, out);
  return check_cuda(cudaGetLastError(), "k_eq_apply launch");
}

}  // namespace apap

using namespace apap;

extern "C" int apap_equalize_hist(const uint8_t *bgr, int h, int w, uint32_t *hist, uint8_t *lut, uint8_t *out,
                                  void *stream) {
  if (h <= 0 || w <= 0) return fail(APAP_E_BADARG, "equalize_hist: image sizes must be > 0");
  if ((long long)h * w > 2147483647LL) return fail(APAP_E_TOOBIG, "equalize_hist: image too large");
  if (!bgr || !hist || !lut) return fail(APAP_E_BADARG, "equalize_hist: null pointer");
  return launch_equalize_hist(bgr, h, w, hist, lut, out, static_cast<cudaStream_t>(stream));
}
