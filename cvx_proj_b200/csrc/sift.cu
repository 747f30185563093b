// SIFT descriptors at given keypoints -- cv.SIFT.compute at the keypoints of the reference's keypoint-pair producer
// (pyviz/utils.py:143-147: cv.KeyPoint(x, y, 1) -> octave 0, layer 0, angle -1), SURVEY 8f row N3.
//
// With provided octave-0 keypoints OpenCV builds one octave (firstOctave = 0, actualNOctaves = 1) and calcDescriptors
// reads only gpyr[0]: the gray image blurred once by sig = sqrtf(1.6^2 - 0.5^2) = 1.5198685f.  So two kernels:
//   k_sift_base : BGR uint8 -> gray (cv.cvtColor's 15-bit fixed point, bit-exact) -> 13-tap Gaussian, horizontal then
//                 vertical, BORDER_REFLECT_101 -> float32 [h][w] scratch (33 MB at 3840 x 2160, read back from L2 by
//                 the next kernel).
//   k_sift_desc : one warp per keypoint, calcSIFTDescriptor: gradients at the samples of a (2 radius + 1)^2 window,
//                 trilinear 4 x 4 x 8 histogram, fold, clip at 0.2 |h|, scale to 512, round and saturate to 0..255.
// The per-sample quantities that depend only on (size, angle) -- offsets, rbin, cbin, the Gaussian weight, the bin test
// -- come from a host table, so no device transcendental enters.  Every operation is rounded on its own
// (__fmul_rn / __fadd_rn / __fdiv_rn, no FMA contraction) and the histogram is updated sample by sample in OpenCV's
// order, which makes both kernels bit-identical to their numpy restatement (oracle/sift_oracle.py); that restatement
// is within +-2 per component of OpenCV's own SIMD build (almost every component equal).
#include <float.h>

#include "common.cuh"

namespace apap {

constexpr int kSiftD = 4, kSiftN = 8;                               // SIFT_DESCR_WIDTH, SIFT_DESCR_HIST_BINS
constexpr int kSiftDim = kSiftD * kSiftD * kSiftN;                  // 128
constexpr int kSiftSlots = (kSiftD + 2) * (kSiftD + 2) * (kSiftN + 2);  // 360-float histogram with padding cells
constexpr int kSiftR = 6;                                           // blur half-width: ksize = cvRound(sig * 8 + 1) | 1 = 13
// cv.getGaussianKernel(13, 1.5198685f, CV_32F): exp(-x^2 / 2 sig^2) normalised in float64, rounded to float32
__constant__ float kSiftTaps[2 * kSiftR + 1] = {
    0x1.c6a114p-14f, 0x1.334e76p-10f, 0x1.0d783cp-7f, 0x1.328774p-5f, 0x1.c45502p-4f, 0x1.b0f2f2p-3f, 0x1.0cc9bap-2f,
    0x1.b0f2f2p-3f, 0x1.c45502p-4f, 0x1.328774p-5f, 0x1.0d783cp-7f, 0x1.334e76p-10f, 0x1.c6a114p-14f};

constexpr int kBaseTW = 64, kBaseTH = 32, kBaseThreads = 256;       // output tile of k_sift_base
constexpr int kBaseInW = kBaseTW + 2 * kSiftR, kBaseInH = kBaseTH + 2 * kSiftR;   // 76 x 44 with the halo
constexpr int kBaseRun = 8;     // outputs per thread and pass: 20 shared loads for 8 x 13 taps (13 per output unblocked)

__device__ __forceinline__ int reflect101(int p, int n) {          // cv::borderInterpolate(p, n, BORDER_REFLECT_101)
  if (n == 1) return 0;
  while ((unsigned)p >= (unsigned)n) p = p < 0 ? -p : 2 * (n - 1) - p;
  return p;
}

// ((t0 x0 + t1 x1) + t2 x2) + ... for the kBaseRun outputs of x[0 .. kBaseRun + 12)
__device__ __forceinline__ void blur_run(const float (&x)[kBaseRun + 2 * kSiftR], float (&acc)[kBaseRun]) {
#pragma unroll
  for (int o = 0; o < kBaseRun; ++o) {
    acc[o] = __fmul_rn(kSiftTaps[0], x[o]);
#pragma unroll
    for (int k = 1; k <= 2 * kSiftR; ++k) acc[o] = __fadd_rn(acc[o], __fmul_rn(kSiftTaps[k], x[o + k]));
  }
}

// kLut: the image is seen through a per-channel LUT (lut: uint8 [3][256], B G R; staged in shared memory), the
// equalised image of csrc/equalize.cu without materialising it.  k_sift_base<false> ignores lut.
template <bool kLut>
__global__ void __launch_bounds__(kBaseThreads) k_sift_base(const uint8_t *__restrict__ bgr, int h, int w,
                                                            float *__restrict__ base, const uint8_t *__restrict__ lut) {
  __shared__ __align__(16) float gray[kBaseInH][kBaseInW];
  __shared__ __align__(16) float horiz[kBaseInH][kBaseTW];
  __shared__ uint8_t lut_s[kLut ? 3 * 256 : 1];
  if constexpr (kLut) {
    for (int i = threadIdx.x; i < 3 * 256; i += kBaseThreads) lut_s[i] = lut[i];
    __syncthreads();
  }
  const int x0 = blockIdx.x * kBaseTW, y0 = blockIdx.y * kBaseTH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int ty = warp; ty < kBaseInH; ty += kBaseThreads / 32) {
    const uint8_t *row = bgr + (size_t)reflect101(y0 + ty - kSiftR, h) * w * 3;
    for (int tx = lane; tx < kBaseInW; tx += 32) {
      const uint8_t *p = row + (size_t)reflect101(x0 + tx - kSiftR, w) * 3;
      // cv.cvtColor(COLOR_BGR2GRAY) for 8-bit input: 15-bit coefficients, rounded
      if constexpr (kLut)
        gray[ty][tx] = (float)((3735 * lut_s[p[0]] + 19235 * lut_s[256 + p[1]] + 9798 * lut_s[512 + p[2]] + (1 << 14)) >> 15);
      else
        gray[ty][tx] = (float)((3735 * p[0] + 19235 * p[1] + 9798 * p[2] + (1 << 14)) >> 15);
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < kBaseInH * (kBaseTW / kBaseRun); e += kBaseThreads) {      // horizontal taps
    const int ty = e / (kBaseTW / kBaseRun), tx0 = (e % (kBaseTW / kBaseRun)) * kBaseRun;
    float x[kBaseRun + 2 * kSiftR], acc[kBaseRun];
    const float4 *src = reinterpret_cast<const float4 *>(&gray[ty][tx0]);
#pragma unroll
    for (int q = 0; q < (kBaseRun + 2 * kSiftR) / 4; ++q) {
      const float4 v = src[q];
      x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
    }
    blur_run(x, acc);
    float4 *dst = reinterpret_cast<float4 *>(&horiz[ty][tx0]);
#pragma unroll
    for (int q = 0; q < kBaseRun / 4; ++q) dst[q] = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < (kBaseTH / kBaseRun) * kBaseTW; e += kBaseThreads) {     // vertical taps
    const int tx = e % kBaseTW, ty0 = (e / kBaseTW) * kBaseRun;
    float x[kBaseRun + 2 * kSiftR], acc[kBaseRun];
#pragma unroll
    for (int q = 0; q < kBaseRun + 2 * kSiftR; ++q) x[q] = horiz[ty0 + q][tx];
    blur_run(x, acc);
    if (x0 + tx < w) {
#pragma unroll
      for (int o = 0; o < kBaseRun; ++o)
        if (y0 + ty0 + o < h) base[(size_t)(y0 + ty0 + o) * w + x0 + tx] = acc[o];
    }
  }
}

// cv::fastAtan2(y, x) in degrees: degree-7 polynomial in min / (max + (float)DBL_EPSILON), then the quadrant fix-ups
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float c = __fdiv_rn(fminf(ax, ay), __fadd_rn(fmaxf(ax, ay), 0x1p-52f));
  const float c2 = __fmul_rn(c, c);
  float a = __fmul_rn(-0x1.4515b2p+1f, c2);                         // atan2_p7 .. p1 = (0.99979, -0.32581, 0.15558,
  a = __fmul_rn(__fadd_rn(a, 0x1.1d3f7ep+3f), c2);                  //   -0.04433) * (float)(180 / pi)
  a = __fmul_rn(__fadd_rn(a, -0x1.2aaddcp+4f), c2);
  a = __fmul_rn(__fadd_rn(a, 0x1.ca44dep+5f), c);
  if (!(ax >= ay)) a = __fsub_rn(90.f, a);
  if (x < 0.f) a = __fsub_rn(180.f, a);
  if (y < 0.f) a = __fsub_rn(360.f, a);
  return a;
}

constexpr int kDescWarps = 4;                                       // keypoints per CTA
constexpr int kHistPitch = kSiftSlots + 8;                          // slot -1 (guard) + 360 + padding

struct DescWarpSmem {
  float hist[kHistPitch];     // hist[0] = slot -1: a sample with o0 = -1 in the corner cell writes there, nothing reads it
  int idx[32];                // staged samples of the current batch: first histogram slot (guard included)
  float v[8][32];             //   and the 8 trilinear contributions v_rco000, 001, 010, 011, 100, 101, 110, 111
};

__global__ void __launch_bounds__(kDescWarps * 32) k_sift_desc(const float *__restrict__ base, int h, int w,
                                                               const float *__restrict__ pts, int n_kp,
                                                               const float *__restrict__ table, int n_samples, float ori,
                                                               float *__restrict__ desc) {
  __shared__ DescWarpSmem smem[kDescWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kp = blockIdx.x * kDescWarps + warp;
  if (kp >= n_kp) return;                                           // whole warps leave; no CTA barrier below
  DescWarpSmem &s = smem[warp];
  for (int e = lane; e < kHistPitch; e += 32) s.hist[e] = 0.f;
  // cvRound (half to even); far-away or non-finite points are clamped well outside the image: no sample is kept
  const int px = __float2int_rn(fminf(fmaxf(pts[2 * kp], -0x1p24f), 0x1p24f));
  const int py = __float2int_rn(fminf(fmaxf(pts[2 * kp + 1], -0x1p24f), 0x1p24f));
  const float bins_per_deg = 0x1.6c16c2p-6f;                        // n / 360.f
  // lane q < 8 adds contribution q of every staged sample: slot offsets 0, 1, n+2, n+3, (d+2)(n+2), +1, (d+3)(n+2), +1
  const int my_off = (lane & 1) + ((lane >> 1) & 1) * (kSiftN + 2) + (lane >> 2) * (kSiftD + 2) * (kSiftN + 2);
  __syncwarp();
  for (int b0 = 0; b0 < n_samples; b0 += 32) {
    const int sidx = b0 + lane;
    bool keep = false;
    if (sidx < n_samples) {
      const float *t = table + (size_t)sidx * 5;
      const int r = py + (int)__ldg(t), c = px + (int)__ldg(t + 1);
      if (r > 0 && r < h - 1 && c > 0 && c < w - 1) {
        const float rbin = __ldg(t + 2), cbin = __ldg(t + 3), wgt = __ldg(t + 4);
        const float *row = base + (size_t)r * w + c;
        const float dx = __fsub_rn(row[1], row[-1]);
        const float dy = __fsub_rn(row[-w], row[w]);
        const float o = fast_atan2_deg(dy, dx);
        const float mag = __fmul_rn(__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))), wgt);
        float obin = __fmul_rn(__fsub_rn(o, ori), bins_per_deg);
        const int r0 = __float2int_rd(rbin), c0 = __float2int_rd(cbin);
        int o0 = __float2int_rd(obin);
        const float rb = __fsub_rn(rbin, (float)r0), cb = __fsub_rn(cbin, (float)c0);
        obin = __fsub_rn(obin, (float)o0);
        if (o0 < 0) o0 += kSiftN;
        if (o0 >= kSiftN) o0 -= kSiftN;
        // o0 = -1 is OpenCV's own result for an orientation within 1 degree below ori - 360 (ori = 361 for angle -1):
        // its first contribution lands in slot n+1 of the previous cell (folded into that cell's bin 1)
        const int idx = ((r0 + 1) * (kSiftD + 2) + c0 + 1) * (kSiftN + 2) + o0 + 1;     // + 1: the guard slot
        keep = idx >= 0 && idx + (kSiftD + 3) * (kSiftN + 2) + 1 <= kSiftSlots;       // always, for a host-built table
        if (keep) {
          const float v_r1 = __fmul_rn(mag, rb), v_r0 = __fsub_rn(mag, v_r1);
          const float v_rc11 = __fmul_rn(v_r1, cb), v_rc10 = __fsub_rn(v_r1, v_rc11);
          const float v_rc01 = __fmul_rn(v_r0, cb), v_rc00 = __fsub_rn(v_r0, v_rc01);
          const float v_rco111 = __fmul_rn(v_rc11, obin), v_rco110 = __fsub_rn(v_rc11, v_rco111);
          const float v_rco101 = __fmul_rn(v_rc10, obin), v_rco100 = __fsub_rn(v_rc10, v_rco101);
          const float v_rco011 = __fmul_rn(v_rc01, obin), v_rco010 = __fsub_rn(v_rc01, v_rco011);
          const float v_rco001 = __fmul_rn(v_rc00, obin), v_rco000 = __fsub_rn(v_rc00, v_rco001);
          s.idx[lane] = idx;
          s.v[0][lane] = v_rco000; s.v[1][lane] = v_rco001; s.v[2][lane] = v_rco010; s.v[3][lane] = v_rco011;
          s.v[4][lane] = v_rco100; s.v[5][lane] = v_rco101; s.v[6][lane] = v_rco110; s.v[7][lane] = v_rco111;
        }
      }
    }
    unsigned todo = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    // commit in sample order: the 8 slots of one sample are distinct, so 8 lanes add them at once; samples one by one
    // keep OpenCV's summation order in every slot
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      if (lane < 8) {
        float *slot = s.hist + s.idx[src] + my_off;
        *slot = __fadd_rn(*slot, s.v[lane][src]);
      }
      __syncwarp();
    }
  }
  // fold the circular padding (bins n, n+1 -> 0, 1) of the 4 x 4 interior cells; lane l owns components l + 32 m
  float raw[4];
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const int comp = lane + 32 * m, cell = comp >> 3, bin = comp & 7;
    const int at = 1 + (((cell >> 2) + 1) * (kSiftD + 2) + (cell & 3) + 1) * (kSiftN + 2) + bin;
    raw[m] = bin < 2 ? __fadd_rn(s.hist[at], s.hist[at + kSiftN]) : s.hist[at];
  }
  float nrm2 = __fmul_rn(raw[0], raw[0]);
#pragma unroll
  for (int m = 1; m < 4; ++m) nrm2 = __fadd_rn(nrm2, __fmul_rn(raw[m], raw[m]));
#pragma unroll
  for (int off = 16; off; off >>= 1) nrm2 = __fadd_rn(nrm2, __shfl_xor_sync(0xffffffffu, nrm2, off));
  const float thr = __fmul_rn(__fsqrt_rn(nrm2), 0.2f);               // SIFT_DESCR_MAG_THR
#pragma unroll
  for (int m = 0; m < 4; ++m) raw[m] = fminf(raw[m], thr);
  nrm2 = __fmul_rn(raw[0], raw[0]);
#pragma unroll
  for (int m = 1; m < 4; ++m) nrm2 = __fadd_rn(nrm2, __fmul_rn(raw[m], raw[m]));
#pragma unroll
  for (int off = 16; off; off >>= 1) nrm2 = __fadd_rn(nrm2, __shfl_xor_sync(0xffffffffu, nrm2, off));
  const float scale = __fdiv_rn(512.f, fmaxf(__fsqrt_rn(nrm2), FLT_EPSILON));   // SIFT_INT_DESCR_FCTR
  float *out = desc + (size_t)kp * kSiftDim;
#pragma unroll
  for (int m = 0; m < 4; ++m) {                                     // saturate_cast<uchar>: round half to even, clamp
    const int q = __float2int_rn(__fmul_rn(raw[m], scale));
    out[lane + 32 * m] = (float)min(max(q, 0), 255);
  }
}

int launch_sift_describe(const uint8_t *bgr, int h, int w, const uint8_t *lut, const float *pts, int n_kp,
                         const float *table, int n_samples, float ori, float *base, float *desc, cudaStream_t st) {
  const dim3 grid((w + kBaseTW - 1) / kBaseTW, (h + kBaseTH - 1) / kBaseTH);
  if (lut)
    k_sift_base<true><<<grid, kBaseThreads, 0, st>>>(bgr, h, w, base, lut);
  else
    k_sift_base<false><<<grid, kBaseThreads, 0, st>>>(bgr, h, w, base, nullptr);
  int rc = check_cuda(cudaGetLastError(), lut ? "k_sift_base<true> launch" : "k_sift_base launch");
  if (rc) return rc;
  k_sift_desc<<<(n_kp + kDescWarps - 1) / kDescWarps, kDescWarps * 32, 0, st>>>(base, h, w, pts, n_kp, table, n_samples,
                                                                                  ori, desc);
  return check_cuda(cudaGetLastError(), "k_sift_desc launch");
}

}  // namespace apap

using namespace apap;

// the argument checks of both entry points; lut is null for the plain image
static int sift_describe_checked(const uint8_t *bgr, int h, int w, const uint8_t *lut, const float *pts, int n_kp,
                                 const float *table, int n_samples, float ori, float *base_scratch, float *desc,
                                 void *stream) {
  if (n_kp < 0 || n_samples < 0) return fail(APAP_E_BADARG, "sift_describe: negative size");
  if (n_kp == 0) return 0;
  if (h <= 0 || w <= 0) return fail(APAP_E_BADARG, "sift_describe: image sizes must be > 0");
  if ((long long)h * w > 2147483647LL || h >= (1 << 24) || w >= (1 << 24))
    return fail(APAP_E_TOOBIG, "sift_describe: image too large");
  if (!bgr || !pts || (!table && n_samples) || !base_scratch || !desc) return fail(APAP_E_BADARG, "sift_describe: null pointer");
  // ori = 360 - angle for angle in [-1, 360): keeps every trilinear slot inside the histogram
  if (!(ori >= 0.f && ori <= 361.f)) return fail(APAP_E_BADARG, "sift_describe: ori must be in [0, 361]");
  return launch_sift_describe(bgr, h, w, lut, pts, n_kp, table, n_samples, ori, base_scratch, desc,
                              static_cast<cudaStream_t>(stream));
}

extern "C" int apap_sift_describe(const uint8_t *bgr, int h, int w, const float *pts, int n_kp, const float *table,
                                  int n_samples, float ori, float *base_scratch, float *desc, void *stream) {
  return sift_describe_checked(bgr, h, w, nullptr, pts, n_kp, table, n_samples, ori, base_scratch, desc, stream);
}

extern "C" int apap_sift_describe_lut(const uint8_t *bgr, int h, int w, const uint8_t *lut, const float *pts, int n_kp,
                                      const float *table, int n_samples, float ori, float *base_scratch, float *desc,
                                      void *stream) {
  if (!lut) return fail(APAP_E_BADARG, "sift_describe_lut: null lut");
  return sift_describe_checked(bgr, h, w, lut, pts, n_kp, table, n_samples, ori, base_scratch, desc, stream);
}
