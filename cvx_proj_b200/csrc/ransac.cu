// RANSAC homography: the hypothesis loop of cv.findHomography(src, dst, cv.RANSAC, thr) (OpenCV 4.x,
// RANSACPointSetRegistrator::run) of the reference's keypoint-pair producer (baseline_stitch_test.py:41).  The device
// produces every hypothesis the loop can draw, up to max_iters, and its inlier count; the host scans the counts with
// the adaptive stop (RANSACUpdateNumIters), so the same subsets, counts and choice come out as in OpenCV.
//   k_ransac_sample : one warp.  Lane 0 runs cv::RNG(0xFFFFFFFFFFFFFFFF) serially and draws 32 candidate subsets of 4
//                     distinct indices (getSubset); the 32 lanes run checkSubset on them at once; lane 0 keeps the
//                     accepted ones in draw order.  10000 rejected candidates in a row end the sequence (getSubset
//                     fails: the loop breaks, or has no model when that happens on iteration 0).  One warp (CTA)
//                     per pair, each pair on its own cv::RNG(0xFFFFFFFFFFFFFFFF) like a separate findHomography call.
//   k_ransac_fit    : one thread per hypothesis: runKernel in float64 step by step (centroid, mean absolute
//                     deviation, the DBL_EPSILON exit, LtL, cv::eigen's cyclic Jacobi, H = invHnorm V8 Hnorm2 / H22),
//                     every operation rounded on its own, so each hypothesis is OpenCV's bit for bit.  One thread per
//                     (pair, hypothesis).
//   k_ransac_score  : a CTA takes 32 hypotheses of one pair and walks that pair's points 1024 at a time with a grid
//                     stride: computeError in float32 with every operation rounded on its own (no contraction),
//                     err <= (float)(thr * thr), integer counts by warp reductions and atomics (exact in any order).
//                     Invalid hypotheses (0 models) keep count -1.
// A batch is independent point sets stored back to back, pair p at [offsets[p], offsets[p + 1]); every output is laid
// out [batch][max_iters]..., and pair p's record is the record of a single call on its points.  The single call
// (apap_ransac_homography) is a batch of one with offsets == nullptr: its pair is [0, max_n).
#include <cfloat>

#include "common.cuh"

namespace apap {

constexpr int kRansacMaxAttempts = 10000;          // getSubset(..., 10000) in RANSACPointSetRegistrator::run
constexpr unsigned long long kRngCoeff = 4164903690ull;
constexpr int kFitThreads = 128;
constexpr int kScoreThreads = 256;
constexpr int kScoreHyps = 32;                     // hypotheses per CTA
constexpr int kScorePtsPerThread = 4;
constexpr int kScorePts = kScoreThreads * kScorePtsPerThread;
constexpr int kHf = 9;                             // workspace row: (float)H[0..7], valid flag
constexpr int kMaxGridZ = 65535;                   // pairs per score launch

// [begin, end) of pair p's points
__device__ __forceinline__ int2 pair_range(const int *__restrict__ offsets, int p, int max_n) {
  return offsets ? make_int2(offsets[p], offsets[p + 1]) : make_int2(0, max_n);
}

// ------------------------------------------------------------------------------------------------ checkSubset
// haveCollinearPoints(m, 4): the last point against the line through each pair of the earlier three.  Point2f
// differences are float32, widened to double for the cross product and the FLT_EPSILON bound.
__device__ __forceinline__ bool have_collinear(const float2 (&p)[4]) {
  bool col = false;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const double dx1 = (double)__fsub_rn(p[j].x, p[3].x), dy1 = (double)__fsub_rn(p[j].y, p[3].y);
#pragma unroll
    for (int k = 0; k < j; ++k) {
      const double dx2 = (double)__fsub_rn(p[k].x, p[3].x), dy2 = (double)__fsub_rn(p[k].y, p[3].y);
      const double cross = __dsub_rn(__dmul_rn(dx2, dy1), __dmul_rn(dy2, dx1));
      const double bound = __dmul_rn((double)FLT_EPSILON,
                                     __dadd_rn(__dadd_rn(__dadd_rn(fabs(dx1), fabs(dy1)), fabs(dx2)), fabs(dy2)));
      col |= fabs(cross) <= bound;
    }
  }
  return col;
}

// determinant(Matx33d(x0, y0, 1, x1, y1, 1, x2, y2, 1)) in Matx_DetOp<double, 3>'s order
__device__ __forceinline__ double det3(float2 a, float2 b, float2 c) {
  const double x0 = a.x, y0 = a.y, x1 = b.x, y1 = b.y, x2 = c.x, y2 = c.y;
  return __dadd_rn(__dsub_rn(__dmul_rn(x0, __dsub_rn(y1, y2)), __dmul_rn(y0, __dsub_rn(x1, x2))),
                   __dsub_rn(__dmul_rn(x1, y2), __dmul_rn(x2, y1)));
}

__device__ bool check_subset(const float2 (&s)[4], const float2 (&d)[4]) {
  if (have_collinear(s) || have_collinear(d)) return false;
  int negative = 0;                                 // triangles {0,1,2}, {1,2,3}, {0,2,3}, {0,1,3}
  negative += __dmul_rn(det3(s[0], s[1], s[2]), det3(d[0], d[1], d[2])) < 0.0;
  negative += __dmul_rn(det3(s[1], s[2], s[3]), det3(d[1], d[2], d[3])) < 0.0;
  negative += __dmul_rn(det3(s[0], s[2], s[3]), det3(d[0], d[2], d[3])) < 0.0;
  negative += __dmul_rn(det3(s[0], s[1], s[3]), det3(d[0], d[1], d[3])) < 0.0;
  return negative == 0 || negative == 4;
}

// ------------------------------------------------------------------------------------------------ sampling
__device__ __forceinline__ uint32_t rng_uniform(unsigned long long &state, uint32_t n) {   // RNG::uniform(0, n)
  state = (unsigned long long)(uint32_t)state * kRngCoeff + (state >> 32);
  return (uint32_t)state % n;
}

__global__ void __launch_bounds__(32) k_ransac_sample(const float2 *__restrict__ src, const float2 *__restrict__ dst,
                                                      const int *__restrict__ offsets, int max_n, int max_iters,
                                                      int4 *__restrict__ subsets, int *__restrict__ n_sampled) {
  __shared__ int4 cand[32];
  const int lane = threadIdx.x, pair = blockIdx.x;
  const int2 r = pair_range(offsets, pair, max_n);
  const int n = r.y - r.x;
  if (n < 5) {                                      // 4 points are a single fit; fewer could never draw 4 distinct
    if (lane == 0) n_sampled[pair] = 0;
    return;
  }
  src += r.x;
  dst += r.x;
  subsets += (size_t)pair * max_iters;
  unsigned long long state = ~0ull;                 // lane 0's RNG
  int accepted = 0, run = 0;                        // run: rejected candidates since the last accepted one
  bool done = false;
  while (!done) {
    if (lane == 0) {
      for (int c = 0; c < 32; ++c) {
        int idx[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          int j;
          bool dup;
          do {
            j = (int)rng_uniform(state, (uint32_t)n);
            dup = false;
#pragma unroll
            for (int k = 0; k < i; ++k) dup |= idx[k] == j;
          } while (dup);
          idx[i] = j;
        }
        cand[c] = make_int4(idx[0], idx[1], idx[2], idx[3]);
      }
    }
    __syncwarp();
    const int4 q = cand[lane];
    const float2 s[4] = {src[q.x], src[q.y], src[q.z], src[q.w]};
    const float2 d[4] = {dst[q.x], dst[q.y], dst[q.z], dst[q.w]};
    const unsigned ok = __ballot_sync(0xffffffffu, check_subset(s, d));
    if (lane == 0) {
      for (int c = 0; c < 32 && !done; ++c) {
        if ((ok >> c) & 1u) {
          subsets[accepted++] = cand[c];
          run = 0;
          done = accepted == max_iters;
        } else if (++run == kRansacMaxAttempts) {
          done = true;
        }
      }
    }
    done = __shfl_sync(0xffffffffu, done, 0);
    __syncwarp();
  }
  if (lane == 0) n_sampled[pair] = accepted;
}

// ------------------------------------------------------------------------------------------------ runKernel
// hypot of OpenCV's lapack.cpp (not std::hypot)
__device__ __forceinline__ double cv_hypot(double a, double b) {
  a = fabs(a);
  b = fabs(b);
  if (a > b) {
    b = __ddiv_rn(b, a);
    return __dmul_rn(a, __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(b, b))));
  }
  if (b > 0) {
    a = __ddiv_rn(a, b);
    return __dmul_rn(b, __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(a, a))));
  }
  return 0.0;
}

__device__ __forceinline__ void jacobi_rotate(double &v0, double &v1, double c, double s) {
  const double a0 = v0, b0 = v1;
  v0 = __dsub_rn(__dmul_rn(a0, c), __dmul_rn(b0, s));
  v1 = __dadd_rn(__dmul_rn(a0, s), __dmul_rn(b0, c));
}

__device__ __forceinline__ void jacobi_row_max(const double *A, int k, int *ind_r) {
  int m = k + 1;
  double mv = fabs(A[9 * k + k + 1]);
  for (int i = k + 2; i < 9; ++i) {
    const double val = fabs(A[9 * k + i]);
    if (mv < val) mv = val, m = i;
  }
  ind_r[k] = m;
}

__device__ __forceinline__ void jacobi_col_max(const double *A, int k, int *ind_c) {
  int m = 0;
  double mv = fabs(A[k]);
  for (int i = 1; i < k; ++i) {
    const double val = fabs(A[9 * i + k]);
    if (mv < val) mv = val, m = i;
  }
  ind_c[k] = m;
}

// cv::eigen of a symmetric 9x9 float64 matrix, i.e. JacobiImpl_ of OpenCV 4.x core/src/lapack.cpp step by step: the
// largest off-diagonal element of the upper triangle as pivot (through per-row and per-column maxima), at most
// 30 n^2 rotations, stop at |pivot| <= DBL_EPSILON, every operation rounded on its own.  A (upper triangle read and
// destroyed), W and V (eigenvectors as rows) as OpenCV holds them; OpenCV then sorts the eigenvalues descending by
// selection sort, which is replayed on a row permutation.  Returns the row of V that the sort puts last.
__device__ __noinline__ int jacobi9(double *A, double *W, double *V) {
  int ind_r[9], ind_c[9];
  for (int i = 0; i < 81; ++i) V[i] = (i / 9 == i % 9) ? 1.0 : 0.0;
  for (int k = 0; k < 9; ++k) {
    W[k] = A[10 * k];
    if (k < 8) jacobi_row_max(A, k, ind_r);
    if (k > 0) jacobi_col_max(A, k, ind_c);
  }
  for (int iters = 0; iters < 9 * 9 * 30; ++iters) {
    int k = 0;
    double mv = fabs(A[ind_r[0]]);
    for (int i = 1; i < 8; ++i) {
      const double val = fabs(A[9 * i + ind_r[i]]);
      if (mv < val) mv = val, k = i;
    }
    int l = ind_r[k];
    for (int i = 1; i < 9; ++i) {
      const double val = fabs(A[9 * ind_c[i] + i]);
      if (mv < val) mv = val, k = ind_c[i], l = i;
    }
    const double p = A[9 * k + l];
    if (fabs(p) <= DBL_EPSILON) break;
    const double y = __dmul_rn(__dsub_rn(W[l], W[k]), 0.5);
    double t = __dadd_rn(fabs(y), cv_hypot(p, y));
    double s = cv_hypot(p, t);
    const double c = __ddiv_rn(t, s);
    s = __ddiv_rn(p, s);
    t = __dmul_rn(__ddiv_rn(p, t), p);
    if (y < 0) s = -s, t = -t;
    A[9 * k + l] = 0.0;
    W[k] = __dsub_rn(W[k], t);
    W[l] = __dadd_rn(W[l], t);
    for (int i = 0; i < k; ++i) jacobi_rotate(A[9 * i + k], A[9 * i + l], c, s);
    for (int i = k + 1; i < l; ++i) jacobi_rotate(A[9 * k + i], A[9 * i + l], c, s);
    for (int i = l + 1; i < 9; ++i) jacobi_rotate(A[9 * k + i], A[9 * l + i], c, s);
    for (int i = 0; i < 9; ++i) jacobi_rotate(V[9 * k + i], V[9 * l + i], c, s);
    for (int j = 0; j < 2; ++j) {
      const int idx = j == 0 ? k : l;
      if (idx < 8) jacobi_row_max(A, idx, ind_r);
      if (idx > 0) jacobi_col_max(A, idx, ind_c);
    }
  }
  int row[9];
  for (int i = 0; i < 9; ++i) row[i] = i;
  for (int k = 0; k < 8; ++k) {
    int m = k;
    for (int i = k + 1; i < 9; ++i)
      if (W[m] < W[i]) m = i;
    if (k != m) {
      const double w = W[m];
      W[m] = W[k];
      W[k] = w;
      const int r = row[m];
      row[m] = row[k];
      row[k] = r;
    }
  }
  return row[8];
}

// c = a b for row-major 3x3 float64, each entry ((a0 b0 + a1 b1) + a2 b2) with every operation rounded on its own
__device__ __forceinline__ void mat3(const double (&a)[9], const double (&b)[9], double (&c)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      c[3 * i + j] = __dadd_rn(__dadd_rn(__dmul_rn(a[3 * i], b[j]), __dmul_rn(a[3 * i + 1], b[3 + j])),
                               __dmul_rn(a[3 * i + 2], b[6 + j]));
}

__global__ void __launch_bounds__(kFitThreads) k_ransac_fit(const float2 *__restrict__ src,
                                                            const float2 *__restrict__ dst,
                                                            const int *__restrict__ offsets, int max_n, int batch,
                                                            int max_iters, const int4 *__restrict__ subsets,
                                                            const int *__restrict__ n_sampled,
                                                            double *__restrict__ hyps, float *__restrict__ hf,
                                                            int *__restrict__ counts) {
  const int h = blockIdx.x * kFitThreads + threadIdx.x;   // (pair, hypothesis); batch * max_iters <= 2^20
  const int pair = h / max_iters;
  if (pair >= batch || h - pair * max_iters >= n_sampled[pair]) return;
  const int base = pair_range(offsets, pair, max_n).x;
  const int4 q = subsets[h];
  const int id[4] = {q.x, q.y, q.z, q.w};
  float2 M[4], m[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    M[i] = src[base + id[i]];
    m[i] = dst[base + id[i]];
  }
  double cmx = 0, cmy = 0, cMx = 0, cMy = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    cmx = __dadd_rn(cmx, m[i].x); cmy = __dadd_rn(cmy, m[i].y);
    cMx = __dadd_rn(cMx, M[i].x); cMy = __dadd_rn(cMy, M[i].y);
  }
  cmx = __ddiv_rn(cmx, 4.0); cmy = __ddiv_rn(cmy, 4.0); cMx = __ddiv_rn(cMx, 4.0); cMy = __ddiv_rn(cMy, 4.0);
  double smx = 0, smy = 0, sMx = 0, sMy = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    smx = __dadd_rn(smx, fabs(__dsub_rn(m[i].x, cmx))); smy = __dadd_rn(smy, fabs(__dsub_rn(m[i].y, cmy)));
    sMx = __dadd_rn(sMx, fabs(__dsub_rn(M[i].x, cMx))); sMy = __dadd_rn(sMy, fabs(__dsub_rn(M[i].y, cMy)));
  }
  double *out = hyps + (size_t)h * 9;
  float *outf = hf + (size_t)h * kHf;
  if (fabs(smx) < DBL_EPSILON || fabs(smy) < DBL_EPSILON || fabs(sMx) < DBL_EPSILON ||
      fabs(sMy) < DBL_EPSILON) {                  // runKernel returns 0 models
#pragma unroll
    for (int i = 0; i < 9; ++i) out[i] = __longlong_as_double(0x7ff8000000000000ll);
    outf[8] = 0.f;
    counts[h] = -1;
    return;
  }
  smx = __ddiv_rn(4.0, smx); smy = __ddiv_rn(4.0, smy); sMx = __ddiv_rn(4.0, sMx); sMy = __ddiv_rn(4.0, sMy);
  double A[81], V[81], W[9];                        // LtL (upper triangle), eigenvectors as rows, eigenvalues
#pragma unroll
  for (int i = 0; i < 81; ++i) A[i] = 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double x = __dmul_rn(__dsub_rn(m[i].x, cmx), smx), y = __dmul_rn(__dsub_rn(m[i].y, cmy), smy);
    const double X = __dmul_rn(__dsub_rn(M[i].x, cMx), sMx), Y = __dmul_rn(__dsub_rn(M[i].y, cMy), sMy);
    const double lx[9] = {X, Y, 1.0, 0.0, 0.0, 0.0, -__dmul_rn(x, X), -__dmul_rn(x, Y), -x};
    const double ly[9] = {0.0, 0.0, 0.0, X, Y, 1.0, -__dmul_rn(y, X), -__dmul_rn(y, Y), -y};
#pragma unroll
    for (int j = 0; j < 9; ++j)
#pragma unroll
      for (int k = j; k < 9; ++k)
        A[9 * j + k] = __dadd_rn(A[9 * j + k], __dadd_rn(__dmul_rn(lx[j], lx[k]), __dmul_rn(ly[j], ly[k])));
  }
  const int r8 = jacobi9(A, W, V);                  // cv::eigen: the row of V with the smallest eigenvalue
  double v[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) v[i] = V[9 * r8 + i];
  // H = invHnorm * H0 * Hnorm2 as cv::gemm computes it: every term of each dot product, in order
  const double inv_hnorm[9] = {__ddiv_rn(1.0, smx), 0.0, cmx, 0.0, __ddiv_rn(1.0, smy), cmy, 0.0, 0.0, 1.0};
  const double hnorm2[9] = {sMx, 0.0, __dmul_rn(-cMx, sMx), 0.0, sMy, __dmul_rn(-cMy, sMy), 0.0, 0.0, 1.0};
  double t[9], H[9];
  mat3(inv_hnorm, v, t);
  mat3(t, hnorm2, H);
  const double s22 = __ddiv_rn(1.0, H[8]);
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const double e = __dmul_rn(H[i], s22);
    out[i] = e;
    if (i < 8) outf[i] = (float)e;
  }
  outf[8] = 1.f;
  counts[h] = 0;
}

// ------------------------------------------------------------------------------------------------ computeError
__global__ void __launch_bounds__(kScoreThreads) k_ransac_score(const float2 *__restrict__ src,
                                                                const float2 *__restrict__ dst,
                                                                const int *__restrict__ offsets, int max_n,
                                                                int pair0, int max_iters,
                                                                const float *__restrict__ hf,
                                                                const int *__restrict__ n_sampled, float thr_sq,
                                                                int *__restrict__ counts) {
  __shared__ float hs[kScoreHyps][kHf];
  __shared__ int cnt[kScoreHyps];
  const int pair = pair0 + blockIdx.z;
  const size_t h0 = (size_t)pair * max_iters + blockIdx.y * kScoreHyps;   // first hypothesis of the CTA
  const int nh = min(kScoreHyps, n_sampled[pair] - (int)blockIdx.y * kScoreHyps);
  if (nh <= 0) return;
  const int2 r = pair_range(offsets, pair, max_n);
  const int n = r.y - r.x;
  src += r.x;
  dst += r.x;
  for (int i = threadIdx.x; i < nh * kHf; i += kScoreThreads) hs[i / kHf][i % kHf] = hf[h0 * kHf + i];
  if (threadIdx.x < kScoreHyps) cnt[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (int chunk = blockIdx.x; chunk * kScorePts < n; chunk += gridDim.x) {   // a pair beyond max_n is still counted
    float2 M[kScorePtsPerThread], m[kScorePtsPerThread];
    bool live[kScorePtsPerThread];
    const int p0 = chunk * kScorePts + threadIdx.x;
#pragma unroll
    for (int k = 0; k < kScorePtsPerThread; ++k) {
      const int p = p0 + k * kScoreThreads;
      live[k] = p < n;
      M[k] = live[k] ? src[p] : make_float2(0.f, 0.f);
      m[k] = live[k] ? dst[p] : make_float2(0.f, 0.f);
    }
    for (int j = 0; j < nh; ++j) {
      if (hs[j][8] == 0.f) continue;                // invalid hypothesis: uniform across the CTA
      const float *H = hs[j];
      int c = 0;
#pragma unroll
      for (int k = 0; k < kScorePtsPerThread; ++k) {
        const float x = M[k].x, y = M[k].y;
        const float ww = __fdiv_rn(1.f, __fadd_rn(__fadd_rn(__fmul_rn(H[6], x), __fmul_rn(H[7], y)), 1.f));
        const float dx = __fsub_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(H[0], x), __fmul_rn(H[1], y)), H[2]), ww), m[k].x);
        const float dy = __fsub_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(H[3], x), __fmul_rn(H[4], y)), H[5]), ww), m[k].y);
        const float e = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        c += (live[k] && e <= thr_sq) ? 1 : 0;
      }
      c = __reduce_add_sync(0xffffffffu, c);
      if (lane == 0 && c) atomicAdd(&cnt[j], c);
    }
  }
  __syncthreads();
  if (threadIdx.x < nh && hs[threadIdx.x][8] != 0.f && cnt[threadIdx.x]) atomicAdd(counts + h0 + threadIdx.x, cnt[threadIdx.x]);
}

static size_t ransac_workspace(size_t hyps) {
  return (hyps * kHf * sizeof(float) + 255) & ~(size_t)255;
}

// offsets == nullptr: one pair of max_n points
int launch_ransac(const float2 *src, const float2 *dst, const int *offsets, int batch, int max_n, double threshold,
                  int max_iters, float *hf, int4 *subsets, double *hyps, int *counts, int *n_sampled, cudaStream_t st) {
  k_ransac_sample<<<batch, 32, 0, st>>>(src, dst, offsets, max_n, max_iters, subsets, n_sampled);
  int rc = check_cuda(cudaGetLastError(), "k_ransac_sample launch");
  if (rc) return rc;
  const int total = batch * max_iters;
  k_ransac_fit<<<(total + kFitThreads - 1) / kFitThreads, kFitThreads, 0, st>>>(src, dst, offsets, max_n, batch, max_iters,
                                                                                subsets, n_sampled, hyps, hf, counts);
  rc = check_cuda(cudaGetLastError(), "k_ransac_fit launch");
  if (rc) return rc;
  const float thr_sq = (float)(threshold * threshold);
  for (int pair0 = 0; pair0 < batch; pair0 += kMaxGridZ) {
    const dim3 grid(max((max_n + kScorePts - 1) / kScorePts, 1), (max_iters + kScoreHyps - 1) / kScoreHyps,
                    min(batch - pair0, kMaxGridZ));
    k_ransac_score<<<grid, kScoreThreads, 0, st>>>(src, dst, offsets, max_n, pair0, max_iters, hf, n_sampled, thr_sq,
                                                   counts);
    rc = check_cuda(cudaGetLastError(), "k_ransac_score launch");
    if (rc) return rc;
  }
  return 0;
}

}  // namespace apap

using namespace apap;

extern "C" int apap_ransac_workspace_bytes(int max_iters, size_t *bytes) {
  if (max_iters < 1 || max_iters > APAP_RANSAC_MAX_ITERS)
    return fail(APAP_E_BADARG, "ransac: max_iters must be in [1, APAP_RANSAC_MAX_ITERS]");
  if (!bytes) return fail(APAP_E_BADARG, "ransac: null pointer");
  *bytes = ransac_workspace(max_iters);
  return 0;
}

static int check_ransac_args(double threshold, const void *src, const void *dst, const void *workspace,
                             size_t workspace_bytes, size_t hyps_total, const int *subsets, const double *hyps,
                             const int *counts, const int *n_sampled) {
  if (!(threshold > 0.0) || !isfinite(threshold)) return fail(APAP_E_BADARG, "ransac: threshold must be finite and > 0");
  if (!src || !dst || !workspace || !subsets || !hyps || !counts || !n_sampled)
    return fail(APAP_E_BADARG, "ransac: null pointer");
  if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 7u)
    return fail(APAP_E_BADARG, "ransac: src and dst must be 8-byte aligned");
  if ((reinterpret_cast<uintptr_t>(subsets) & 15u) || (reinterpret_cast<uintptr_t>(workspace) & 15u))
    return fail(APAP_E_BADARG, "ransac: subsets and workspace must be 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(hyps) & 7u) return fail(APAP_E_BADARG, "ransac: hyps must be 8-byte aligned");
  if ((reinterpret_cast<uintptr_t>(counts) | reinterpret_cast<uintptr_t>(n_sampled)) & 3u)
    return fail(APAP_E_BADARG, "ransac: counts and n_sampled must be 4-byte aligned");
  if (workspace_bytes < ransac_workspace(hyps_total)) return fail(APAP_E_BADARG, "ransac: workspace too small");
  return 0;
}

extern "C" int apap_ransac_homography(const float *src, const float *dst, int n, double threshold, int max_iters,
                                      void *workspace, size_t workspace_bytes, int *subsets, double *hyps, int *counts,
                                      int *n_sampled, void *stream) {
  if (n < 5) return fail(APAP_E_BADARG, "ransac: n must be >= 5 (4 points are a single fit, no sampling)");
  if (max_iters < 1 || max_iters > APAP_RANSAC_MAX_ITERS)
    return fail(APAP_E_BADARG, "ransac: max_iters must be in [1, APAP_RANSAC_MAX_ITERS]");
  const int rc = check_ransac_args(threshold, src, dst, workspace, workspace_bytes, max_iters, subsets, hyps, counts,
                                   n_sampled);
  if (rc) return rc;
  return launch_ransac(reinterpret_cast<const float2 *>(src), reinterpret_cast<const float2 *>(dst), nullptr, 1, n,
                       threshold, max_iters, static_cast<float *>(workspace), reinterpret_cast<int4 *>(subsets), hyps,
                       counts, n_sampled, static_cast<cudaStream_t>(stream));
}

static bool batch_fits(int batch, int max_iters) {
  return batch >= 1 && max_iters >= 1 && (long long)batch * max_iters <= APAP_RANSAC_MAX_ITERS;
}

extern "C" int apap_ransac_batch_workspace_bytes(int batch, int max_iters, size_t *bytes) {
  if (!batch_fits(batch, max_iters))
    return fail(APAP_E_BADARG, "ransac batch: batch and max_iters must be >= 1 with batch * max_iters <= "
                               "APAP_RANSAC_MAX_ITERS");
  if (!bytes) return fail(APAP_E_BADARG, "ransac: null pointer");
  *bytes = ransac_workspace((size_t)batch * max_iters);
  return 0;
}

extern "C" int apap_ransac_homography_batch(const float *src, const float *dst, const int *offsets, int batch,
                                            int max_n, double threshold, int max_iters, void *workspace,
                                            size_t workspace_bytes, int *subsets, double *hyps, int *counts,
                                            int *n_sampled, void *stream) {
  if (!batch_fits(batch, max_iters))
    return fail(APAP_E_BADARG, "ransac batch: batch and max_iters must be >= 1 with batch * max_iters <= "
                               "APAP_RANSAC_MAX_ITERS");
  if (max_n < 0) return fail(APAP_E_BADARG, "ransac batch: max_n must be >= 0");
  if (!offsets) return fail(APAP_E_BADARG, "ransac: null pointer");
  if (reinterpret_cast<uintptr_t>(offsets) & 3u) return fail(APAP_E_BADARG, "ransac batch: offsets must be 4-byte aligned");
  const int rc = check_ransac_args(threshold, src, dst, workspace, workspace_bytes, (size_t)batch * max_iters, subsets,
                                   hyps, counts, n_sampled);
  if (rc) return rc;
  return launch_ransac(reinterpret_cast<const float2 *>(src), reinterpret_cast<const float2 *>(dst), offsets, batch,
                       max_n, threshold, max_iters, static_cast<float *>(workspace), reinterpret_cast<int4 *>(subsets),
                       hyps, counts, n_sampled, static_cast<cudaStream_t>(stream));
}
