// K1 -- moving-DLT weights + Gram contraction (reference pyviz/apap.py:150-152,159).
//
// For every cell c and keypoint i:   w2 = max(exp(-2 |v_c - x_i| / sigma^2), gamma^2)
//                                    S_t(c) += w2 * P[i][t],  t = 0..23
// i.e. the contraction [cells x N of w^2] . [N x 24] with the weights generated on the fly and
// never written to memory.  FP32 SIMT on the FMA pipe, issued as packed FFMA2 (two FP32 lanes per
// instruction, sm_100): one thread owns R = 4 cells (register tile 4 x 24 accumulators = 48
// register pairs); a CTA is ONE warp = 128 cells x one keypoint split, so the grid is a sea of
// independent warps (12 resident per SM) that balances to within one warp per SM and needs no
// CTA barrier.  Each warp stages its keypoint rows (24 terms + the pre-scaled keypoint) in its own
// shared-memory ring by TMA bulk copies (cp.async.bulk + mbarrier, double buffered) and reads them
// back as warp-wide broadcast LDS.128: 7 loads feed 4 x 12 FFMA2.  The weight costs 2 packed adds,
// a packed multiply and a packed FMA per cell pair, MUFU.SQRT + MUFU.EX2 per cell and one FMNMX;
// coordinates arrive pre-scaled by s = 2 log2(e) / sigma^2 so that w2 = max(2^-|s v - s x|, gamma^2).
//
// Accuracy: each FP32 accumulator sums at most kMaxChainChunks*128 = 1024 keypoints (one
// "split"); the splits are written as partial sums and combined in float64 by K2.  The split
// boundaries depend only on the keypoint count, so a cell's result does not depend on how the
// grid is sharded across GPUs.
#include "common.cuh"

namespace apap {

constexpr int kGramThreads = 32;                 // one warp per CTA
constexpr int kGramCells = 4;                    // cells per thread (register tile)
constexpr int kGramTile = kGramThreads * kGramCells;   // 128 cells per warp
constexpr int kStages = 2;
constexpr int kStageRows = 64;                   // keypoint rows per TMA stage (half an APAP_KP_CHUNK)
constexpr uint32_t kStageBytes = kStageRows * kRowFloats * sizeof(float);   // 7168
static_assert(kChunk % kStageRows == 0, "a chunk must be a whole number of stages");

static int g_sm_count = 0;
int sm_count_cached() {
  if (g_sm_count == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      g_sm_count = n;
    else
      return 148;   // B200; only reached without a device (planning on the host)
  }
  return g_sm_count;
}

constexpr int kSplitDiv = 4;   // target number of keypoint splits
GramPlan make_gram_plan(int cells, int n_kp_padded, int engine) {
  GramPlan p;
  const int n_chunks = n_kp_padded / kChunk;
  int cps = (n_chunks + kSplitDiv - 1) / kSplitDiv;   // a function of N only (see header comment)
  if (cps < 1) cps = 1;
  const int cap = engine == APAP_GRAM_TCGEN05 ? kMaxSplitChunksTc : kMaxChainChunks;
  if (cps > cap) cps = cap;
  p.chunks_per_split = cps;
  p.k_splits = (n_chunks + cps - 1) / cps;
  if (p.k_splits < 1) p.k_splits = 1;
  p.cells_per_thread = kGramCells;
  const int pad = 512;                          // partial rows stay 2 KB aligned whatever the tile
  p.cells_padded = (cells + pad - 1) / pad * pad;
  p.cell_tiles = (cells + kGramTile - 1) / kGramTile;
  return p;
}

__global__ void __launch_bounds__(kGramThreads, 12) k_gram(const float *__restrict__ kp_table,
                                                           const float *__restrict__ anchors, int cells,
                                                           int cells_padded, int n_chunks, int chunks_per_split,
                                                           int k_splits, float gamma_sq,
                                                           float *__restrict__ partials) {
  constexpr int R = kGramCells;
  __shared__ __align__(128) float stage[kStages][kStageRows * kRowFloats];
  __shared__ __align__(8) uint64_t full_bar[kStages];

  const int lane = threadIdx.x;
  const int split = blockIdx.y;
  const int scene = blockIdx.z;
  const int c_begin = split * chunks_per_split;
  const int c_end = min(n_chunks, c_begin + chunks_per_split);
  const int n_local = (c_end - c_begin) * (kChunk / kStageRows);      // stages in this split

  kp_table += (size_t)scene * n_chunks * (kChunk * kRowFloats);
  anchors += (size_t)scene * cells * 2;
  partials += (size_t)scene * k_splits * kTerms * cells_padded;

  // cells of this thread: tile base + r * 32 + lane; anchors (already scaled) as pairs (r, r + 1)
  const int cell0 = blockIdx.x * kGramTile + lane;
  float2 ax[R / 2], ay[R / 2];
#pragma unroll
  for (int r = 0; r < R; r += 2) {
    const float2 v0 = reinterpret_cast<const float2 *>(anchors)[min(cell0 + r * 32, cells - 1)];
    const float2 v1 = reinterpret_cast<const float2 *>(anchors)[min(cell0 + (r + 1) * 32, cells - 1)];
    ax[r / 2] = make_float2(v0.x, v1.x);
    ay[r / 2] = make_float2(v0.y, v1.y);
  }

  float2 acc[R][kTerms / 2];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int t = 0; t < kTerms / 2; ++t) acc[r][t] = make_float2(0.f, 0.f);

  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(&full_bar[s], 1);
    mbar_fence_init();
  }
  __syncwarp();

  const char *gsrc = reinterpret_cast<const char *>(kp_table) + (size_t)c_begin * (kChunk * kRowFloats * sizeof(float));
  if (lane == 0 && n_local > 0) {
    mbar_arrive_expect_tx(&full_bar[0], kStageBytes);
    bulk_g2s(stage[0], gsrc, kStageBytes, &full_bar[0]);
  }

  for (int lc = 0; lc < n_local; ++lc) {
    const int s = lc & 1;
    // prefetch the next stage into the other buffer (released by the __syncwarp that ended lc-1)
    if (lane == 0 && lc + 1 < n_local) {
      mbar_arrive_expect_tx(&full_bar[s ^ 1], kStageBytes);
      bulk_g2s(stage[s ^ 1], gsrc + (size_t)(lc + 1) * kStageBytes, kStageBytes, &full_bar[s ^ 1]);
    }
    mbar_wait(&full_bar[s], (lc >> 1) & 1);

    const float4 *rows = reinterpret_cast<const float4 *>(stage[s]);
#pragma unroll 2
    for (int i = 0; i < kStageRows; ++i) {
      const float4 *row = rows + i * 7;
      const float4 q = row[6];            // s*kx, s*kx, s*ky, s*ky
      const float2 nqx = make_float2(-q.x, -q.y), nqy = make_float2(-q.z, -q.w);
      float w2[R];
#pragma unroll
      for (int h = 0; h < R / 2; ++h) {
        const float2 dx = __fadd2_rn(ax[h], nqx);
        const float2 dy = __fadd2_rn(ay[h], nqy);
        const float2 d2 = __ffma2_rn(dy, dy, __fmul2_rn(dx, dx));
        w2[2 * h + 0] = fmaxf(ex2_approx(-sqrt_approx(d2.x)), gamma_sq);
        w2[2 * h + 1] = fmaxf(ex2_approx(-sqrt_approx(d2.y)), gamma_sq);
      }
#pragma unroll
      for (int v = 0; v < 6; ++v) {
        const float4 p = row[v];
        const float2 plo = make_float2(p.x, p.y), phi = make_float2(p.z, p.w);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float2 ww = make_float2(w2[r], w2[r]);
          acc[r][2 * v + 0] = __ffma2_rn(ww, plo, acc[r][2 * v + 0]);
          acc[r][2 * v + 1] = __ffma2_rn(ww, phi, acc[r][2 * v + 1]);
        }
      }
    }
    __syncwarp();   // every lane is done with stage s before it is refilled
  }

  // partials[split][t][cell]: consecutive lanes write consecutive cells (coalesced)
  float *dst = partials + (size_t)split * kTerms * cells_padded;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int c = cell0 + r * 32;
    if (c < cells) {
#pragma unroll
      for (int t = 0; t < kTerms / 2; ++t) {
        dst[(size_t)(2 * t + 0) * cells_padded + c] = acc[r][t].x;
        dst[(size_t)(2 * t + 1) * cells_padded + c] = acc[r][t].y;
      }
    }
  }
}

int launch_gram(const float *kp_table, const float *anchors, int batch, int cells, int n_kp_padded, float gamma_sq,
                float *partials, cudaStream_t st) {
  const GramPlan p = make_gram_plan(cells, n_kp_padded, APAP_GRAM_FFMA2);
  const int n_chunks = n_kp_padded / kChunk;
  dim3 grid(p.cell_tiles, p.k_splits, batch);
  if (p.k_splits > 65535 || batch > 65535) return fail(APAP_E_TOOBIG, "gram: grid.y/z exceeds 65535");
  k_gram<<<grid, kGramThreads, 0, st>>>(kp_table, anchors, cells, p.cells_padded, n_chunks, p.chunks_per_split,
                                        p.k_splits, gamma_sq, partials);
  return check_cuda(cudaGetLastError(), "k_gram launch");
}

}  // namespace apap
