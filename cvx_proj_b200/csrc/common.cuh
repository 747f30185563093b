// Shared declarations of libapap_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "apap_b200.h"

namespace apap {

constexpr int kTerms = APAP_GRAM_TERMS;     // 24 distinct Gram sums
constexpr int kRowFloats = APAP_KP_ROW;     // 28 floats = 112 B = 7 x 16 B per keypoint row
constexpr int kChunk = APAP_KP_CHUNK;       // keypoint rows per smem stage
constexpr int kHinvRow = APAP_HINV_ROW;     // 12 floats = 48 B per cell

// Longest FP32 accumulation chain the Gram kernel runs before its sum leaves the register
// (SURVEY.md finding 8: <= 1024 sequential FP32 terms, then a float64 combine, keeps the
// per-cell H inside the 1e-4 gate; a single chain over all N does not).
constexpr int kMaxChainChunks = 8;   // FFMA2 engine: 8 x 128 = 1024 keypoints per split
// The tensor-core engine never runs an FP32 chain longer than a 256-keypoint segment (its splits only exist for
// parallelism), so its splits may be longer: fewer partial planes for K2 to read (c3: 311 -> 156 MB).
constexpr int kMaxSplitChunksTc = 16;   // 16 x 128 = 2048 keypoints per split.  32 (4096) was measured in round 2:
// c3 on one GPU 1.734 -> 1.709 ms (K2 reads half the planes), but an eighth of c3 is then 1.8 waves of CTAs instead of 3.5
// and the 8-GPU shard goes from 0.251 to 0.270 ms -- the plan is a function of N only, so the sharded case decides

struct GramPlan {
  int k_splits;
  int chunks_per_split;
  int cells_per_thread;     // register tile: cells handled by one thread
  int cells_padded;         // row pitch of the partial sums (multiple of 512)
  int cell_tiles;
};

GramPlan make_gram_plan(int cells, int n_kp_padded, int engine);
int sm_count_cached();

// error plumbing (abi.cu)
int fail(int code, const char *msg);
int check_cuda(cudaError_t e, const char *what);

// launchers (one per translation unit)
int launch_gram(const float *kp_table, const float *anchors, int batch, int cells, int n_kp_padded,
                float gamma_sq, float *partials, cudaStream_t st);
int launch_gram_tc(const float *kp_blocks, const float *anchors, int batch, int cells, int n_kp_padded,
                   float gamma_sq, const float *t_bound, float *partials, int *tile_done, cudaStream_t st);
int launch_eig(const float *partials, const double *tmats, int batch, int cells, int k_splits,
               float *out_h, int *out_sweeps, int force_jacobi, int *tile_done, cudaStream_t st);
int launch_weight(const double *anchors, const double *kp_xy, int cells, int n_kp, double inv_sigma_sq,
                  double gamma, double *out, cudaStream_t st);
int launch_warp(const uint8_t *src, int src_h, int src_w, const float *cell_fast, const float *cell_hinv,
                const uint32_t *col_lut, const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x,
                int off_y, int row0, int row1, const uint8_t *centre, int centre_h, int centre_w, uint8_t *out_band,
                size_t out_band_bytes, int flags, int multicast, const void *tiles, cudaStream_t st);
int launch_blend(const uint8_t *a, const uint8_t *b, uint8_t *out, size_t n_px, cudaStream_t st);
int launch_probe(int kind, int iters, float *sink, double *ops, cudaStream_t st);
int launch_weight_bound(const float *src_raw, const int *counts, int batch, int n_points, double scale,
                        const float *anchors, int cells, float *t_bound, cudaStream_t st);
int launch_multicast_copy(const void *src, void *mc_dst, size_t bytes, cudaStream_t st);
int launch_peer_copy(const void *src, void *const *peers, int n_peers, size_t bytes, cudaStream_t st);

// ---- small PTX helpers -----------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// TMA 1-D bulk copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// TMA 1-D bulk copy shared -> global (bulk async-group completion).
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_read() {      // the shared source may be reused / released afterwards
  asm volatile("cp.async.bulk.commit_group;\n\tcp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {     // generic-proxy shared writes -> visible to the async proxy
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float add_rd(float a, float b) { return __fadd_rd(a, b); }

}  // namespace apap
