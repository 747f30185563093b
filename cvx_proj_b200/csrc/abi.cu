// extern "C" entry points of libapap_b200.so (declared in include/apap_b200.h).
#include <stdio.h>
#include <string.h>

#include "common.cuh"
#include "warp_common.cuh"

namespace apap {

static thread_local char g_err[512] = "";

int fail(int code, const char *msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}
int check_cuda(cudaError_t e, const char *what) {
  if (e == cudaSuccess) return 0;
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  return (int)e;
}

static int check_table(const void *kp_table, const void *anchors, int batch, int cells, int n_kp_padded) {
  if (!kp_table || !anchors) return fail(APAP_E_BADARG, "null pointer");
  if (batch <= 0 || cells <= 0 || n_kp_padded <= 0) return fail(APAP_E_BADARG, "batch, cells and n_kp_padded must be > 0");
  if (n_kp_padded % kChunk) return fail(APAP_E_BADARG, "n_kp_padded must be a multiple of APAP_KP_CHUNK");
  if (reinterpret_cast<uintptr_t>(kp_table) & 15u) return fail(APAP_E_ALIGN, "kp_table must be 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(anchors) & 7u) return fail(APAP_E_ALIGN, "anchors must be 8-byte aligned");
  return 0;
}

}  // namespace apap

using namespace apap;

extern "C" {

int apap_abi_version(void) { return APAP_ABI_VERSION; }
const char *apap_last_error(void) { return g_err; }

int apap_device_sm_count(int *sm_count) {
  if (!sm_count) return fail(APAP_E_BADARG, "null pointer");
  int dev = 0, n = 0;
  int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice");
  if (rc) return rc;
  rc = check_cuda(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev), "cudaDeviceGetAttribute");
  if (rc) return rc;
  *sm_count = n;
  return 0;
}

int apap_gram_plan(int cells, int n_kp_padded, int engine, int *k_splits, int *cells_padded,
                   size_t *partial_bytes_per_scene) {
  if (engine != APAP_GRAM_TCGEN05 && engine != APAP_GRAM_FFMA2) return fail(APAP_E_BADARG, "gram_plan: unknown engine");
  if (cells <= 0 || n_kp_padded <= 0 || n_kp_padded % kChunk) return fail(APAP_E_BADARG, "gram_plan: bad sizes");
  // the layout (k_splits, cells_padded) does not depend on the SM count; only the register tile does
  const GramPlan p = make_gram_plan(cells, n_kp_padded, engine);
  if (k_splits) *k_splits = p.k_splits;
  if (cells_padded) *cells_padded = p.cells_padded;
  if (partial_bytes_per_scene) *partial_bytes_per_scene = (size_t)p.k_splits * kTerms * p.cells_padded * sizeof(float);
  return 0;
}

int apap_gram_partials(const float *kp_table, const float *anchors, int batch, int cells, int n_kp_padded,
                       float gamma_sq, int engine, const float *t_bound, float *partials, void *stream) {
  int rc = check_table(kp_table, anchors, batch, cells, n_kp_padded);
  if (rc) return rc;
  if (!partials) return fail(APAP_E_BADARG, "null partials");
  if (engine == APAP_GRAM_TCGEN05)
    return launch_gram_tc(kp_table, anchors, batch, cells, n_kp_padded, gamma_sq, t_bound, partials, nullptr,
                          static_cast<cudaStream_t>(stream));
  if (engine != APAP_GRAM_FFMA2) return fail(APAP_E_BADARG, "gram: unknown engine");
  return launch_gram(kp_table, anchors, batch, cells, n_kp_padded, gamma_sq, partials,
                     static_cast<cudaStream_t>(stream));
}

int apap_eig_denorm(const float *partials, const double *tmats, int batch, int cells, int k_splits, int solver,
                    float *out_h, int *out_sweeps, void *stream) {
  if (!partials || !tmats || !out_h) return fail(APAP_E_BADARG, "null pointer");
  if (batch <= 0 || cells <= 0 || k_splits <= 0) return fail(APAP_E_BADARG, "eig: bad sizes");
  if (solver != APAP_EIG_AUTO && solver != APAP_EIG_JACOBI) return fail(APAP_E_BADARG, "eig: unknown solver");
  return launch_eig(partials, tmats, batch, cells, k_splits, out_h, out_sweeps, solver == APAP_EIG_JACOBI, nullptr,
                    static_cast<cudaStream_t>(stream));
}

int apap_local_homography(const float *kp_table, const float *anchors, const double *tmats, int batch, int cells,
                          int n_kp_padded, float gamma_sq, int engine, int solver, const float *t_bound,
                          float *partials, int *tile_counters, float *out_h, int *out_sweeps, void *stream) {
  if (!tile_counters || engine != APAP_GRAM_TCGEN05) {     // plain sequence: K2 starts when K1 has finished
    int rc = apap_gram_partials(kp_table, anchors, batch, cells, n_kp_padded, gamma_sq, engine, t_bound, partials, stream);
    if (rc) return rc;
    return apap_eig_denorm(partials, tmats, batch, cells, make_gram_plan(cells, n_kp_padded, engine).k_splits, solver,
                           out_h, out_sweeps, stream);
  }
  int rc = check_table(kp_table, anchors, batch, cells, n_kp_padded);
  if (rc) return rc;
  if (!partials || !tmats || !out_h) return fail(APAP_E_BADARG, "null pointer");
  if (solver != APAP_EIG_AUTO && solver != APAP_EIG_JACOBI) return fail(APAP_E_BADARG, "eig: unknown solver");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = launch_gram_tc(kp_table, anchors, batch, cells, n_kp_padded, gamma_sq, t_bound, partials, tile_counters, st);
  if (rc) return rc;
  return launch_eig(partials, tmats, batch, cells, make_gram_plan(cells, n_kp_padded, engine).k_splits, out_h, out_sweeps,
                    solver == APAP_EIG_JACOBI, tile_counters, st);
}

int apap_local_weight(const double *anchors, const double *kp_xy, int cells, int n_kp, double inv_sigma_sq,
                      double gamma, double *out, void *stream) {
  if (!anchors || !kp_xy || !out) return fail(APAP_E_BADARG, "null pointer");
  if (cells < 0 || n_kp < 0) return fail(APAP_E_BADARG, "local_weight: negative size");
  if (reinterpret_cast<uintptr_t>(kp_xy) & 15u) return fail(APAP_E_ALIGN, "local_weight: kp_xy must be 16-byte aligned");
  return launch_weight(anchors, kp_xy, cells, n_kp, inv_sigma_sq, gamma, out, static_cast<cudaStream_t>(stream));
}

int apap_warp(const uint8_t *src, int src_h, int src_w, const float *cell_fast, const float *cell_hinv,
              const uint32_t *col_lut, const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x,
              int off_y, int row0, int row1, const uint8_t *centre, int centre_h, int centre_w, uint8_t *out_band,
              size_t out_band_bytes, int flags, int multicast, const void *tiles, void *stream) {
  if (!src || !cell_fast || !cell_hinv || !col_lut || !out_band) return fail(APAP_E_BADARG, "null pointer");
  if (flags & ~(APAP_WARP_FORCE_EXACT | APAP_WARP_LEGACY)) return fail(APAP_E_BADARG, "warp: unknown flag");
  if (n_blocks < 0 || (n_blocks > 0 && !row_blocks)) return fail(APAP_E_BADARG, "warp: bad row blocks");
  if (src_h <= 0 || src_w <= 0 || canvas_w <= 0 || grid_cols <= 0) return fail(APAP_E_BADARG, "warp: sizes must be > 0");
  if (centre && (centre_h <= 0 || centre_w <= 0)) return fail(APAP_E_BADARG, "warp: bad centre image size");
  if (row0 < 0 || row1 < row0) return fail(APAP_E_BADARG, "warp: bad row band");
  if (out_band_bytes < (size_t)(row1 - row0) * (size_t)canvas_w * 3)
    return fail(APAP_E_BADARG, "warp: out_band is smaller than the rows [row0, row1) of the canvas");
  return launch_warp(src, src_h, src_w, cell_fast, cell_hinv, col_lut, row_blocks, n_blocks, grid_cols, canvas_w, off_x,
                     off_y, row0, row1, centre, centre_h, centre_w, out_band, out_band_bytes, flags, multicast, tiles,
                     static_cast<cudaStream_t>(stream));
}

int apap_warp_bilinear(const uint8_t *src, int src_h, int src_w, const float *cell_hinv, const uint32_t *col_lut,
                       const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x, int off_y, int row0,
                       int row1, uint8_t *out_band, size_t out_band_bytes, void *stream) {
  if (!src || !cell_hinv || !col_lut || !out_band || (n_blocks > 0 && !row_blocks)) return fail(APAP_E_BADARG, "null pointer");
  if (n_blocks < 0 || src_h <= 0 || src_w <= 0 || canvas_w <= 0 || grid_cols <= 0 || row0 < 0 || row1 < row0)
    return fail(APAP_E_BADARG, "bilinear warp: bad sizes");
  if ((long long)src_w * src_h > 2147483647LL) return fail(APAP_E_TOOBIG, "bilinear warp: source image too large");
  if (out_band_bytes < (size_t)(row1 - row0) * (size_t)canvas_w * 3)
    return fail(APAP_E_BADARG, "bilinear warp: out_band is smaller than the rows [row0, row1) of the canvas");
  if ((reinterpret_cast<uintptr_t>(col_lut) & 7u) || (reinterpret_cast<uintptr_t>(row_blocks) & 7u))
    return fail(APAP_E_ALIGN, "bilinear warp: col_lut / row_blocks must be 8-byte aligned");
  WarpParams p;
  memset(&p, 0, sizeof(p));
  p.src = src; p.src_h = src_h; p.src_w = src_w; p.cell_hinv = cell_hinv;
  p.col_lut = reinterpret_cast<const uint2 *>(col_lut); p.row_blocks = reinterpret_cast<const uint2 *>(row_blocks);
  p.n_blocks = n_blocks; p.grid_cols = grid_cols; p.canvas_w = canvas_w; p.off_x = off_x; p.off_y = off_y;
  p.row0 = row0; p.band_rows = row1 - row0; p.out = out_band;
  return launch_warp_bilinear(p, static_cast<cudaStream_t>(stream));
}

int apap_warp_tiles_bytes(int canvas_w, int n_blocks, size_t *bytes) {
  if (!bytes || canvas_w <= 0 || n_blocks < 0) return fail(APAP_E_BADARG, "warp_tiles_bytes: bad arguments");
  *bytes = warp_tiles_bytes(canvas_w, n_blocks);
  return 0;
}

int apap_warp_tiles(const float *cell_fast, const float *cell_hinv, const uint32_t *col_lut, const int *col_extent,
                    const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x, int off_y, int src_h,
                    int src_w, void *tiles, size_t tiles_bytes, void *stream) {
  if (!cell_fast || !cell_hinv || !col_lut || !col_extent || (n_blocks > 0 && !row_blocks))
    return fail(APAP_E_BADARG, "warp_tiles: null pointer");
  if (n_blocks < 0 || grid_cols <= 0 || canvas_w <= 0 || src_h <= 0 || src_w <= 0) return fail(APAP_E_BADARG, "warp_tiles: bad sizes");
  if ((reinterpret_cast<uintptr_t>(cell_fast) & 15u) || (reinterpret_cast<uintptr_t>(col_lut) & 7u) ||
      (reinterpret_cast<uintptr_t>(row_blocks) & 7u) || (reinterpret_cast<uintptr_t>(col_extent) & 7u))
    return fail(APAP_E_ALIGN, "warp_tiles: cell_fast must be 16-byte, col_lut / row_blocks / col_extent 8-byte aligned");
  WarpParams p;
  memset(&p, 0, sizeof(p));
  p.cell_fast = reinterpret_cast<const float4 *>(cell_fast); p.cell_hinv = cell_hinv;
  p.col_lut = reinterpret_cast<const uint2 *>(col_lut); p.row_blocks = reinterpret_cast<const uint2 *>(row_blocks);
  p.n_blocks = n_blocks; p.grid_cols = grid_cols; p.canvas_w = canvas_w; p.off_x = off_x; p.off_y = off_y;
  p.src_h = src_h; p.src_w = src_w;
  return launch_warp_tiles(p, col_extent, tiles, tiles_bytes, static_cast<cudaStream_t>(stream));
}

int apap_blend(const uint8_t *a, const uint8_t *b, uint8_t *out, size_t n_px, void *stream) {
  if (!a || !b || !out) return fail(APAP_E_BADARG, "null pointer");
  return launch_blend(a, b, out, n_px, static_cast<cudaStream_t>(stream));
}

int apap_multicast_copy(const void *src, void *multicast_dst, size_t bytes, void *stream) {
  if (!src || !multicast_dst) return fail(APAP_E_BADARG, "multicast_copy: null pointer");
  if ((bytes & 15u) || (reinterpret_cast<uintptr_t>(src) & 15u) || (reinterpret_cast<uintptr_t>(multicast_dst) & 15u))
    return fail(APAP_E_ALIGN, "multicast_copy: size and both addresses must be multiples of 16 bytes");
  return launch_multicast_copy(src, multicast_dst, bytes, static_cast<cudaStream_t>(stream));
}

int apap_peer_copy(const void *src, void *const *peer_dsts, int n_peers, size_t bytes, void *stream) {
  if (!src || (!peer_dsts && n_peers)) return fail(APAP_E_BADARG, "peer_copy: null pointer");
  if (n_peers < 0 || n_peers > APAP_MAX_PEERS) return fail(APAP_E_BADARG, "peer_copy: 0 <= n_peers <= APAP_MAX_PEERS");
  if ((bytes & 15u) || (reinterpret_cast<uintptr_t>(src) & 15u)) return fail(APAP_E_ALIGN, "peer_copy: size and addresses must be multiples of 16 bytes");
  for (int k = 0; k < n_peers; ++k)
    if (!peer_dsts[k] || (reinterpret_cast<uintptr_t>(peer_dsts[k]) & 15u))
      return fail(APAP_E_ALIGN, "peer_copy: peer addresses must be non-null multiples of 16 bytes");
  return launch_peer_copy(src, peer_dsts, n_peers, bytes, static_cast<cudaStream_t>(stream));
}

int apap_pipe_probe(int kind, int iters, float *sink, double *ops, void *stream) {
  if (!sink || iters <= 0) return fail(APAP_E_BADARG, "probe: bad arguments");
  return launch_probe(kind, iters, sink, ops, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
