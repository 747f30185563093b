/*
 * apap_b200.h -- C ABI of libapap_b200.so: the APAP (moving-DLT + mesh warp) hot path of
 * Enigmatisms/cvx_proj as hand-written sm_100a CUDA kernels.
 *
 * The reference has no FFI today: the path is plain Python (pyviz/apap.py, pyviz/apap_utils.py).
 * Each entry point below names the reference code it replaces.  The Python host layer
 * (cvx_proj_b200/apap.py, apap_utils.py) binds these with ctypes and keeps the reference's
 * own call surface; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer owned by the caller (no hidden allocation, no
 *     hidden host<->device copy); `stream` is a cudaStream_t passed as void*; calls are
 *     asynchronous on that stream;
 *   - return value 0 = ok; > 0 = a cudaError_t; < 0 = an APAP_E_* argument error;
 *     apap_last_error() gives a thread-local message for the last non-zero return;
 *   - a "cell" is one mesh cell of the APAP grid (row-major, row = y cell, col = x cell), a
 *     "keypoint" one matched pair, a "canvas" the stitched output image (HxWx3 uint8,
 *     OpenCV BGR order, rows packed, 3 bytes per pixel).
 */
#ifndef APAP_B200_H
#define APAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APAP_ABI_VERSION 23

/* Layout constants shared with the host layer. */
#define APAP_GRAM_TERMS 24   /* distinct non-zero sums of the 9x9 Gram matrix (4 sym. 3x3 blocks) */
#define APAP_KP_ROW     28   /* floats per keypoint row: 24 product terms, s*kx (x2), s*ky (x2)   */
#define APAP_KP_CHUNK   128  /* keypoint tables are padded to a multiple of this many keypoints   */
#define APAP_KP_BLOCK   8    /* keypoints per block of the tensor-core table (K of one TF32 MMA)  */
#define APAP_KP_BLOCK_FLOATS 528 /* floats per block: [Ph | Pl] tile 512, s*kx[8], s*ky[8]           */
#define APAP_HINV_ROW   12   /* floats per cell of the warp's fast-path record (see apap_warp)    */
#define APAP_WARP_BLOCK_ROWS 4 /* most canvas rows per row block of the warp kernel               */

#define APAP_E_BADARG   (-1)
#define APAP_E_ALIGN    (-2)
#define APAP_E_TOOBIG   (-3)

int apap_abi_version(void);
const char *apap_last_error(void);

/* Number of SMs of the current device (grid sizing, reporting). */
int apap_device_sm_count(int *sm_count);

/*
 * Plan the moving-DLT contraction: how many keypoint splits the Gram kernel of `engine` uses for
 * n_kp_padded keypoints (a function of the keypoint count and the engine only, so a grid computed in
 * row shards equals the unsharded grid bit for bit) and how many bytes of partial sums it needs per scene.
 *   partial layout: float [k_splits][APAP_GRAM_TERMS][cells_padded]   (term-major, coalesced)
 *   engine FFMA2: a split is at most 1024 keypoints, the longest FP32 chain the kernel runs before the
 *   float64 combine of K2; engine TCGEN05 (chains of 256 keypoints whatever the split): at most 2048.
 */
#define APAP_GRAM_TCGEN05 0
#define APAP_GRAM_FFMA2   1
int apap_gram_plan(int cells, int n_kp_padded, int engine, int *k_splits, int *cells_padded,
                   size_t *partial_bytes_per_scene);

/*
 * K1 -- weights + Gram contraction.  Replaces, for every cell, pyviz/apap.py:150-152 (the
 * weight w_i = max(exp(-|v - x_i| / sigma^2), gamma)) and the row scaling + SVD input build of
 * pyviz/apap.py:159: it accumulates S_t(cell) = sum_i w_i^2 * P[i][t] for the 24 product terms.
 * Coordinates arrive pre-scaled by s = 2 log2(e) / sigma^2, so w_i^2 = max(2^-|s v - s x_i|, gamma^2).
 *   engine   : APAP_GRAM_TCGEN05 -- 3xTF32 tcgen05.mma, weights generated into tensor memory;
 *              APAP_GRAM_FFMA2   -- FP32 SIMT (packed FFMA2)
 *   kp_table : engine FFMA2:   float [batch][n_kp_padded][APAP_KP_ROW]: 24 product terms, then
 *              s*kx, s*kx, s*ky, s*ky (the keypoint, each coordinate twice);
 *              engine TCGEN05: float [batch][n_kp_padded / 8][APAP_KP_BLOCK_FLOATS]: per block of 8
 *              keypoints the 8 x 64 tile [Ph | Pl] -- TF32 head and tail (P = Ph + Pl) of the 8 x 32
 *              (24 terms + 8 zero columns) product matrix -- in the K-major core-matrix layout of the
 *              MMA: element (keypoint k, column m) at float (k/4)*256 + (m/8)*32 + (m%8)*4 + k%4, m = n
 *              for Ph, 32 + n for Pl; then s*kx[8], s*ky[8];
 *              rows / blocks past the real keypoints are zero
 *   anchors  : float [batch][cells][2] = s * (x, y) of the cell anchor points (get_vertice)
 *   partials : float [batch][k_splits][24][cells_padded]  (same layout for both engines)
 *   gamma_sq = gamma^2
 *   t_bound  : optional float [batch] from apap_weight_bound (device memory): an upper bound of |s v - s x| over
 *              the scene's (anchor, keypoint) pairs.  Engine TCGEN05 drops the clamp max(w, gamma^2) of
 *              pyviz/apap.py:152 for a scene whose bound shows no weight can reach it (1.001 t + 0.001 <
 *              -log2 gamma^2; the reference's gamma = 0.5, sigma = 100 on a 4K canvas is such a scene): the same
 *              bits, 16 of ~180 instructions per 16 keypoints less.  NULL = always clamp.
 */
int apap_gram_partials(const float *kp_table, const float *anchors, int batch, int cells,
                       int n_kp_padded, float gamma_sq, int engine, const float *t_bound, float *partials,
                       void *stream);

/*
 * K2 -- per-cell 9x9 symmetric eigensolve + de-normalisation.  Replaces cv.SVDecomp + V[-1]
 * (pyviz/apap.py:160-161) and pyviz/apap.py:164-168: sums the k_splits partials (apap_gram_plan) in float64,
 * expands the 24 sums to the 9x9 Gram matrix, finds the eigenvector h of its smallest eigenvalue
 * and stores float32 H = T2inv * reshape(h,3,3) * T1, divided by H[2][2].
 *   solver : APAP_EIG_AUTO = float64 LDL^T inverse iteration, cyclic Jacobi for the cells whose
 *            iteration does not settle (tiny spectral gap); APAP_EIG_JACOBI = Jacobi for every cell
 *   tmats  : double [batch][18] = T2inv (row-major 3x3) then T1, T2inv = inv(N2) inv(C2), T1 = C1 N1
 *   out_h  : float [batch][cells][9]
 *   out_sweeps : optional int32 [batch][cells]: > 0 Jacobi sweeps used, < 0 minus the number of
 *            inverse-iteration steps (NULL to skip)
 * Planes scaled by a power of two give the same bits (K2 divides by sum(w^2) first).  A cell whose 24 sums are all
 * zero (no weight at all) has the Gram matrix 0 / 0: it reports 0 Jacobi sweeps and stores T2inv e0 T1 divided by
 * its [2][2] entry -- 0 for tmats whose last rows are [0 0 1] -- i.e. NaN where T2inv[:][0] T1[0][:] is 0, +-inf
 * elsewhere.
 */
#define APAP_EIG_AUTO   0
#define APAP_EIG_JACOBI 1
int apap_eig_denorm(const float *partials, const double *tmats, int batch, int cells,
                    int k_splits, int solver, float *out_h, int *out_sweeps, void *stream);

/*
 * K1 + K2 on `stream` (what APAP.local_homography calls).
 *   tile_counters : optional int32 [batch][ceil(cells / 128)] scratch, ALL ZERO on entry and all zero again when the
 *                   call has completed.  When given (engine TCGEN05), K2 is launched as a programmatic dependent of
 *                   K1: K1 counts the finished keypoint splits of every 128-cell tile there and K2's CTAs start on
 *                   finished tiles while K1's last CTAs are still running, instead of after the whole grid.
 *                   NULL = K2 starts when K1 has finished.
 */
int apap_local_homography(const float *kp_table, const float *anchors, const double *tmats,
                          int batch, int cells, int n_kp_padded, float gamma_sq, int engine, int solver,
                          const float *t_bound, float *partials, int *tile_counters, float *out_h, int *out_sweeps,
                          void *stream);

/*
 * The whole of APAP.local_homography (pyviz/apap.py:121-169) in ONE call, from the raw inputs as the caller has them:
 * anchors = float32(vertices * scale), apap_condition, apap_kp_rows, apap_weight_bound, apap_kp_blocks (engine TCGEN05),
 * then apap_local_homography -- the same kernels in the same order as the separate entry points (same bits), without a
 * host round trip between them.  What the Python class calls.
 *   src, dst  : float [batch][n_points][2] raw matched points;  counts : int32 [batch] or NULL
 *   vertices  : double [batch][cells][2] = get_vertice's anchor points, unscaled;  scale = s = 2 log2(e) / sigma^2
 *   workspace : device scratch, 256-byte aligned, >= apap_pass_workspace_bytes(batch, n_points, cells, engine)
 *   tile_counters, out_h, out_sweeps : as in apap_local_homography
 */
int apap_pass_workspace_bytes(int batch, int n_points, int cells, int engine, size_t *bytes);
int apap_local_homography_points(const float *src, const float *dst, const int *counts, int batch, int n_points,
                                 const double *vertices, int cells, double scale, float gamma_sq, int engine, int solver,
                                 void *workspace, size_t workspace_bytes, int *tile_counters, float *out_h,
                                 int *out_sweeps, void *stream);

/*
 * Second output of APAP.local_homography (pyviz/apap.py:144,153): float64 weights
 *   out[c][i] = max(exp(-|anchor_c - kp_i| / sigma^2), gamma),  c in [0, cells), i in [0, n_kp)
 *   anchors : double [cells][2];  kp_xy : double [n_kp][2] (16-byte aligned; float32 keypoints promoted by the caller,
 *   which is what numpy does in `vertices[i, j] - src_point`, so float64 keypoints keep their bits too)
 */
int apap_local_weight(const double *anchors, const double *kp_xy, int cells, int n_kp,
                      double inv_sigma_sq, double gamma, double *out, void *stream);

/*
 * K3 -- mesh warp.  Replaces the pixel loop of APAP.local_warp (pyviz/apap.py:206-215): for the
 * canvas rows covered by `row_blocks` looks the cell up (col_lut / row_blocks restate
 * np.where(k < edges) of :207,:209), applies that cell's H^-1 to (j - off_x, i - off_y, 1), divides,
 * and copies src[int(ty)][int(tx)] when 0 < tx < src_w and 0 < ty < src_h (else leaves 0).  Pixel
 * selection is bit-identical to the reference's float64 arithmetic: a float32 fast path on
 * cell-relative coefficients (cell_fast) decides every pixel whose coordinates are farther than the
 * cell's guard band eps from an integer, the rest are recomputed in float64 from cell_hinv.
 *   cell_fast : float [grid_rows*grid_cols][APAP_HINV_ROW] = A0 B0 C0 A1 B1 C1 A2 B2 C2,
 *               int32 bits of (qbx - 0x4B400000), (qby - 0x4B400000), g; with dx, dy the pixel's
 *               offset inside its cell:  src_x = qbx + floor((A0 dx + B0 dy + C0) / (A2 dx + B2 dy + C2));
 *               g = 0.5 - eps (eps = the cell's guard band), g < 0 = the whole cell takes the float64
 *               path, g > 1 = the whole cell maps outside the source image and is left black
 *   cell_hinv : float [grid_rows*grid_cols][9], the inverted grid of pyviz/apap.py:201-203
 *   col_lut   : uint32 [canvas_w][2] = {cell column, float32 bits of dx}
 *   row_blocks: uint32 [n_blocks][2] = {first canvas row | rows << 28 (rows = 1..APAP_WARP_BLOCK_ROWS),
 *               cell row | dy of the first row << 16}, in canvas order and contiguous (block k+1 starts at or
 *               before the row after block k's last); a block never crosses a cell row; the blocks passed are
 *               the rows that get written (a row band of a sharded run = its blocks); canvas rows < 2^28, cell
 *               rows and dy < 2^16
 *   row0, row1: out_band holds the canvas rows [row0, row1); every row block lies inside
 *   out_band  : uint8 [row1 - row0][canvas_w][3], out_band_bytes >= that and < 2 GiB
 *   centre    : optional uint8 [centre_h][centre_w][3] pasted at (off_x, off_y) and blended with
 *               the warped pixel by the uniform_blend rule (fused K3+K4, pyviz/apap.py:259-261);
 *               NULL = plain warp
 *   flags     : APAP_WARP_FORCE_EXACT = every pixel takes the float64 path (validation switch);
 *               APAP_WARP_LEGACY = the strip kernel even when `tiles` is given
 *   tiles     : the band's tile records from apap_warp_tiles (same tables, same band), or NULL.  With tiles, no centre
 *               and a source whose rows are 16-byte aligned (src % 16 == 0, src_w * 3 % 16 == 0), the TILE ENGINE runs
 *               (csrc/warp_tile.cu): persistent warp-specialised CTAs; per 128 x 32 canvas tile the source box the
 *               tile can pick from is staged in shared memory by one tensor-map TMA copy (zero outside the image),
 *               gathers are LDS, the output leaves as 16-row tensor-map TMA stores when the band is 16-byte aligned
 *               and canvas_w % 16 == 0.  Otherwise the STRIP KERNEL of round 1 runs (one warp per 32 columns,
 *               gathers from global memory, shuffle re-pack).  Same bytes either way.
 *   multicast   : non-zero = out_band is an NVLS multicast address (one mapping of the same panorama buffer on every
 *                 GPU of the group, e.g. torch symmetric memory's multicast_ptr + band offset): the kernel stores with
 *                 multimem.st, so the NVSwitch writes this rank's row band into every GPU's panorama -- the panorama
 *                 is assembled by the warp itself, no all-gather.  Stores are 16 bytes wide, whole 384-byte tile rows
 *                 (tile engine): needs canvas_w % 16 == 0 and a 16-byte aligned band; the caller synchronises the
 *                 group afterwards.
 */
#define APAP_WARP_FORCE_EXACT 1
#define APAP_WARP_LEGACY      2
int apap_warp(const uint8_t *src, int src_h, int src_w, const float *cell_fast, const float *cell_hinv,
              const uint32_t *col_lut, const uint32_t *row_blocks, int n_blocks,
              int grid_cols, int canvas_w, int off_x, int off_y, int row0, int row1,
              const uint8_t *centre, int centre_h, int centre_w,
              uint8_t *out_band, size_t out_band_bytes, int flags, int multicast,
              const void *tiles, void *stream);

/*
 * The tile engine's per-tile records for a band: for every 128-column x 8-row-block tile of the canvas, the source
 * box its pixels can pick from (the corners of every cell x tile rectangle mapped through the cell's H^-1), the
 * tensor-map box shape, its rows grouped by cell row, and whether it is all black.  They depend on the tables and
 * the geometry only -- not on the images -- so they are built once per inverted grid and band (with
 * apap_warp_tables) and reused by every apap_warp call on it.
 *   col_extent : int32 [grid_cols][2] = {first, last} canvas column of the cell column (as for apap_warp_tables)
 *   tiles      : out, 16-byte aligned, apap_warp_tiles_bytes(canvas_w, n_blocks) bytes (192 per tile)
 */
int apap_warp_tiles_bytes(int canvas_w, int n_blocks, size_t *bytes);
int apap_warp_tiles(const float *cell_fast, const float *cell_hinv, const uint32_t *col_lut, const int *col_extent,
                    const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x, int off_y,
                    int src_h, int src_w, void *tiles, size_t tiles_bytes, void *stream);

/*
 * Opt-in bilinear mode of the mesh warp (no reference counterpart: APAP.local_warp truncates, pyviz/apap.py:214-215;
 * BASELINE.json's north_star asks for a bilinear sample within +-1 LSB of a float64 restatement).  Same cell lookup,
 * float64 coordinates and strict bounds test as the pixel loop of pyviz/apap.py:206-215 decide which pixels are
 * written; the value is the bilinear sample at (tx, ty) with cv.warpPerspective's convention (pyviz/utils.py:114):
 * x0 = floor(tx), fx = tx - x0, taps clamped to the image, rounded half up.  Tables as for apap_warp.
 */
int apap_warp_bilinear(const uint8_t *src, int src_h, int src_w, const float *cell_hinv, const uint32_t *col_lut,
                       const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x, int off_y,
                       int row0, int row1, uint8_t *out_band, size_t out_band_bytes, void *stream);

/*
 * K4 -- uniform_blend (pyviz/apap_utils.py:75-88): out = both non-black ? (a + b) >> 1 : a + b,
 * per pixel of n_px 3-byte pixels.  All three pointers 16-byte aligned.
 */
int apap_blend(const uint8_t *a, const uint8_t *b, uint8_t *out, size_t n_px, void *stream);

/*
 * Panorama blend of placed layers (driver.stitch_panorama): out [canvas_h][canvas_w][3] uint8 (device, any alignment,
 * out_bytes >= canvas_h x canvas_w x 3) gets, per pixel, the per-channel floor((sum of the layers' pixels) / n), n =
 * the number of layers whose pixel there is non-empty (any channel > 0), and 0 where n = 0.  With two equal layers at
 * one origin this is apap_blend bit for bit; the result does not depend on the layer order.
 *   layers   : HOST long long [n_layers][6] = {device address, h, w, row pitch in bytes, x0, y0}: an [h][w][3] uint8
 *              image whose pixel (0, 0) lies at canvas (x0, y0).  Any address and any pitch >= 3 w (ignored for
 *              h = 1), so crops of a larger image need no copy; origins may be negative and layers may stick out of
 *              the canvas (clipped).  Sizes in [1, 2^30], origins in [-2^30, 2^30].
 *   n_layers : 1 .. APAP_BLEND_MAX_LAYERS (255 x 256 fits the kernel's 16-bit sums)
 * One kernel (k_blend_layers), one pass over the canvas; every layer byte inside the canvas is read once.
 */
#define APAP_BLEND_MAX_LAYERS 256
int apap_blend_layers(const long long *layers, int n_layers, int canvas_h, int canvas_w, uint8_t *out,
                      size_t out_bytes, void *stream);

/*
 * Feather blend of placed layers (utils.feather_blend, driver.stitch_panorama(blend="feather")): out [canvas_h]
 * [canvas_w][3] uint8 (device, any alignment, out_bytes >= canvas_h x canvas_w x 3) is bit for bit what
 * cv.detail.FeatherBlender(sharpness) gives after prepare((0, 0, canvas_w, canvas_h)), feed(P_k as int16, mask_k,
 * (0, 0)) for every layer in order and blend(), converted to uint8.  P_k is layer k pasted into a zero canvas
 * (clipped), mask_k its non-empty pixels (any channel > 0).  Per pixel and layer w = min(fl(D s), 1), D = the L1
 * distance to the nearest empty pixel of P_k (the canvas border is not empty); acc += trunc(v w) per channel, wsum +=
 * w in layer order; out = trunc(acc / (wsum + 1e-5)), 0 where wsum <= 1e-5.  Where one layer alone has weight 1 the
 * result is v - 1 (v >= 1), as OpenCV's.
 *   layers    : HOST long long [n_layers][6], as apap_blend_layers
 *   n_layers  : 1 .. APAP_FEATHER_MAX_LAYERS (OpenCV's int16 accumulator holds 128 x 255)
 *   sharpness : finite, >= FLT_MIN (a normal float), and apap_feather_distance_cap accepts it with this canvas
 *   workspace : device scratch of apap_feather_workspace_bytes (2 bytes per layer pixel inside the canvas), 16-byte
 *               aligned
 * Three kernels (k_feather_rows, k_feather_cols, k_feather_blend) on `stream`.
 * apap_feather_distance_cap: the distance the kernels store in place of larger ones (host only) -- the smallest
 * integer d with fl(d s) >= 1, or canvas_h + canvas_w - 1 when that is smaller; APAP_E_TOOBIG when the cap exceeds
 * 65535 (s below about 1.5e-5 on a canvas with canvas_h + canvas_w > 65536); APAP_E_BADARG for a sharpness that is
 * not finite or below FLT_MIN.
 */
#define APAP_FEATHER_MAX_LAYERS 128
int apap_feather_distance_cap(float sharpness, int canvas_h, int canvas_w, int *cap);
int apap_feather_workspace_bytes(const long long *layers, int n_layers, int canvas_h, int canvas_w, size_t *bytes);
int apap_feather_blend(const long long *layers, int n_layers, int canvas_h, int canvas_w, float sharpness,
                       void *workspace, size_t workspace_bytes, uint8_t *out, size_t out_bytes, void *stream);

/*
 * Input preparation on the device (what the host layer used to build in numpy; both reproduce their
 * numpy restatements in cvx_proj_b200/apap.py bit for bit).
 *
 * apap_kp_rows: the keypoint row table (layout under apap_gram_partials) from the conditioned keypoint pairs --
 * the Gram terms of the two DLT rows pyviz/apap.py:106-118 builds per match, float64 products rounded once.
 *   src_cond, dst_cond : float [batch][n_points][2], the conditioned source / target points (pyviz/apap.py:136-141)
 *   src_raw            : float [batch][n_points][2], the raw source points the weights are measured from (:150)
 *   counts             : int32 [batch] matches per scene (rows past it are zero), or NULL = n_points everywhere
 *   scale              : 2 log2(e) / sigma^2;  kp_table : float [batch][n_kp_padded][APAP_KP_ROW] (out)
 *
 * apap_kp_blocks: the keypoint row table of engine FFMA2 -> the block table of engine TCGEN05 (layouts under
 * apap_gram_partials; the TF32 split of the product terms pyviz/apap.py:106-118 feeds the tensor cores).
 *   kp_table : float [batch][n_kp_padded][APAP_KP_ROW];  kp_blocks : float [batch][n_kp_padded / 8][APAP_KP_BLOCK_FLOATS]
 *
 * apap_warp_tables: the fast-path records `cell_fast` of apap_warp from the inverted grid (the per-pixel
 * arithmetic of pyviz/apap.py:211-215 rewritten per cell, with its error bound).
 *   cell_hinv  : float [grid_rows*grid_cols][9], the inverted grid of pyviz/apap.py:201-203
 *   col_extent : int32 [grid_cols][2] = {first, last} canvas column mapped to the cell column by the
 *                reference's lookup (pyviz/apap.py:209), first > last = no canvas column; row_extent alike
 *   cell_fast  : float [grid_rows*grid_cols][APAP_HINV_ROW] (out)
 */
/*
 * apap_invert_grid: the per-cell inverse of APAP.local_warp, pyviz/apap.py:201-203 (np.linalg.inv of every float32
 * 3x3 cell = LAPACK dgesv on the float64 promotion, rounded once).  grid_inv gets the float64 partial-pivoting inverse
 * rounded to float32; flags[c] = 0 where that is PROVABLY the float32 numpy returns (every entry farther from a
 * float32 rounding boundary than twice the forward-error bound of the solve, no pivot ties, no zero / tiny / huge /
 * non-finite entries), 1 where the caller must invert the cell with numpy / LAPACK itself (singular cells included).
 *   grid, grid_inv : float [cells][9] (device);  flags : uint8 [cells] (device)
 */
int apap_invert_grid(const float *grid, int cells, float *grid_inv, unsigned char *flags, void *stream);

/*
 * apap_condition: the O(N) prologue of APAP.local_homography on the device (pyviz/apap.py:129-141): Hartley
 * normalisers (getNormalize2DPts, :35-59), conditioners (getConditionerFromPts, :63-89), conditioned points
 * (point_normalize, :92-100) and the two de-normalisation matrices of :165-166, for `batch` scenes.  Reductions run
 * in float64 in a fixed order; the matrices are rounded to float32 and the per-point arithmetic is float32, as in the
 * reference.  (The Python class keeps the reference's static methods on the host, bit-exact; this entry point is what
 * its local_homography uses, the results agree to ~1e-6 of the per-cell gate.)
 *   src, dst : float [batch][n_points][2] raw matched points;  counts : int32 [batch] or NULL
 *   cond     : out float [2][batch][n_points][2]: conditioned source points, conditioned target points
 *              (= src_cond / dst_cond of apap_kp_rows); points past a scene's count are zero
 *   mats     : out float [batch][2][2][9]: per scene {N1, C1, N2, C2} (normaliser and conditioner per set)
 *   tmats    : out double [batch][18] = T2inv then T1 (the `tmats` of apap_eig_denorm)
 */
int apap_condition(const float *src, const float *dst, const int *counts, int batch, int n_points, float *cond,
                   float *mats, double *tmats, void *stream);

/*
 * apap_weight_bound: t_bound[scene] = an upper bound of |s v - s x| over the scene's cell anchors v and matched source
 * points x (the distance of pyviz/apap.py:150-151 in the pre-scaled units of K1): the diagonal of the two sets' joint
 * bounding box, rounded up; +inf for a scene without points or with non-finite coordinates.  The `t_bound` of
 * apap_gram_partials / apap_local_homography.
 *   src_raw : float [batch][n_points][2] raw source points;  counts : int32 [batch] or NULL;  scale = s
 *   anchors : float [batch][cells][2] = s * anchor (the `anchors` of K1);  t_bound : out float [batch]
 */
int apap_weight_bound(const float *src_raw, const int *counts, int batch, int n_points, double scale,
                      const float *anchors, int cells, float *t_bound, void *stream);

int apap_kp_rows(const float *src_cond, const float *dst_cond, const float *src_raw, const int *counts, int batch,
                 int n_points, int n_kp_padded, double scale, float *kp_table, void *stream);
int apap_kp_blocks(const float *kp_table, int batch, int n_kp_padded, float *kp_blocks, void *stream);
int apap_warp_tables(const float *cell_hinv, const int *col_extent, const int *row_extent, int grid_rows,
                     int grid_cols, int off_x, int off_y, int src_w, int src_h, float *cell_fast, void *stream);

/*
 * Global-homography warp of the reference's README pipeline (SURVEY.md 8f row N4): `image_warping`,
 * pyviz/utils.py:93-127 = cv.warpPerspective(img2warp, Ht.H, canvas) (bilinear, constant border 0) followed by the
 * base image pasted over the canvas (:124-125) or the mean-blend loop (:115-123).  Bit-exact with OpenCV's 8-bit
 * fixed-point bilinear warp (coordinates in 1/32 pixel, 15-bit weights).
 *   inverse_map : double [9] HOST memory, row-major: canvas (x, y, 1) -> source pixel, i.e. cv::invert(Ht.H)
 *   dst         : uint8 [dst_h][dst_w][3] canvas (device), every pixel written
 *   base        : optional uint8 [base_h][base_w][3] (device) placed at (off_x, off_y) on the canvas
 *   mode        : 0 warp only; 1 paste the base over the warp (direct_blend=True); 2 mean blend: inside the base
 *                 rectangle (warp + base) >> 1 where any channel of the warp is non-zero, else the base pixel
 */
int apap_warp_perspective(const uint8_t *src, int src_h, int src_w, const double *inverse_map, uint8_t *dst,
                          int dst_h, int dst_w, const uint8_t *base, int base_h, int base_w, int off_x, int off_y,
                          int mode, void *stream);

/*
 * Spectral match weighting of the reference's README pipeline (SURVEY.md 8f row N4): calculate_M,
 * pyviz/spectral_method.py:96-125.
 * apap_affinity_matrix: M [n][n] float64 (device): M[i][i] = diag[i] (match score + epipolar term, :104-111, computed
 *   by the caller), M[i][j] = max(4.5 - ((|s_i - s_j|^2 - |d_i - d_j|^2)^2) * rcp_value, 0) in numpy's float32
 *   arithmetic (:112-118); src_pts / dst_pts: float [n][2] (device), rcp_value = 1 / (2 affinity_eps^2).
 * apap_power_iterate: `steps` steps of the power iteration that replaces np.linalg.svd(M) + |U[:, 0]| (:122-123),
 *   y_{k+1} = M (y_k / |y_k|), one kernel per step, then x = y / |y| of the last iterate and *max_diff_bits = the bits of
 *   max_i |x[i] - x_before[i]| (x_before = the normalised iterate one step earlier) for the caller's convergence test.
 *   y: double [2][n] ping-pong, iterate k lives in y[k & 1]; norms: double [3] ring, |y_k|^2 in norms[k % 3].  Before
 *   the first call (first_step = 0) the caller stores a positive start vector in y[0], its squared norm in norms[0]
 *   and zero in norms[1]; later calls pass first_step = the number of steps already done.
 */
int apap_affinity_matrix(const float *src_pts, const float *dst_pts, const double *diag, int n, float rcp_value,
                         double *m, void *stream);
int apap_power_iterate(const double *m, int n, double *y, double *norms, int first_step, int steps, double *x,
                       unsigned long long *max_diff_bits, void *stream);

/*
 * Exact 1-nearest-neighbour descriptor matching: the matcher step of the reference's keypoint-pair producer,
 * cv.FlannBasedMatcher().match(feats_cp, feats_op) (pyviz/utils.py:149-150; SURVEY 8f row N3).  FLANN is approximate
 * and not reproducible, so the contract is cv.BFMatcher(cv.NORM_L2).match on the same descriptors: per query the train
 * index with the smallest sum_k (q_k - t_k)^2 (float32; the lowest index on a tie) and distance = sqrt of that sum --
 * bit-identical to OpenCV for integer-valued descriptors (SIFT: 0..255), equal up to float32 near-ties otherwise.
 *   query : float [nq][dim], train : float [nt][dim] (device, 8-byte aligned; dim even, <= 256)
 *   scratch : uint64 [nq] (device);  idx : out int32 [nq] (-1 when nt == 0);  dist : out float [nq]
 */
int apap_match_nn(const float *query, const float *train, int nq, int nt, int dim, unsigned long long *scratch,
                  int *idx, float *dist, void *stream);

/*
 * SIFT descriptors at given keypoints: cv.SIFT.compute(image, keypoints) of the reference's keypoint-pair producer
 * (pyviz/utils.py:143-147; SURVEY 8f row N3) for keypoints of octave 0 that share one size and one angle -- the
 * reference builds them as cv.KeyPoint(x, y, 1): size 1, angle -1.  Such keypoints read only the first image of
 * OpenCV's pyramid, the gray image blurred once (sigma^2 = 1.6^2 - 0.5^2), so the call is two kernels: gray + 13-tap
 * blur into base_scratch, then calcSIFTDescriptor per keypoint.  Every component is within +-2 of OpenCV 4.x and almost
 * every one equal (the blur's and the norms' summation orders differ); a keypoint with no sample inside the image gives
 * a zero row.
 *   bgr   : uint8 [h][w][3] (device);  pts : float [n_kp][2] (x, y; device), rounded half to even like cvRound
 *   table : float [n_samples][5] (device): (i, j, rbin, cbin, weight) of every window sample that passes the bin test,
 *           i (row offset) outer and j inner -- what depends only on size and angle, built on the host in float32
 *           exactly as calcSIFTDescriptor does (cvx_proj_b200.utils.sift_sample_table);  ori = 360 - angle
 *           (0 within FLT_EPSILON of 360; 361 for angle -1), in [0, 361]
 *   base_scratch : float [h][w] (device);  desc : out float [n_kp][128] (device), integers 0..255 as OpenCV returns
 */
int apap_sift_describe(const uint8_t *bgr, int h, int w, const float *pts, int n_kp, const float *table, int n_samples,
                       float ori, float *base_scratch, float *desc, void *stream);

/*
 * apap_sift_describe of the image seen through a per-channel LUT: the descriptors of the image whose byte (y, x, c) is
 * lut[c][bgr[y][x][c]], without that image being written (the LUT is read in the gray conversion).  With the LUT of
 * apap_equalize_hist this describes the per-channel equalised image, as the reference does (pyviz/apap.py:234-236).
 *   lut : uint8 [3][256] (device, B G R), not null;  every other argument as in apap_sift_describe
 */
int apap_sift_describe_lut(const uint8_t *bgr, int h, int w, const uint8_t *lut, const float *pts, int n_kp,
                           const float *table, int n_samples, float ori, float *base_scratch, float *desc, void *stream);

/*
 * Per-channel histogram equalisation: cv.merge([cv.equalizeHist(c) for c in cv.split(image)]) of the reference's
 * visualize_equalized_hist (pyviz/utils.py:85-91), bit for bit.  Histograms, then OpenCV's LUT per channel, then
 * (when out is given) the equalised image.
 *   bgr  : uint8 [h][w][3] (device), any byte alignment;  h, w > 0, h w <= INT_MAX
 *   hist : uint32 [3][256] scratch (device), zeroed here;  out: the three histograms
 *   lut  : out uint8 [3][256] (device): OpenCV's LUT per channel (entries below the first non-zero bin are 0)
 *   out  : nullable out uint8 [h][w][3] (device): lut[c][bgr[y][x][c]]
 */
int apap_equalize_hist(const uint8_t *bgr, int h, int w, uint32_t *hist, uint8_t *lut, uint8_t *out, void *stream);

/*
 * The hypothesis loop of cv.findHomography(src, dst, cv.RANSAC, threshold) (OpenCV 4.x RANSACPointSetRegistrator) in
 * the reference's keypoint-pair producer (baseline_stitch_test.py:41): every hypothesis the loop can draw, up to
 * max_iters, with its inlier count.  The subsets come from OpenCV's cv::RNG(0xFFFFFFFFFFFFFFFF) stream with its
 * duplicate rejection, checkSubset and the 10000-attempt limit; the counts use computeError's float32 arithmetic, so
 * subsets and counts are OpenCV's.  The caller applies the adaptive stop (RANSACUpdateNumIters) to the counts and
 * refits the chosen hypothesis's inliers (cvx_proj_b200.utils.find_homography_ransac).
 *   src, dst   : float [n][2] (device, 8-byte aligned), n >= 5;  threshold > 0 (pixels; inlier: err <= (float)(t t))
 *   max_iters  : 1 .. APAP_RANSAC_MAX_ITERS;  workspace: device scratch of apap_ransac_workspace_bytes, 16-byte aligned
 *   subsets    : out int32 [max_iters][4] (device, 16-byte aligned), the accepted subsets in draw order
 *   hyps       : out double [max_iters][9] (device, 8-byte aligned): each subset's homography, OpenCV's runKernel
 *                bit for bit (cv::eigen's Jacobi restated; H22 = 1; NaN when runKernel finds 0 models)
 *   counts     : out int32 [max_iters] (device, 4-byte aligned): inliers of each hypothesis, -1 for 0 models
 *   n_sampled  : out int32 [1] (device, 4-byte aligned): hypotheses filled; < max_iters when the attempt limit ended
 *                the sequence (0: OpenCV finds no model)
 * All max_iters subsets are drawn whatever the adaptive stop would do (the counts that decide it come after), so on
 * degenerate data -- most candidates rejected by checkSubset -- the sampler can run up to 10000 candidates per
 * subset, max_iters x 10000 in all, on one warp: about 16 us per 32 candidates on a B200, i.e. seconds at the
 * default 2000.  OpenCV may stop after one hypothesis on such data.
 */
#define APAP_RANSAC_MAX_ITERS (1 << 20)
int apap_ransac_workspace_bytes(int max_iters, size_t *bytes);
int apap_ransac_homography(const float *src, const float *dst, int n, double threshold, int max_iters, void *workspace,
                           size_t workspace_bytes, int *subsets, double *hyps, int *counts, int *n_sampled,
                           void *stream);

/*
 * apap_ransac_homography for a batch of independent point sets in one launch per kernel (one sampler warp per pair,
 * one fit thread per pair and hypothesis, score CTAs per pair): the reference's multi-image mode matches every image
 * of a case against one centre, and the pairs' serial samplers run side by side on different SMs.  Pair p's record
 * is exactly apap_ransac_homography's record of its points (each pair starts its own cv::RNG(0xFFFFFFFFFFFFFFFF)).
 *   src, dst   : float [total][2] (device, 8-byte aligned), the pairs back to back
 *   offsets    : int32 [batch + 1] (device, 4-byte aligned): pair p is [offsets[p], offsets[p + 1]); a pair of fewer
 *                than 5 points is not sampled (n_sampled 0)
 *   batch      : >= 1, with batch * max_iters <= APAP_RANSAC_MAX_ITERS;  max_n >= 0 sizes the score grid (the
 *                largest pair; a larger pair is still scored completely, with fewer CTAs per hypothesis)
 *   threshold, max_iters : as apap_ransac_homography;  workspace: apap_ransac_batch_workspace_bytes, 16-byte aligned
 *   subsets    : out int32 [batch][max_iters][4] (16-byte aligned), indices local to the pair
 *   hyps       : out double [batch][max_iters][9] (8-byte aligned);  counts: out int32 [batch][max_iters]
 *   n_sampled  : out int32 [batch]
 * The launch ends when its slowest sampler ends: one degenerate pair, most candidates rejected by checkSubset, holds
 * the whole batch for up to max_iters x 10000 candidates (seconds at 2000), as it would hold a single call.
 */
int apap_ransac_batch_workspace_bytes(int batch, int max_iters, size_t *bytes);
int apap_ransac_homography_batch(const float *src, const float *dst, const int *offsets, int batch, int max_n,
                                 double threshold, int max_iters, void *workspace, size_t workspace_bytes,
                                 int *subsets, double *hyps, int *counts, int *n_sampled, void *stream);

/*
 * Panorama assembly of a sharded pass without an all-gather: broadcast `bytes` of device memory at `src` (this
 * rank's row band, already warped) into every GPU's panorama through an NVLS multicast mapping -- `multicast_dst` is
 * the band's address inside the multicast mapping of the panorama buffers (torch symmetric memory's multicast_ptr +
 * offset).  One 16-byte multimem store per 16 bytes: the NVSwitch replicates it, so a rank sends its band once
 * whatever the number of GPUs.  Size and both addresses must be multiples of 16; the caller synchronises the group.
 */
int apap_multicast_copy(const void *src, void *multicast_dst, size_t bytes, void *stream);

/*
 * The same assembly by unicast stores: `bytes` at `src` are written to each of the `n_peers` device addresses in the
 * HOST array `peer_dsts` (the band's address inside every OTHER GPU's panorama: peer-mapped pointers, e.g. torch
 * symmetric memory's buffer_ptrs[r] + offset).  The rank sends its band n_peers times, but no GPU receives its own band
 * back from the switch as it does through a multicast mapping that includes the sender.  Size and all addresses
 * multiples of 16; the caller synchronises the group.
 */
#define APAP_MAX_PEERS 15
int apap_peer_copy(const void *src, void *const *peer_dsts, int n_peers, size_t bytes, void *stream);

/*
 * Pipe probes for the roofline denominators that MEASURED_PEAKS.json does not hold.  Runs `iters` x 16
 * independent operations per thread on every SM and returns the operation count in `ops`; the caller
 * times the launch with events.
 *   APAP_PROBE_FFMA : FP32 FMA pipe, ops = flop (2 per FFMA)   -> the FFMA2 Gram kernel's peak
 *   APAP_PROBE_MUFU : XU pipe (MUFU.EX2), ops = lane operations -> the tcgen05 Gram kernel's peak
 *                     (its weight generation costs 2 MUFU per cell-keypoint pair)
 * sink: float [1] device scratch.
 */
#define APAP_PROBE_FFMA 0
#define APAP_PROBE_MUFU 1
int apap_pipe_probe(int kind, int iters, float *sink, double *ops, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* APAP_B200_H */
