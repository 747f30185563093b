// K3, tile engine -- mesh warp through shared-memory tiles (reference APAP.local_warp pixel loop,
// pyviz/apap.py:206-215).  The plain warp only: fused with K4, the warp runs on the strip kernel of
// csrc/warp_blend.cu, whose batched centre loads beat centre gathers inside the tile loop (c2 49 us against 65 us:
// profiles/r02_warp_tile_history.md).  The engine reads no environment: its schedule is the constants below.
//
// A tile is 128 canvas columns x 8 consecutive row blocks (<= 32 rows).
//
// k_tile_prep (apap_warp_tiles: part of the warp tables, built once per inverted grid and row band like the
//   cell records), one warp per tile: everything about a tile that does not depend on the images, written as
//   one 192-byte TileInfo record --
//     footprint: lane = (cell column, row block) maps the four corners of that pixel rectangle of the
//     tile through the cell's H^-1 (float32 is enough: the result is widened by half a pixel).  Inside a
//     fast-path cell the maps are ratios of affine functions with a denominator of constant sign, so
//     every source pixel the tile can pick lies inside the bounding box of the corner images;
//     the box shape (three tensor maps: wide, square-ish, tall; the first that holds the box);
//     the tile's rows grouped by cell row ("runs"); the mode:
//       black   every cell of the tile maps outside the source: the workers only clear their output
//       staged  gather from the staged box
//       global  no box (it fits none of the shapes, column LUT not monotone): same arithmetic with a
//               bounds test, gathers from global memory
//
// k_warp_tile (apap_warp), persistent warp-specialised CTAs (8 worker warps + 1 producer warp) that claim tiles dynamically
//   (one global counter per launch):
//   producer warp, one tile ahead of the workers (two-stage ring, full / empty mbarriers): streams the
//     tile records into the stage and issues ONE 2-D tensor-map TMA copy (cp.async.bulk.tensor.2d, SASS UTMALDG)
//     that stages the source box; the part of the box outside the image arrives as zeros, which is
//     exactly the reference's "leave black", so no pixel needs a bounds test.  Bulk copies on the same
//     mbarrier stage the fast-path records of the tile's cells, plain stores the tile's column LUT
//     entries: the workers read nothing from global memory.  The lines of the NEXT tile's box are
//     prefetched into L2 through the LSU path a tile ahead;
//   worker warps: 32 columns x 16 rows each; per run the lane's cell record is set up once, then four rows
//     per loop iteration: the float32 fast path with the guard band of csrc/warp_blend.cu (identical
//     decisions), LDS.U8 gathers from the staged box, STS.U8 into the warp's own output block; guard-band
//     pixels are re-decided in float64 and fetched from global memory exactly like the reference;
//   output: every warp stores its own 16 x 96-byte block (double buffered) with one tensor-map TMA store
//     (UTMASTG) -- no CTA-wide barrier anywhere in the tile loop.  An NVLS multicast panorama (16-byte
//     multimem.st, whole 384-byte rows) and canvases whose rows are not 16-byte aligned are written by
//     all workers together after a named barrier.
#include <cuda.h>

#include <atomic>
#include <limits.h>
#include <stddef.h>
#include <string.h>

#include "common.cuh"
#include "warp_common.cuh"

namespace apap {

constexpr int kTileCtas = 3;                              // resident CTAs per SM, 2 stages each: 6 boxes in flight per SM
constexpr int kWorkerWarps = 8;
constexpr int kWorkerThreads = kWorkerWarps * 32;
constexpr int kTileThreads = kWorkerThreads + 32;         // + the producer warp
constexpr int kTileCols = 128;                            // 4 chunks of 32 columns
// source-box stages of the ring x row blocks per tile: 2 x 8 (32 rows, 20 KB box); 3 x 6 (24 rows, 16 KB box) measured
// the same (profiles/r02_warp_tile_history.md)
constexpr int kStages = 2;
constexpr int kTileBlocks = 8;                            // row blocks per tile
constexpr int kTileRows = kTileBlocks * kBlockRows;       // 32
constexpr int kWarpRows = kTileRows / 2;                  // 16 canvas rows per worker warp
static_assert(kTileBlocks <= 8 && kTileBlocks % 2 == 0 && kStages >= 2, "tile shape");
constexpr int kWarpPitch = 32 * 3;                        // 96 B: a worker warp's 32 columns
constexpr int kWarpOutBytes = kWarpRows * kWarpPitch;     // 1536 B: a warp's dense output block
constexpr int kBoxBytes = 20 * 1024;                      // staged source box
constexpr uint32_t kFlagOff = kBoxBytes + 4;              // staged mode, "guard band" marker: reads the zero word behind the box
constexpr uint32_t kNoPixel = 0xffffffffu;                // global mode: "leave black"
constexpr uint32_t kFlagPixel = 0xfffffffeu;              // global mode: guard band
constexpr int kMaxCellCols = 32;                          // footprint: at most this many cell columns per tile
constexpr int kCounterSlots = 64;                         // tile counters: launch n uses slot n % 64
constexpr int kGroupRows = 4;                             // rows a lane processes per loop iteration (independent gathers in flight)
constexpr int kRecRuns = 4;                               // cell rows of a tile whose records are staged ...
constexpr int kRecCols = 16;                              // ... for at most this many cell columns (else global loads)

enum TileMode : int { kBlack = 0, kStagedMode = 1, kGlobal = 3, kDone = 4 };

// box shapes of the staged source: {bytes per row, rows (<= 256)}, each <= kBoxBytes.  The row pitch is a multiple
// of 128 bytes = all 32 banks: the 32 gathers of a warp walk along a source row and step to the next one somewhere
// in the middle, and with this pitch the bytes behind the step fall into the banks the row would have continued
// in (a 448-byte pitch: 2.6 M bank conflicts on the gathers of c3, this one: 0.95 M; ncu, profiles/)
constexpr int kBoxShapes = 3;
__host__ __device__ constexpr int box_w(int m) { return m == 0 ? 512 : m == 1 ? 256 : 128; }
__host__ __device__ constexpr int box_h(int m) { return kBoxBytes / box_w(m) > 256 ? 256 : kBoxBytes / box_w(m); }

struct TileInfo {                // one tile, as k_tile_prep writes it and the workers read it (192 bytes = 12 x uint4)
  int x_lo, y_lo;                // first source pixel column / row of the staged box (kGlobal: 0, 0)
  int pitch;                     // bytes per staged row (kGlobal: pixels per image row)
  int shift;                     // byte offset of pixel x_lo inside a staged row
  int mode;
  int r_first, n_rows;           // canvas rows of the tile
  int c_lo;                      // first cell column of the tile
  int rec_ok;                    // the cell records of the tile are staged in Stage::rec (slot = run index)
  int n_runs;
  int j0, jw;                    // canvas columns of the tile
  int shape;                     // box shape (tensor map) of the staged box, -1 = none
  int c0;                        // first uint32 column of the box in the source's tensor map
  int ncc;                       // cell columns of the tile
  int pad;
  int4 run[8];                   // the tile's rows by cell row: {first canvas row, rows, cell row, dy of the first row}
};
static_assert(sizeof(TileInfo) == 192, "TileInfo is copied as 12 uint4");

struct Stage {
  alignas(128) uint8_t box[kBoxBytes];
  alignas(16) uint8_t zero[16];
  alignas(16) float4 rec[kRecRuns][kRecCols][3];          // fast-path records of the tile's cells
  alignas(16) uint2 lut[kTileCols];                       // the tile's column LUT entries
};

struct TileSmem {
  Stage st[kStages];
  alignas(128) uint8_t out[2][kWorkerWarps][kWarpOutBytes];   // double buffered, per worker warp: 16 rows x 96 B, dense
  alignas(16) TileInfo info[kStages];
  alignas(8) uint64_t full[kStages];
  uint64_t empty[kStages];
};

static_assert(offsetof(Stage, zero) == kBoxBytes, "the zero word sits right behind the staged box");
static_assert(box_w(0) * box_h(0) <= kBoxBytes && box_w(1) * box_h(1) <= kBoxBytes && box_w(2) * box_h(2) <= kBoxBytes, "box shapes");
static_assert(sizeof(TileSmem) * kTileCtas + 1024 * kTileCtas <= 227 * 1024, "shared memory of the resident CTAs");

__device__ unsigned int g_tile_next[kCounterSlots];       // tiles handed out beyond the first gridDim.x
__device__ unsigned int g_tile_done[kCounterSlots];       // CTAs that have stopped claiming (the last one resets the slot)

struct TileParams {
  CUtensorMap maps[kBoxShapes];  // the source image as uint32 [src_h][src_w * 3 / 4], one map per box shape
  CUtensorMap out_map;           // the output band as uint32 [band_rows][canvas_w * 3 / 4], box = 16 rows x 96 bytes
  WarpParams w;
  const int2 *col_ext;           // [grid_cols] {first, last} canvas column of the cell column
  int store_mode;                // 0 bytes, 1 words, 2 TMA (one tensor-map store per warp block), 3 multimem
  int tiles_x, n_tiles;
  int slot;                      // which pair of tile counters this launch uses
  TileInfo *tiles;               // [n_tiles]: written by k_tile_prep (apap_warp_tiles), streamed by the producer warps
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// waiting worker: sleep between polls, so that the polls of warps that ran ahead do not take issue slots from the others
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) __nanosleep(64);
}
__device__ __forceinline__ void worker_barrier() {          // the 8 worker warps only (named barrier 1)
  asm volatile("bar.sync 1, %0;" ::"n"(kWorkerThreads) : "memory");
}
// 2-D tensor-map TMA copy global -> shared (SASS: UTMALDG); coordinates in elements of the map, out-of-range parts
// of the box arrive as zeros.  The innermost coordinate times the element size must be a multiple of 16 bytes
// (anything else raises "illegal instruction": tools/tma_lab.cu).
__device__ __forceinline__ void tma_load_2d(void *dst_smem, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}
// 2-D tensor-map TMA store shared -> global (SASS: UTMASTG); the part of the box outside the tensor is dropped
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, int c0, int c1, const void *src_smem) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(src_smem)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_but_one() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }

// kRows (1, 2 or 4) consecutive canvas rows of one lane (same cell): gather offsets on the float32 fast path --
// packed FP32x2, two rows per instruction; same arithmetic and decisions as block_issue of csrc/warp_blend.cu --,
// gathers, bytes into the warp's output block; then the float64 path for the rows whose quotient lies inside
// the guard band.  All kRows pixels are independent: that many gathers are in flight per lane.
//   kStaged: the shared-memory address of the pixel comes straight from the float bits of the floors
//   (address = ty_bits * pitch + tx_bits * 3 + kbase), no bounds test: whatever the tile can pick is inside
//   the staged box and the box is zero outside the image;  else: test against the image, gather from global memory.
template <bool kStaged, int kRows>
__device__ __forceinline__ void tile_rows(const WarpParams &p, const CellState &c, int pitch, int kbase, uint32_t guard_addr,
                                          uint8_t *__restrict__ orow, float dy0, int x, int y) {
  constexpr int kPairs = (kRows + 1) / 2;
  const uint32_t guard = kStaged ? guard_addr : kFlagPixel;
  const float2 km = make_float2(kMagic, kMagic), nkm = make_float2(-kMagic, -kMagic), nh = make_float2(-0.5f, -0.5f);
  uint32_t so[2 * kPairs];                     // kStaged: shared-memory address; else pixel index / kNoPixel / kFlagPixel
#pragma unroll
  for (int k = 0; k < kPairs; ++k) {
    const float2 dy = __fadd2_rn(make_float2(dy0, dy0), make_float2((float)(2 * k), (float)(2 * k + 1)));
    const float2 n0 = __ffma2_rn(make_float2(c.b0, c.b0), dy, make_float2(c.m0, c.m0));
    const float2 n1 = __ffma2_rn(make_float2(c.b1, c.b1), dy, make_float2(c.m1, c.m1));
    const float2 d = __ffma2_rn(make_float2(c.b2, c.b2), dy, make_float2(c.m2, c.m2));
    const float2 r = make_float2(rcp_approx(d.x), rcp_approx(d.y));
    const float2 qxq = __fmul2_rn(n0, r), qyq = __fmul2_rn(n1, r);
    const float2 tx = __fadd2_rd(qxq, km), ty = __fadd2_rd(qyq, km);            // floor + kMagic
    const float2 gx = __fadd2_rn(tx, nkm), gy = __fadd2_rn(ty, nkm);            // floor
    const float2 fx = __fadd2_rn(qxq, make_float2(-gx.x, -gx.y));               // exact fraction in [0, 1)
    const float2 fy = __fadd2_rn(qyq, make_float2(-gy.x, -gy.y));
    const float2 hx = __fadd2_rn(fx, nh), hy = __fadd2_rn(fy, nh);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float txe = e ? tx.y : tx.x, tye = e ? ty.y : ty.x;
      const float hxe = e ? hx.y : hx.x, hye = e ? hy.y : hy.x;
      const bool clear = fmaxf(fabsf(hxe), fabsf(hye)) <= c.hme;
      uint32_t off;
      if (kStaged) {
        off = (uint32_t)(__float_as_int(tye) * pitch + (__float_as_int(txe) * 3 + kbase));
      } else {
        // a lane whose cell maps outside the source (mixed warp) carries an x base beyond the image (tile_warp_rows)
        const int ix = __float_as_int(txe) + c.qbx;
        const int iy = __float_as_int(tye) + c.qby;
        const uint32_t in_off = (uint32_t)(iy * p.src_w + ix);
        asm("{\n\t.reg .pred p;\n\t"
            "setp.lt.u32 p, %1, %2;\n\t"
            "setp.lt.and.u32 p, %3, %4, p;\n\t"
            "selp.b32 %0, %5, %6, p;\n\t}"
            : "=r"(off)
            : "r"(ix), "r"(p.src_w), "r"(iy), "r"(p.src_h), "r"(in_off), "r"(kNoPixel));
      }
      so[2 * k + e] = clear ? off : guard;
    }
  }
  bool any_guard = false;
#pragma unroll
  for (int k = 0; k < kRows; ++k) {
    const uint32_t o = so[k];
    any_guard = any_guard || o == guard;
    uint32_t b0, b1, b2;
    if (kStaged) {
      asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b0) : "r"(o));
      asm volatile("ld.shared.u8 %0, [%1+1];" : "=r"(b1) : "r"(o));
      asm volatile("ld.shared.u8 %0, [%1+2];" : "=r"(b2) : "r"(o));
    } else {
      b0 = b1 = b2 = 0;
      if (o < kFlagPixel) {
        const uint8_t *q = p.src + (size_t)o * 3;
        b0 = __ldg(q); b1 = __ldg(q + 1); b2 = __ldg(q + 2);
      }
    }
    uint8_t *dst = orow + k * kWarpPitch;
    dst[0] = (uint8_t)b0; dst[1] = (uint8_t)b1; dst[2] = (uint8_t)b2;
  }
  // rare: the reference's float64 arithmetic, bytes from global memory
  if (__any_sync(0xffffffffu, any_guard)) {
    const float *hinv = p.cell_hinv + (size_t)c.cell * 9;
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      if (so[k] != guard) continue;
      const int idx = exact_lookup(hinv, x, y + k, p.src_w, p.src_h);
      uint32_t val = 0;
      if (idx >= 0) {
        const uint8_t *q = p.src + (size_t)(unsigned)idx * 3;
        val = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16);
      }
      uint8_t *dst = orow + k * kWarpPitch;
      dst[0] = (uint8_t)val; dst[1] = (uint8_t)(val >> 8); dst[2] = (uint8_t)(val >> 16);
    }
  }
}

// A worker warp's share of one tile: 32 columns x the canvas rows [row_lo, row_hi].  The tile's rows come as runs of
// one cell row each; per run the lane's cell record is set up once (from shared memory, where the producer staged
// it), then the rows go by four at a time.
template <bool kStaged>
__device__ __forceinline__ void tile_warp_rows(const WarpParams &p, const TileInfo &f, const Stage &stg,
                                               uint8_t *__restrict__ warp_out, const uint2 cl, int x, int lane, int row_lo,
                                               int row_hi) {
  // tile-invariant values into registers once (the byte stores into the output block could alias them for the compiler)
  const int x_lo = f.x_lo, y_lo = f.y_lo, bpitch = f.pitch, shift = f.shift, rec_ok = f.rec_ok, n_runs = f.n_runs;
  const int rec_col = (int)cl.x - f.c_lo, grid_cols = p.grid_cols, off_y = p.off_y, force = p.force_exact;
  const float dxf = __uint_as_float(cl.y);
  const uint32_t box_addr = smem_u32(stg.box), guard_addr = box_addr + kFlagOff;
  uint8_t *const out_lane = warp_out + lane * 3 - row_lo * kWarpPitch;   // row r of the canvas -> out_lane + r * 96
  CellState c;
#pragma unroll 1
  for (int ri = 0; ri < n_runs; ++ri) {
    const int4 run = f.run[ri];
    int lo = max(run.x, row_lo);
    const int hi = min(run.x + run.y - 1, row_hi);
    if (lo > hi) continue;                      // warp-uniform: none of this run's rows are this warp's
    c.cell_row = run.z;
    c.cell = run.z * grid_cols + (int)cl.x;
    float4 u, v, w;
    if (rec_ok) {
      const float4 *rec = stg.rec[ri][rec_col];
      u = rec[0]; v = rec[1]; w = rec[2];
    } else {
      const float4 *rec = p.cell_fast + (size_t)c.cell * 3;
      u = __ldg(rec); v = __ldg(rec + 1); w = __ldg(rec + 2);
    }
    c.m0 = fmaf(u.x, dxf, u.z); c.b0 = u.y;
    c.m1 = fmaf(u.w, dxf, v.y); c.b1 = v.x;
    c.m2 = fmaf(v.z, dxf, w.x); c.b2 = v.w;
    c.qby = __float_as_int(w.z);
    // g = 0.5 - eps; a record with g < 0 (degenerate cell, forced) never passes; NaN never passes; an outside
    // cell (g = 2) always passes
    c.hme = force ? -1.f : w.w;
    c.outside = w.w > 1.f && !force;
    // global mode, a lane whose cell maps outside the source in a mixed warp: an x index beyond the image
    c.qbx = (!kStaged && c.outside) ? 0x40000000 : __float_as_int(w.y);
    // staged: address = box + (iy - y_lo) * pitch + (ix - x_lo) * 3 + shift, iy = ty_bits + qby, ix = tx_bits + qbx
    const int kbase = (int)box_addr + (c.qby - y_lo) * bpitch + (c.qbx - x_lo) * 3 + shift;
    uint8_t *orow = out_lane + lo * kWarpPitch;
    int y = lo - off_y;
    if (__all_sync(0xffffffffu, c.outside)) {   // every pixel of these rows stays black under this warp
      for (; lo <= hi; ++lo, orow += kWarpPitch) { orow[0] = 0; orow[1] = 0; orow[2] = 0; }
      continue;
    }
    float dyf = (float)(run.w + lo - run.x);
#pragma unroll 1
    for (; lo + kGroupRows <= hi + 1; lo += kGroupRows, y += kGroupRows, orow += kGroupRows * kWarpPitch, dyf += (float)kGroupRows)
      tile_rows<kStaged, kGroupRows>(p, c, bpitch, kbase, guard_addr, orow, dyf, x, y);
    if (lo + 2 <= hi + 1) {                     // the last 0 .. 3 rows
      tile_rows<kStaged, 2>(p, c, bpitch, kbase, guard_addr, orow, dyf, x, y);
      lo += 2; y += 2; orow += 2 * kWarpPitch; dyf += 2.f;
    }
    if (lo == hi) tile_rows<kStaged, 1>(p, c, bpitch, kbase, guard_addr, orow, dyf, x, y);
  }
}

// One warp per tile: the TileInfo record.  Runs ahead of k_warp_tile in the same apap_warp call; thousands of these
// latency-bound warps are in flight at once, where a single producer warp per CTA doing the same per tile sat on the
// critical path (3.3 us per tile; with no pixel work at all c3 still took 78 us: profiles/r02_warp_tile_history.md).
__global__ void __launch_bounds__(256) k_tile_prep(const __grid_constant__ TileParams tp) {
  const WarpParams &p = tp.w;
  const int lane = threadIdx.x & 31;
  const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tile >= tp.n_tiles) return;                          // warp-uniform
  const int tiles_x = tp.tiles_x;
  const int b = lane & 7, ccs = lane >> 3;                 // this lane's footprint items: row block b, cell columns ccs + 4 u
  const int ty = tile / tiles_x, txi = tile - ty * tiles_x;
  const int j0 = txi * kTileCols, jw = min(kTileCols, p.canvas_w - j0), j1 = j0 + jw - 1;
  const int tb0 = ty * kTileBlocks, nbt = min(kTileBlocks, p.n_blocks - tb0);
  const uint2 e = __ldg(p.row_blocks + tb0 + min(b, nbt - 1));
  const int i0 = (int)(e.x & 0x0fffffffu), n = (int)(e.x >> 28), cr = (int)(e.y & 0xffffu);
  // every cell column of the tile must lie in [c_lo, c_hi] (always, for the monotone LUT of a sorted mesh)
  uint2 lut[kTileCols / 32];
#pragma unroll
  for (int q = 0; q < kTileCols / 32; ++q) lut[q] = __ldg(p.col_lut + min(j0 + lane + 32 * q, j1));
  const int c_lo = (int)__shfl_sync(0xffffffffu, lut[0].x, 0);
  const int c_hi = (int)__shfl_sync(0xffffffffu, lut[(kTileCols - 1) / 32].x, 31);     // entry of column j1 (clamped)
  bool bad_lut = c_hi < c_lo;
#pragma unroll
  for (int q = 0; q < kTileCols / 32; ++q) bad_lut = bad_lut || (int)lut[q].x < c_lo || (int)lut[q].x > c_hi;
  bad_lut = __any_sync(0xffffffffu, bad_lut);
  bool odd = bad_lut || c_hi - c_lo >= kMaxCellCols;
  float bx0 = 3e9f, bx1 = -3e9f, by0 = 3e9f, by1 = -3e9f;
  bool all_out = true;
  if (!odd) {
    const float ya = (float)(i0 - p.off_y), yb = (float)(i0 + n - 1 - p.off_y);
    const int trips = (c_hi - c_lo + 4) >> 2;              // warp-uniform
#pragma unroll 2
    for (int u = 0; u < trips; ++u) {
      const int cc = c_lo + ccs + 4 * u;
      const int ccl = min(cc, c_hi);                       // loads stay in range; the item counts only if cc <= c_hi
      const int2 ce = __ldg(tp.col_ext + ccl);
      const size_t cell = (size_t)(cr * p.grid_cols + ccl);
      const float g = __ldg(reinterpret_cast<const float *>(p.cell_fast) + cell * kHinvRow + 11);
      const float *h = p.cell_hinv + cell * 9;
      const float h0 = __ldg(h + 0), h1 = __ldg(h + 1), h2 = __ldg(h + 2), h3 = __ldg(h + 3), h4 = __ldg(h + 4);
      const float h5 = __ldg(h + 5), h6 = __ldg(h + 6), h7 = __ldg(h + 7), h8 = __ldg(h + 8);
      const int xa = max(ce.x, j0), xb = min(ce.y, j1);
      const bool item = cc <= c_hi && b < nbt && xa <= xb;
      const float xfa = (float)(xa - p.off_x), xfb = (float)(xb - p.off_x);
      float qx[4], qy[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const float xf = (v & 1) ? xfb : xfa, yf = (v & 2) ? yb : ya;
        const float rt = rcp_approx(fmaf(h6, xf, fmaf(h7, yf, h8)));
        qx[v] = fmaf(h0, xf, fmaf(h1, yf, h2)) * rt;
        qy[v] = fmaf(h3, xf, fmaf(h4, yf, h5)) * rt;
      }
      const float lx = fminf(fminf(qx[0], qx[1]), fminf(qx[2], qx[3])), ux = fmaxf(fmaxf(qx[0], qx[1]), fmaxf(qx[2], qx[3]));
      const float ly = fminf(fminf(qy[0], qy[1]), fminf(qy[2], qy[3])), uy = fmaxf(fmaxf(qy[0], qy[1]), fmaxf(qy[2], qy[3]));
      // finite and small?  (fminf / fmaxf drop a NaN, so test every corner)
      bool fin = true;
#pragma unroll
      for (int v = 0; v < 4; ++v) fin = fin && fabsf(qx[v]) < 1e9f && fabsf(qy[v]) < 1e9f;
      if (item) {
        all_out = all_out && g > 1.f;
        if (fin) { bx0 = fminf(bx0, lx); bx1 = fmaxf(bx1, ux); by0 = fminf(by0, ly); by1 = fmaxf(by1, uy); }
        else odd = true;                                   // cannot bound this rectangle's image
      }
    }
  }
  odd = __any_sync(0xffffffffu, odd);
  all_out = __all_sync(0xffffffffu, all_out) && !odd;
  // the pixel picked is floor(q): widen by half a pixel for the float32 evaluation, then floor
  const int ix0 = __reduce_min_sync(0xffffffffu, __float2int_rd(bx0 - 0.5f));
  const int ix1 = __reduce_max_sync(0xffffffffu, __float2int_rd(bx1 + 0.5f));
  const int iy0 = __reduce_min_sync(0xffffffffu, __float2int_rd(by0 - 0.5f));
  const int iy1 = __reduce_max_sync(0xffffffffu, __float2int_rd(by1 + 0.5f));

  // cell-row runs of the tile's blocks (lanes 0 .. nbt-1 hold block b = lane): run index = record slot
  const int cr_prev = __shfl_up_sync(0xffffffffu, cr, 1);
  const unsigned starts = __ballot_sync(0xffffffffu, lane < nbt && (lane == 0 || cr != cr_prev));
  const int n_runs = __popc(starts), ncc = c_hi - c_lo + 1;
  const bool rec_ok = n_runs <= kRecRuns && ncc >= 1 && ncc <= kRecCols && !all_out && !bad_lut;
  // lane r: run r = blocks run_first .. run_last
  const int run_id = min(lane, n_runs - 1);
  const int run_first = __fns(starts, 0, run_id + 1);
  const int run_last = (run_id + 1 < n_runs ? (int)__fns(starts, 0, run_id + 2) : nbt) - 1;
  const int run_row0 = __shfl_sync(0xffffffffu, i0, run_first);
  const int run_row1 = __shfl_sync(0xffffffffu, i0 + n - 1, run_last);
  const int run_cr = __shfl_sync(0xffffffffu, cr, run_first);
  const int run_dy = __shfl_sync(0xffffffffu, (int)(e.y >> 16), run_first);

  int mode = kGlobal, x_lo = 0, y_lo = 0, bpitch = p.src_w, shift = 0, shape = -1, c0 = 0;
  if (!odd && all_out) {
    mode = kBlack;
  } else if (!odd && ix0 <= ix1 && iy0 <= iy1) {
    // the box starts at a 16-byte aligned byte of the row (TMA: innermost coordinate x element size % 16 == 0)
    const long long need_w = ((long long)ix1 - ix0 + 1) * 3 + 15, need_h = (long long)iy1 - iy0 + 1;
#pragma unroll
    for (int m = kBoxShapes - 1; m >= 0; --m)
      if (need_w <= box_w(m) && need_h <= box_h(m)) shape = m;
    if (shape >= 0) {
      c0 = ((ix0 * 3) >> 4) << 2;                          // floor to 16 bytes: first uint32 element of the box
      mode = kStagedMode;
      x_lo = ix0; y_lo = iy0;
      bpitch = shape == 0 ? box_w(0) : shape == 1 ? box_w(1) : box_w(2);
      shift = ix0 * 3 - (c0 << 2);
    }
  }
  const int r_first = __shfl_sync(0xffffffffu, i0, 0);
  const int r_last = __shfl_sync(0xffffffffu, i0 + n - 1, nbt - 1);
  TileInfo &f = tp.tiles[tile];
  if (lane < 8)
    f.run[lane] = lane < n_runs ? make_int4(run_row0, run_row1 - run_row0 + 1, run_cr, run_dy) : make_int4(0, 0, 0, 0);
  if (lane == 0) {
    f.x_lo = x_lo; f.y_lo = y_lo; f.pitch = bpitch; f.shift = shift; f.mode = mode;
    f.r_first = r_first; f.n_rows = r_last - r_first + 1; f.c_lo = c_lo; f.rec_ok = rec_ok ? 1 : 0;
    f.n_runs = n_runs; f.j0 = j0; f.jw = jw; f.shape = shape; f.c0 = c0; f.ncc = ncc; f.pad = 0;
  }
}

__global__ void __launch_bounds__(kTileThreads, kTileCtas) k_warp_tile(const __grid_constant__ TileParams tp) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem &sm = *reinterpret_cast<TileSmem *>(smem_raw);
  const WarpParams &p = tp.w;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    for (int q = 0; q < kStages; ++q) { mbar_init(&sm.full[q], 1); mbar_init(&sm.empty[q], kWorkerWarps); }
    mbar_fence_init();
  }
  if (tid < 4 * kStages) reinterpret_cast<uint32_t *>(sm.st[tid >> 2].zero)[tid & 3] = 0u;
  __syncthreads();

  if (warp == kWorkerWarps) {
    // =============================== producer warp ==================================================
    // Streams the tiles' records (k_tile_prep) into the stages and issues the copies.  Tiles are claimed two ahead
    // and the record + column LUT entries of the next tile are loaded while the current one is published, so the
    // per-tile path is: wait for the stage, 5 shared stores, arrive, TMA.
    const int tiles_x = tp.tiles_x;
    const size_t src_pitch = (size_t)p.src_w * 3;
    const uint4 *table = reinterpret_cast<const uint4 *>(tp.tiles);
    int tile = blockIdx.x;                                 // the first tile is static, the others are claimed
    int tile_next = 0, claim = 0;
    if (lane == 0) tile_next = (int)(gridDim.x + atomicAdd(&g_tile_next[tp.slot], 1u));
    tile_next = __shfl_sync(0xffffffffu, tile_next, 0);
    // record (lanes 0-11: one uint4 each) and LUT entries of `tile`
    uint4 rec = make_uint4(0u, 0u, 0u, 0u);
    uint2 lut[kTileCols / 32];
#pragma unroll
    for (int q = 0; q < kTileCols / 32; ++q) lut[q] = make_uint2(0u, 0u);
    auto fetch = [&](int t) {
      if (t < tp.n_tiles) {
        if (lane < 12) rec = __ldg(table + (size_t)t * 12 + lane);
        const int txi = t % tiles_x, j0 = txi * kTileCols, j1 = min(j0 + kTileCols, p.canvas_w) - 1;
#pragma unroll
        for (int q = 0; q < kTileCols / 32; ++q) lut[q] = __ldg(p.col_lut + min(j0 + lane + 32 * q, j1));
      }
    };
    fetch(tile);
    for (int k = 0;; ++k) {
      const int s = k % kStages;
      const uint32_t ring_par = (uint32_t)(k / kStages) & 1u;
      TileInfo &f = sm.info[s];
      if (tile >= tp.n_tiles) {                            // no tiles left: tell the workers, release the counter slot
        mbar_wait(&sm.empty[s], ring_par ^ 1u);
        if (lane == 0) {
          f.mode = kDone;
          mbar_arrive(&sm.full[s]);
          __threadfence();
          if (atomicAdd(&g_tile_done[tp.slot], 1u) == gridDim.x - 1) {   // every CTA has made its last claim
            g_tile_next[tp.slot] = 0u;
            g_tile_done[tp.slot] = 0u;
            __threadfence();
          }
        }
        break;
      }
      if (lane == 0 && tile_next < tp.n_tiles) claim = (int)(gridDim.x + atomicAdd(&g_tile_next[tp.slot], 1u));
      // what this warp needs of the current record, before the registers take the next one
      const uint4 cur = rec;
      const int y_lo = __shfl_sync(0xffffffffu, (int)rec.y, 0);          // uint4 #0 = {x_lo, y_lo, pitch, shift}
      const int bpitch = __shfl_sync(0xffffffffu, (int)rec.z, 0);
      const int mode = __shfl_sync(0xffffffffu, (int)rec.x, 1);          // uint4 #1 = {mode, r_first, n_rows, c_lo}
      const int c_lo = __shfl_sync(0xffffffffu, (int)rec.w, 1);
      const int rec_ok = __shfl_sync(0xffffffffu, (int)rec.x, 2);        // uint4 #2 = {rec_ok, n_runs, j0, jw}
      const int n_runs = __shfl_sync(0xffffffffu, (int)rec.y, 2);
      const int shape = __shfl_sync(0xffffffffu, (int)rec.x, 3);         // uint4 #3 = {shape, c0, ncc, pad}
      const int c0 = __shfl_sync(0xffffffffu, (int)rec.y, 3);
      const int ncc = __shfl_sync(0xffffffffu, (int)rec.z, 3);
      const int run_cr = __shfl_sync(0xffffffffu, (int)rec.z, 4 + min(lane, 7));   // uint4 #4+r = run r
      uint2 cur_lut[kTileCols / 32];
#pragma unroll
      for (int q = 0; q < kTileCols / 32; ++q) cur_lut[q] = lut[q];
      fetch(tile_next);                                      // in flight while this tile is published

      mbar_wait(&sm.empty[s], ring_par ^ 1u);                // the workers have left this stage
      if (lane < 12) reinterpret_cast<uint4 *>(&f)[lane] = cur;
#pragma unroll
      for (int q = 0; q < kTileCols / 32; ++q) sm.st[s].lut[lane + 32 * q] = cur_lut[q];
      __syncwarp();
      const uint32_t box_bytes = shape < 0 ? 0u : (uint32_t)(bpitch * (shape == 0 ? box_h(0) : shape == 1 ? box_h(1) : box_h(2)));
      const uint32_t rec_bytes = (rec_ok && mode != kBlack) ? (uint32_t)(ncc * kHinvRow * 4) : 0u;
      if (lane == 0) {
        if (box_bytes + rec_bytes) mbar_arrive_expect_tx(&sm.full[s], box_bytes + rec_bytes * n_runs);
        else mbar_arrive(&sm.full[s]);
        if (shape >= 0) tma_load_2d(sm.st[s].box, &tp.maps[shape], c0, y_lo, &sm.full[s]);
      }
      __syncwarp();
      if (rec_bytes && lane < n_runs)                        // one bulk copy per cell row: the records of cells c_lo .. c_hi
        bulk_g2s(&sm.st[s].rec[lane][0][0], p.cell_fast + (size_t)(run_cr * p.grid_cols + c_lo) * 3, rec_bytes, &sm.full[s]);
      // The next tile's record has arrived by now: pull the lines of its box into L2 through the LSU path.  The copy
      // into the stage cannot start before the workers free the stage, a tile from now; a cold box then took 2.5-3.4 us
      // to arrive (a tile is 2 us of work) although the same copy from L2 takes 0.4 us (tools/tma_lab.cu).
      if (tile_next < tp.n_tiles) {
        const int nshape = __shfl_sync(0xffffffffu, (int)rec.x, 3), nc0 = __shfl_sync(0xffffffffu, (int)rec.y, 3);
        const int ny = __shfl_sync(0xffffffffu, (int)rec.y, 0);
        if (nshape >= 0) {
          const int bw = nshape == 0 ? box_w(0) : nshape == 1 ? box_w(1) : box_w(2);
          const int bh = nshape == 0 ? box_h(0) : nshape == 1 ? box_h(1) : box_h(2);
          const int lines = bw >> 7;                         // 128-byte lines per box row: 4, 2 or 1
          for (int q = lane; q < bh * lines; q += 32) {
            const int r = q / lines, l = q - r * lines;
            const long long yy = (long long)ny + r, xb = (long long)nc0 * 4 + l * 128;
            if (yy >= 0 && yy < p.src_h && xb >= 0 && xb < (long long)src_pitch) prefetch_l2(p.src + (size_t)yy * src_pitch + (size_t)xb);
          }
        }
      }
      tile = tile_next;
      tile_next = __shfl_sync(0xffffffffu, claim, 0);
      if (tile >= tp.n_tiles) tile_next = tp.n_tiles;        // nothing was claimed behind the end
    }
    return;
  }

  // ================================= worker warps ===================================================
  const int cw = warp & 3, half = warp >> 2;               // column chunk, first / second half of the tile's rows
  const int lane_col = cw * 32 + lane;
  const uint32_t pitch = (uint32_t)p.canvas_w * 3u;
  for (int k = 0;; ++k) {
    const int s = k % kStages;
    uint8_t *warp_out = sm.out[k & 1][warp];
    if (tp.store_mode == 2) bulk_wait_read_but_one();        // this thread's store of two tiles ago has read its block
    mbar_wait_relaxed(&sm.full[s], (uint32_t)(k / kStages) & 1u);   // box, records, LUT and info of this tile have landed
    const TileInfo &f = sm.info[s];
    const int mode = f.mode;
    if (mode == kDone) break;
    const int r_first = f.r_first, n_rows = f.n_rows, j0 = f.j0, jw = f.jw;
    const uint2 cl = sm.st[s].lut[lane_col];
    const int x = j0 + lane_col - p.off_x;                 // lanes at or past jw: bytes that are never stored
    // the two warps of a column chunk share the tile's rows: the first 16 and the last 16 (a tile of 31 rows has its
    // middle row computed by both, same bytes), so that every warp's block is one whole 16-row store; a tile of fewer
    // than 16 rows (end of a band) is all the first warp's
    const int row_lo = (half && n_rows >= kWarpRows) ? r_first + n_rows - kWarpRows : r_first + half * kWarpRows;
    const int row_hi = half ? r_first + n_rows - 1 : min(r_first + kWarpRows, r_first + n_rows) - 1;
    if (mode == kStagedMode) {
      tile_warp_rows<true>(p, f, sm.st[s], warp_out, cl, x, lane, row_lo, row_hi);
    } else if (mode == kGlobal) {
      tile_warp_rows<false>(p, f, sm.st[s], warp_out, cl, x, lane, row_lo, row_hi);
    } else {                                                  // kBlack: clear the block
      for (int q = lane; q < kWarpOutBytes / 16; q += 32) reinterpret_cast<uint4 *>(warp_out)[q] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.empty[s]);                // this warp no longer reads the stage (f is dead from here)
    const int my_rows = row_hi - row_lo + 1;
    if (tp.store_mode == 2) {
      // this warp's block leaves on its own: one tensor-map store of its 16 rows (columns past the canvas are dropped
      // by the map)
      fence_proxy_async_smem();
      __syncwarp();
      const int cbytes = min(kWarpPitch, jw * 3 - cw * kWarpPitch);    // bytes of this warp's columns inside the canvas
      if (lane == 0 && cbytes > 0) {
        if (my_rows == kWarpRows) {                          // the whole block: one tensor-map store
          tma_store_2d(&tp.out_map, (j0 * 3 + cw * kWarpPitch) >> 2, row_lo - p.row0, warp_out);
        } else {                                             // end of a band: row by row
          uint8_t *g = p.out + ((size_t)(row_lo - p.row0) * pitch + (size_t)j0 * 3 + cw * kWarpPitch);
          for (int r = 0; r < my_rows; ++r) bulk_s2g(g + (size_t)r * pitch, warp_out + r * kWarpPitch, (uint32_t)cbytes);
        }
      }
      bulk_commit();
    } else {
      // all workers together: whole rows of the tile out of the eight blocks (tile row r < 16: first warps' blocks,
      // row r; else the second warps' blocks, row r - second0)
      worker_barrier();
      const uint8_t *blocks = sm.out[k & 1][0];
      const int second0 = n_rows >= kWarpRows ? n_rows - kWarpRows : kWarpRows;
      const uint32_t row_bytes = (uint32_t)jw * 3u;
      uint8_t *gout = p.out + ((size_t)(r_first - p.row0) * pitch + (size_t)j0 * 3);
      if (tp.store_mode == 3) {
        const int per_row = (int)(row_bytes >> 4);
        for (int q = tid; q < n_rows * per_row; q += kWorkerThreads) {
          const int r = q / per_row, u = q - r * per_row, h2 = r >= kWarpRows, c2 = u / (kWarpPitch / 16);
          const uint4 v = *reinterpret_cast<const uint4 *>(blocks + (h2 * 4 + c2) * kWarpOutBytes + (r - h2 * second0) * kWarpPitch +
                                                           (u - c2 * (kWarpPitch / 16)) * 16);
          multimem_st_v4(gout + (size_t)r * pitch + u * 16, v.x, v.y, v.z, v.w);
        }
      } else if (tp.store_mode == 1) {
        const int per_row = (int)(row_bytes >> 2);
        for (int q = tid; q < n_rows * per_row; q += kWorkerThreads) {
          const int r = q / per_row, u = q - r * per_row, h2 = r >= kWarpRows, c2 = u / (kWarpPitch / 4);
          *reinterpret_cast<uint32_t *>(gout + (size_t)r * pitch + u * 4) = *reinterpret_cast<const uint32_t *>(
              blocks + (h2 * 4 + c2) * kWarpOutBytes + (r - h2 * second0) * kWarpPitch + (u - c2 * (kWarpPitch / 4)) * 4);
        }
      } else {
        for (int q = tid; q < n_rows * (int)row_bytes; q += kWorkerThreads) {
          const int r = q / (int)row_bytes, u = q - r * (int)row_bytes, h2 = r >= kWarpRows, c2 = u / kWarpPitch;
          gout[(size_t)r * pitch + u] = blocks[(h2 * 4 + c2) * kWarpOutBytes + (r - h2 * second0) * kWarpPitch + (u - c2 * kWarpPitch)];
        }
      }
      // (the blocks of this stage are written again two tiles from now, behind the next tile's barrier)
    }
  }
  if (tp.store_mode == 2) bulk_wait_read_all();               // shared memory must outlive the last stores' reads
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
    (void)cudaGetLastError();
  }
  return fn;
}

// a uint8 image with 16-byte aligned rows as uint32 [rows][pitch / 4]
static bool encode_u32_rows(CUtensorMap *map, const void *base, size_t pitch, int rows, int box_bytes, int box_rows,
                            CUtensorMapL2promotion promo) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || rows <= 0) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)(pitch / 4), (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)pitch};
  const cuuint32_t box[2] = {(cuuint32_t)(box_bytes / 4), (cuuint32_t)box_rows};
  const cuuint32_t ones[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void *>(base), dims, strides, box, ones,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

size_t warp_tiles_bytes(int canvas_w, int n_blocks) {
  const long long tiles = (long long)((canvas_w + kTileCols - 1) / kTileCols) * ((n_blocks + kTileBlocks - 1) / kTileBlocks);
  return (size_t)tiles * sizeof(TileInfo);
}

static int tile_counts(const WarpParams &w, TileParams &tp) {
  tp.tiles_x = (w.canvas_w + kTileCols - 1) / kTileCols;
  const long long tiles_y = (w.n_blocks + kTileBlocks - 1) / kTileBlocks;
  if (tiles_y * tp.tiles_x > 2147483647LL) return fail(APAP_E_TOOBIG, "warp: too many tiles in one launch (split the band)");
  tp.n_tiles = (int)(tiles_y * tp.tiles_x);
  return 0;
}

// the tile records of a band (apap_warp_tiles); `w` needs the tables, the canvas and source geometry, no images
int launch_warp_tiles(const WarpParams &w, const int *col_ext, void *tiles, size_t tiles_bytes, cudaStream_t st) {
  TileParams tp;
  memset(&tp, 0, sizeof(tp));
  tp.w = w;
  tp.col_ext = reinterpret_cast<const int2 *>(col_ext);
  const int rc = tile_counts(w, tp);
  if (rc) return rc;
  if (tp.n_tiles == 0) return 0;
  if (!tiles || (reinterpret_cast<uintptr_t>(tiles) & 15u) || tiles_bytes < (size_t)tp.n_tiles * sizeof(TileInfo))
    return fail(APAP_E_BADARG, "warp tiles: buffer missing, not 16-byte aligned or smaller than apap_warp_tiles_bytes()");
  tp.tiles = static_cast<TileInfo *>(tiles);
  k_tile_prep<<<(tp.n_tiles + 7) / 8, 256, 0, st>>>(tp);
  return check_cuda(cudaGetLastError(), "k_tile_prep launch");
}

// can this source / band go through the tile engine?  (16-byte aligned source rows for the tensor maps)
bool warp_tile_usable(const WarpParams &w) {
  return ((size_t)w.src_w * 3) % 16 == 0 && !(reinterpret_cast<uintptr_t>(w.src) & 15u) && encode_tiled_fn() != nullptr;
}

int launch_warp_tile(const WarpParams &w, bool words, const void *tiles, cudaStream_t st) {
  TileParams tp;
  memset(&tp, 0, sizeof(tp));
  tp.w = w;
  const size_t src_pitch = (size_t)w.src_w * 3;
  for (int m = 0; m < kBoxShapes; ++m)                     // the source as uint32 [src_h][src_w * 3 / 4], three box shapes
    if (!encode_u32_rows(&tp.maps[m], w.src, src_pitch, w.src_h, box_w(m), box_h(m), CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
      return fail(APAP_E_BADARG, "warp: cuTensorMapEncodeTiled refused the source image");
  // the band as uint32 [band_rows][canvas_w * 3 / 4], box 16 rows x 96 B
  const bool rows16 = (w.canvas_w % 16 == 0) && !(reinterpret_cast<uintptr_t>(w.out) & 15u) && !w.multicast &&
                      encode_u32_rows(&tp.out_map, w.out, (size_t)w.canvas_w * 3, w.band_rows, kWarpPitch, kWarpRows,
                                      CU_TENSOR_MAP_L2_PROMOTION_NONE);
  tp.store_mode = w.multicast ? 3 : rows16 ? 2 : words ? 1 : 0;
  const int rc = tile_counts(w, tp);
  if (rc) return rc;
  tp.tiles = const_cast<TileInfo *>(static_cast<const TileInfo *>(tiles));
  static bool configured[64] = {};                         // > 48 KB of dynamic shared memory is opt-in, per device
  const size_t smem = sizeof(TileSmem);
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return check_cuda(e, "cudaGetDevice");
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    e = cudaFuncSetAttribute(k_warp_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return check_cuda(e, "k_warp_tile shared memory opt-in");
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  const int grid = min(tp.n_tiles, sm_count_cached() * kTileCtas);
  static std::atomic<unsigned> launch_seq{0};              // concurrent launches (other streams) get different counters
  tp.slot = (int)(launch_seq.fetch_add(1u) % kCounterSlots);
  k_warp_tile<<<grid, kTileThreads, smem, st>>>(tp);
  return check_cuda(cudaGetLastError(), "k_warp_tile launch");
}

}  // namespace apap
