// K3 -- mesh warp (reference APAP.local_warp pixel loop, pyviz/apap.py:206-215), optionally
// fused with K4, and K4 -- uniform_blend (pyviz/apap_utils.py:75-88).
//
// HBM-bound byte work: every canvas pixel is written once (3 B), every source pixel is read at
// most once from HBM.  The host cuts the canvas rows into "row blocks" of at most 4 rows that
// never cross a cell row.  A warp owns 32 consecutive canvas columns (lane = column) and walks a
// strip of consecutive row blocks downwards, so everything that depends on the column only -- the
// cell column, dx, the store lane pattern -- is loop invariant, and a lane needs one cell record
// per block (reloaded only when the strip enters a new cell row).  Per block, three phases:
//   1. source pixel index of the 4 rows on packed FP32x2 arithmetic (two rows per instruction),
//      straight-line; pixels inside the guard band are flagged and re-decided in float64 after it;
//   2. issue the 12 byte gathers of the lane (the 32 lanes of a row read ~96 contiguous source
//      bytes: 1-2 L1 wavefronts per byte plane);
//   3. combine, blend, re-pack the warp's 96 output bytes of a row into 24 aligned 32-bit stores
//      with two shuffles + one byte-permute.
// A warp visits two consecutive blocks at a time and finishes the first before it issues the second
// (both blocks' gathers in flight before the first store: the same plain, +13 % fused at c2 --
// profiles/r01_warp_variants.txt).
//
// Pixel selection must equal the reference's float64 arithmetic (float32 H^-1 promoted to
// float64, divide, strict bounds, truncate).  The float32 fast path works in cell-relative
// coordinates: the host rewrites each cell's H^-1 relative to the cell's first pixel (dx, dy
// small) and to an integer base (qbx, qby) near the cell's source position, and normalises the
// denominator to ~1, so numerators and quotient are O(cell size) instead of O(image size) and the
// float32 error is ~1e-5 px:   src_x = qbx + floor((A0 dx + B0 dy + C0) / (A2 dx + B2 dy + C2)).
// The host also supplies, per cell, a rigorous bound eps on that error.  A quotient farther than
// eps from every integer has the same floor and the same bounds decision in both arithmetics;
// the others (~1e-4 of the pixels) are recomputed in float64 exactly as the reference does.
#include "common.cuh"
#include "warp_common.cuh"

namespace apap {

constexpr int kWarpCtas = 4;     // resident CTAs per SM the kernel is compiled for: register cap 64 (3 CTAs, cap 85:
                                 // c2 36.9 against 32.8 us -- profiles/r01_warp_variants.txt)
constexpr int kWarpThreads = 256;
constexpr int kWarpsPerCta = kWarpThreads / 32;
// Phases 1 + 2 of one row block of one lane: the source pixel index of every row, then all byte
// gathers issued together.  kFull: the block has exactly kBlockRows rows (the host makes every
// block full unless its cell row has fewer canvas rows than that): straight-line code; the
// partial form predicates each row on n_rows.
template <bool kBlend, bool kFull>
__device__ __forceinline__ void block_issue(const WarpParams &p, const uint8_t *__restrict__ src, int i0, int n_rows,
                                            float dy0, int x, bool col_ok, const CellState &c,
                                            uint32_t (&b0)[kBlockRows], uint32_t (&b1)[kBlockRows],
                                            uint32_t (&b2)[kBlockRows], uint32_t (&c0)[kBlockRows],
                                            uint32_t (&c1)[kBlockRows], uint32_t (&c2)[kBlockRows]) {
  constexpr int P = kBlockRows;
  const int y0 = i0 - p.off_y;

  // ---- phase 1: source pixel index of every row (-1 = leave black) ---------------------------
  int idx[P];
  if (__all_sync(0xffffffffu, c.outside)) {
#pragma unroll
    for (int k = 0; k < P; ++k) idx[k] = -1;
  } else {
    const float2 km = make_float2(kMagic, kMagic), nkm = make_float2(-kMagic, -kMagic), nh = make_float2(-0.5f, -0.5f);
    unsigned flagged = 0;                           // rows whose quotient is inside the guard band
#pragma unroll
    for (int k = 0; k < P; k += 2) {
      // two rows at once on packed FP32x2 arithmetic (identical roundings to the scalar form)
      const float2 dy = make_float2(dy0 + (float)k, dy0 + (float)(k + 1));
      const float2 n0 = __ffma2_rn(make_float2(c.b0, c.b0), dy, make_float2(c.m0, c.m0));
      const float2 n1 = __ffma2_rn(make_float2(c.b1, c.b1), dy, make_float2(c.m1, c.m1));
      const float2 d = __ffma2_rn(make_float2(c.b2, c.b2), dy, make_float2(c.m2, c.m2));
      const float2 r = make_float2(rcp_approx(d.x), rcp_approx(d.y));
      const float2 qx = __fmul2_rn(n0, r), qy = __fmul2_rn(n1, r);
      const float2 tx = __fadd2_rd(qx, km), ty = __fadd2_rd(qy, km);             // floor + kMagic
      const float2 gx = __fadd2_rn(tx, nkm), gy = __fadd2_rn(ty, nkm);           // floor
      const float2 fx = __fadd2_rn(qx, make_float2(-gx.x, -gx.y));               // exact fraction in [0, 1)
      const float2 fy = __fadd2_rn(qy, make_float2(-gy.x, -gy.y));
      const float2 hx = __fadd2_rn(fx, nh), hy = __fadd2_rn(fy, nh);
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float txe = e ? tx.y : tx.x, tye = e ? ty.y : ty.x;
        const float hxe = e ? hx.y : hx.x, hye = e ? hy.y : hy.x;
        const bool clear = fmaxf(fabsf(hxe), fabsf(hye)) <= c.hme;
        const int ix = __float_as_int(txe) + c.qbx;
        const int iy = __float_as_int(tye) + c.qby;
        const bool inb = ((unsigned)ix < (unsigned)p.src_w) & ((unsigned)iy < (unsigned)p.src_h);
        idx[k + e] = (inb && !c.outside) ? iy * p.src_w + ix : -1;
        if (!clear && !c.outside) flagged |= 1u << (k + e);
      }
    }
    if (!kFull) flagged &= (1u << n_rows) - 1u;
    if (__any_sync(0xffffffffu, flagged != 0)) {    // rare: re-decide the flagged pixels in float64
      const float *h = p.cell_hinv + (size_t)c.cell * 9;
#pragma unroll
      for (int k = 0; k < P; ++k)
        if (flagged & (1u << k)) idx[k] = exact_lookup(h, x, y0 + k, p.src_w, p.src_h);
    }
  }

  // ---- phase 2: every byte load of the block in flight together -------------------------------
#pragma unroll
  for (int k = 0; k < P; ++k) {
    b0[k] = b1[k] = b2[k] = 0;
    if (idx[k] >= 0 && (kFull || k < n_rows)) {
      const uint8_t *q = src + (size_t)(unsigned)idx[k] * 3;
      b0[k] = __ldg(q); b1[k] = __ldg(q + 1); b2[k] = __ldg(q + 2);
    }
  }
  if (kBlend) {
    // centre image pasted at (off_x, off_y) (pyviz/apap.py:259-260)
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const int cy = y0 + k;
      c0[k] = c1[k] = c2[k] = 0;
      if ((kFull || k < n_rows) && (unsigned)cy < (unsigned)p.centre_h && (unsigned)x < (unsigned)p.centre_w && col_ok) {
        const uint8_t *q = p.centre + ((size_t)cy * p.centre_w + x) * 3;
        c0[k] = __ldg(q); c1[k] = __ldg(q + 1); c2[k] = __ldg(q + 2);
      }
    }
  }
}

// Phase 3 of one row block: combine, blend, re-pack across the warp, store.
// kWords: the band's rows are 4-byte aligned (canvas_w % 4 == 0): the warp's 32 pixels of a row
// leave as 24 packed 32-bit stores; otherwise three byte stores per lane.
template <bool kBlend, bool kWords, bool kFull>
__device__ __forceinline__ void block_store(const WarpParams &p, int i0, int n_rows, const uint32_t (&b0)[kBlockRows],
                                            const uint32_t (&b1)[kBlockRows], const uint32_t (&b2)[kBlockRows],
                                            const uint32_t (&c0)[kBlockRows], const uint32_t (&c1)[kBlockRows],
                                            const uint32_t (&c2)[kBlockRows], uint32_t lane_off, uint32_t pitch,
                                            int lane_a, int lane_b, uint32_t sel, int n_store) {
  // n_store: 32-bit words this warp writes per row (kWords), or 1 / 0 for a valid / invalid column (byte stores)
  const bool store_ok = (int)(threadIdx.x & 31) < n_store || (!kWords && n_store > 0);
  uint8_t *d = p.out + ((uint32_t)(i0 - p.row0) * pitch + lane_off);   // the band is < 2^31 bytes (launch_warp)
#pragma unroll
  for (int k = 0; k < kBlockRows; ++k) {
    if (kFull || k < n_rows) {                     // warp-uniform
      uint32_t val = __byte_perm(__byte_perm(b0[k], b1[k], 0x1140), b2[k], 0x3410);   // b0 | b1<<8 | b2<<16
      if (kBlend) {                                // uniform_blend (pyviz/apap_utils.py:75-88)
        const uint32_t cv = __byte_perm(__byte_perm(c0[k], c1[k], 0x1140), c2[k], 0x3410);
        if (cv != 0) val = (val != 0) ? __vhaddu4(val, cv) : cv;
      }
      if (kWords) {
        const uint32_t va = __shfl_sync(0xffffffffu, val, lane_a);
        const uint32_t vb = __shfl_sync(0xffffffffu, val, lane_b);
        const uint32_t word = __byte_perm(va, vb, sel);
        if (p.multicast) {                         // warp-uniform
          // NVLS stores, 16 bytes each (4-byte packets waste the links): lane l < 6 collects the words 4l .. 4l+3 of
          // the row's 24 and stores them with one multimem.st.v4 (launch_warp checks canvas_w % 16 == 0, so a row
          // segment is a whole number of 16-byte groups, 16-byte aligned)
          const int lane = threadIdx.x & 31, l4 = (lane << 2) & 31;
          const uint32_t w0 = __shfl_sync(0xffffffffu, word, l4), w1 = __shfl_sync(0xffffffffu, word, l4 + 1);
          const uint32_t w2 = __shfl_sync(0xffffffffu, word, l4 + 2), w3 = __shfl_sync(0xffffffffu, word, l4 + 3);
          if (4 * lane + 3 < n_store) multimem_st_v4(d + 12 * lane, w0, w1, w2, w3);   // d + 12 lane = row segment + 16 lane
        } else if (store_ok) {
          *reinterpret_cast<uint32_t *>(d) = word;
        }
      } else if (store_ok) {
        d[0] = (uint8_t)val;
        d[1] = (uint8_t)(val >> 8);
        d[2] = (uint8_t)(val >> 16);
      }
      d += pitch;
    }
  }
}

__device__ __forceinline__ void prefetch_l1(const void *ptr) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr));
}

// grid.x = groups of 8 column chunks (one per warp of the CTA), grid.y = S "lanes" of strips: the
// warp (chunk, s) visits the block pairs s, s + S, s + 2S, ... of the band, so every warp samples
// the whole height of the canvas (mapped and unmapped regions alike -> even load) while its
// column state stays loop invariant.  The cell record of the next visit is prefetched into L1
// while the current visit's gathers are in flight.
template <bool kBlend, bool kWords>
__global__ void __launch_bounds__(kWarpThreads, kWarpCtas) k_warp(const WarpParams p) {
  const int lane = threadIdx.x & 31;
  const int chunk = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (chunk >= p.chunks_per_row) return;           // warp-uniform
  const int j0 = chunk * 32;

  // column-only state: loop invariant
  const int j = j0 + lane;
  const bool col_ok = j < p.canvas_w;
  const uint2 cl = __ldg(p.col_lut + (col_ok ? j : p.canvas_w - 1));
  const float dxf = __uint_as_float(cl.y);
  const int x = j - p.off_x;
  const uint8_t *__restrict__ src = p.src;
  // kWords: output word w = lane (< 24) takes its 4 bytes from the pixels of lanes lane_a = (4w)/3
  // and lane_a + 1, starting at byte (4w) % 3 of the first
  const int lane_a = (lane + lane / 3) & 31, lane_b = (lane_a + 1) & 31;
  const uint32_t sel = (lane % 3 == 0) ? 0x4210u : (lane % 3 == 1) ? 0x5421u : 0x6542u;
  const int store_ok = kWords ? min(24, (3 * (p.canvas_w - j0)) >> 2) : (col_ok ? 1 : 0);   // words per row / column valid
  const uint32_t pitch = (uint32_t)p.canvas_w * 3u;
  const uint32_t lane_off = (uint32_t)j0 * 3u + (kWords ? 4u : 3u) * lane;

  CellState c;
  c.b0 = c.b1 = c.b2 = c.m0 = c.m1 = 0.f; c.m2 = 1.f; c.hme = -1.f;
  c.qbx = c.qby = 0; c.cell_row = -1; c.cell = 0; c.outside = false;

  const int stride = gridDim.y * 2;
  int t = blockIdx.y * 2;
  if (t >= p.n_blocks) return;
  uint2 nxt0 = __ldg(p.row_blocks + t), nxt1 = __ldg(p.row_blocks + min(t + 1, p.n_blocks - 1));
  for (; t < p.n_blocks; t += stride) {
    const uint2 cur0 = nxt0, cur1 = nxt1;
    if (t + stride < p.n_blocks) {                 // the next visit's entries: in flight during this one
      nxt0 = __ldg(p.row_blocks + t + stride);
      nxt1 = __ldg(p.row_blocks + min(t + stride + 1, p.n_blocks - 1));
    }
    const int i0a = (int)(cur0.x & 0x0fffffffu), na = (int)(cur0.x >> 28);
    const int i0b = (int)(cur1.x & 0x0fffffffu), nb = (t + 1 < p.n_blocks) ? (int)(cur1.x >> 28) : 0;
    uint32_t a0[kBlockRows], a1[kBlockRows], a2[kBlockRows], ca0[kBlockRows], ca1[kBlockRows], ca2[kBlockRows];
    if (na == kBlockRows && nb == kBlockRows) {    // warp-uniform: the hot, straight-line path
      enter_cell_row(p, cl, dxf, (int)(cur0.y & 0xffffu), c);
      block_issue<kBlend, true>(p, src, i0a, na, (float)(cur0.y >> 16), x, col_ok, c, a0, a1, a2, ca0, ca1, ca2);
      // the record the next visit starts with: into L1 while this visit's gathers are in flight
      if (t + stride < p.n_blocks) {
        const char *rec = reinterpret_cast<const char *>(p.cell_fast) +
                          ((size_t)((int)(nxt0.y & 0xffffu) * p.grid_cols + (int)cl.x)) * 48;
        prefetch_l1(rec);
        prefetch_l1(rec + 32);
      }
      block_store<kBlend, kWords, true>(p, i0a, na, a0, a1, a2, ca0, ca1, ca2, lane_off, pitch, lane_a, lane_b, sel, store_ok);
      enter_cell_row(p, cl, dxf, (int)(cur1.y & 0xffffu), c);
      block_issue<kBlend, true>(p, src, i0b, nb, (float)(cur1.y >> 16), x, col_ok, c, a0, a1, a2, ca0, ca1, ca2);
      block_store<kBlend, kWords, true>(p, i0b, nb, a0, a1, a2, ca0, ca1, ca2, lane_off, pitch, lane_a, lane_b, sel, store_ok);
    } else {                                       // partial blocks (cell rows shorter than 4 canvas rows, band end)
      enter_cell_row(p, cl, dxf, (int)(cur0.y & 0xffffu), c);
      block_issue<kBlend, false>(p, src, i0a, na, (float)(cur0.y >> 16), x, col_ok, c, a0, a1, a2, ca0, ca1, ca2);
      block_store<kBlend, kWords, false>(p, i0a, na, a0, a1, a2, ca0, ca1, ca2, lane_off, pitch, lane_a, lane_b, sel, store_ok);
      if (nb > 0) {
        enter_cell_row(p, cl, dxf, (int)(cur1.y & 0xffffu), c);
        block_issue<kBlend, false>(p, src, i0b, nb, (float)(cur1.y >> 16), x, col_ok, c, a0, a1, a2, ca0, ca1, ca2);
        block_store<kBlend, kWords, false>(p, i0b, nb, a0, a1, a2, ca0, ca1, ca2, lane_off, pitch, lane_a, lane_b, sel, store_ok);
      }
    }
  }
}

// ------------------------------------------------------------------------------------ K4 blend
// 16 pixels = 48 B = three 16-byte vectors per thread and per image.
constexpr int kBlendThreads = 256;

// Four pixels = 12 bytes = three words (w0, w1, w2).  One byte per pixel: the OR of its three channel bytes.
__device__ __forceinline__ uint32_t pixel_or4(uint32_t w0, uint32_t w1, uint32_t w2) {
  const uint32_t x = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);   // bytes 0, 3, 6, 9
  const uint32_t y = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);   // bytes 1, 4, 7, 10
  const uint32_t z = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);   // bytes 2, 5, 8, 11
  return x | y | z;
}
// msb of every byte = that byte of v is non-zero (the other bits are junk)
__device__ __forceinline__ uint32_t byte_nonzero_msb(uint32_t v) { return ((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v; }
// prmt.b32 with sign replication: selector nibble 8 + i gives 0xff / 0x00 from the msb of byte i
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %1, %2;" : "=r"(d) : "r"(a), "r"(sel));
  return d;
}

// uniform_blend of 16 pixels = 12 words per image, all in 32-bit SIMD, four pixels = three words at a time.
__device__ __forceinline__ void blend16(const uint32_t (&wa)[12], const uint32_t (&wb)[12], uint32_t (&wo)[12]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const uint32_t *pa = wa + 3 * g, *pb = wb + 3 * g;
    // one flag per pixel: non-black in BOTH images
    const uint32_t both = byte_nonzero_msb(pixel_or4(pa[0], pa[1], pa[2])) &
                          byte_nonzero_msb(pixel_or4(pb[0], pb[1], pb[2]));       // msb of byte k: pixel k
    const uint32_t m[3] = {prmt(both, 0x9888), prmt(both, 0xaa99), prmt(both, 0xbbba)};   // 0xff per byte of a flagged pixel
#pragma unroll
    for (int w = 0; w < 3; ++w) {
      const uint32_t x = pa[w], y = pb[w];
      const uint32_t avg = (x & y) + (((x ^ y) & 0xfefefefeu) >> 1);   // per-byte (a + b) >> 1
      wo[3 * g + w] = (avg & m[w]) | ((x | y) & ~m[w]);                 // else a + b, one of them being 0
    }
  }
}

// the last n_px % 16 pixels, one thread
__device__ __forceinline__ void blend_tail(const uint8_t *__restrict__ a8, const uint8_t *__restrict__ b8,
                                           uint8_t *__restrict__ out8, long long px0, long long n_px) {
  for (long long px = px0; px < n_px; ++px) {
    const uint8_t *pa = a8 + px * 3, *pb = b8 + px * 3;
    const bool both = (pa[0] | pa[1] | pa[2]) && (pb[0] | pb[1] | pb[2]);
    for (int c = 0; c < 3; ++c) {
      const unsigned s = (unsigned)pa[c] + pb[c];
      out8[px * 3 + c] = (uint8_t)(both ? (s >> 1) : s);
    }
  }
}

// CTA = 256 units of 16 pixels = 12 KB per image.  One thread moves the CTA's slice of both images into shared memory
// with two TMA bulk copies and the result back with one (whole 128-byte lines on the wire, no per-thread address
// arithmetic); the threads read their 48 bytes as three LDS.128 (stride 48 B: conflict-free per quarter warp) and
// write the result over their own slice of `a`.
struct BlendSmem {
  uint4 a[kBlendThreads * 3];
  uint4 b[kBlendThreads * 3];
  uint64_t bar;
};

__global__ void __launch_bounds__(kBlendThreads) k_blend(const uint8_t *__restrict__ a8, const uint8_t *__restrict__ b8,
                                                          uint8_t *__restrict__ out8, long long n_vec3, long long n_px) {
  __shared__ __align__(128) BlendSmem sm;
  const long long unit0 = (long long)blockIdx.x * kBlendThreads;
  const long long left = n_vec3 - unit0;
  const int units = left >= kBlendThreads ? kBlendThreads : (left > 0 ? (int)left : 0);
  const uint32_t bytes = (uint32_t)units * 48u;
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(&sm.bar, 1);
    mbar_fence_init();
    if (units > 0) {
      mbar_arrive_expect_tx(&sm.bar, 2 * bytes);
      bulk_g2s(sm.a, a8 + unit0 * 48, bytes, &sm.bar);
      bulk_g2s(sm.b, b8 + unit0 * 48, bytes, &sm.bar);
    }
  }
  __syncthreads();
  if (units > 0) mbar_wait(&sm.bar, 0);
  if (tid < units) {
    uint32_t wa[12], wb[12], wo[12];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const uint4 x = sm.a[tid * 3 + v], y = sm.b[tid * 3 + v];
      wa[4 * v + 0] = x.x; wa[4 * v + 1] = x.y; wa[4 * v + 2] = x.z; wa[4 * v + 3] = x.w;
      wb[4 * v + 0] = y.x; wb[4 * v + 1] = y.y; wb[4 * v + 2] = y.z; wb[4 * v + 3] = y.w;
    }
    blend16(wa, wb, wo);
#pragma unroll
    for (int v = 0; v < 3; ++v) sm.a[tid * 3 + v] = make_uint4(wo[4 * v], wo[4 * v + 1], wo[4 * v + 2], wo[4 * v + 3]);
    fence_proxy_async_smem();
  } else if (tid == units) {
    if (left < kBlendThreads) blend_tail(a8, b8, out8, n_vec3 * 16, n_px);     // only in the CTA that holds the end
  }
  __syncthreads();
  if (tid == 0 && units > 0) {
    bulk_s2g(out8 + unit0 * 48, sm.a, bytes);
    bulk_commit_wait_read();
  }
}

int launch_warp(const uint8_t *src, int src_h, int src_w, const float *cell_fast, const float *cell_hinv,
                const uint32_t *col_lut, const uint32_t *row_blocks, int n_blocks, int grid_cols, int canvas_w, int off_x,
                int off_y, int row0, int row1, const uint8_t *centre, int centre_h, int centre_w, uint8_t *out_band,
                size_t out_band_bytes, int flags, int multicast, const void *tiles, cudaStream_t st) {
  const int force_exact = (flags & APAP_WARP_FORCE_EXACT) ? 1 : 0;
  if ((long long)src_w * src_h > 2147483647LL)
    return fail(APAP_E_TOOBIG, "warp: source image has more than 2^31-1 pixels");
  if ((reinterpret_cast<uintptr_t>(cell_fast) & 15u) || (reinterpret_cast<uintptr_t>(col_lut) & 7u) ||
      (reinterpret_cast<uintptr_t>(row_blocks) & 7u))
    return fail(APAP_E_ALIGN, "warp: cell_fast must be 16-byte, col_lut / row_blocks 8-byte aligned");
  if (n_blocks == 0) return 0;
  if (out_band_bytes > 2147483647ULL) return fail(APAP_E_TOOBIG, "warp: row band larger than 2 GiB (split it)");
  WarpParams p;
  p.src = src; p.cell_fast = reinterpret_cast<const float4 *>(cell_fast); p.cell_hinv = cell_hinv;
  p.col_lut = reinterpret_cast<const uint2 *>(col_lut); p.row_blocks = reinterpret_cast<const uint2 *>(row_blocks);
  p.centre = centre; p.out = out_band;
  p.row0 = row0;
  p.band_rows = row1 - row0;
  p.n_blocks = n_blocks;
  p.chunks_per_row = (canvas_w + 31) / 32;
  p.src_h = src_h; p.src_w = src_w; p.grid_cols = grid_cols; p.canvas_w = canvas_w;
  p.off_x = off_x; p.off_y = off_y; p.centre_h = centre_h; p.centre_w = centre_w; p.force_exact = force_exact;
  p.multicast = multicast;
  const bool words = (canvas_w % 4 == 0) && !(reinterpret_cast<uintptr_t>(out_band) & 3u);
  if (multicast && (!words || canvas_w % 16 != 0 || (reinterpret_cast<uintptr_t>(out_band) & 15u)))
    return fail(APAP_E_ALIGN, "warp: multicast stores need canvas_w % 16 == 0 and a 16-byte aligned band");
  // the tile engine (csrc/warp_tile.cu) for the plain warp when the caller built tile records and the source rows are
  // 16-byte aligned.  Fused with the blend, the warp runs on the strip kernel: its batched centre loads are faster than
  // centre gathers inside the tile loop (c2 49 us against 65 us, c3 169 against 198)
  if (tiles && !centre && !(flags & APAP_WARP_LEGACY) && warp_tile_usable(p)) {
    if (reinterpret_cast<uintptr_t>(tiles) & 15u) return fail(APAP_E_ALIGN, "warp: tiles must be 16-byte aligned");
    return launch_warp_tile(p, words, tiles, st);
  }
  // legacy strip kernel.  One resident wave: grid.x CTAs side by side cover the canvas width, grid.y of them share its height
  const int gx = (p.chunks_per_row + kWarpsPerCta - 1) / kWarpsPerCta;
  const int visits = (n_blocks + 1) / 2;           // a visit = two consecutive row blocks
  int gy = (sm_count_cached() * kWarpCtas) / gx;   // kWarpCtas CTAs of 8 warps resident per SM (launch bounds)
  if (gy < 1) gy = 1;
  if (gy > visits) gy = visits;
  if (gy > 65535) gy = 65535;
  const dim3 grid(gx, gy);
  if (centre) {
    if (words) k_warp<true, true><<<grid, kWarpThreads, 0, st>>>(p);
    else k_warp<true, false><<<grid, kWarpThreads, 0, st>>>(p);
  } else {
    if (words) k_warp<false, true><<<grid, kWarpThreads, 0, st>>>(p);
    else k_warp<false, false><<<grid, kWarpThreads, 0, st>>>(p);
  }
  return check_cuda(cudaGetLastError(), "k_warp launch");
}

int launch_blend(const uint8_t *a, const uint8_t *b, uint8_t *out, size_t n_px, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out)) & 15u)
    return fail(APAP_E_ALIGN, "blend: pointers must be 16-byte aligned");
  if (n_px == 0) return 0;
  const long long n_vec3 = (long long)(n_px / 16);
  const long long threads = n_vec3 + 1;   // +1 thread for the tail
  const long long blocks = (threads + kBlendThreads - 1) / kBlendThreads;
  if (blocks > 2147483647LL) return fail(APAP_E_TOOBIG, "blend: image too large");
  k_blend<<<(unsigned)blocks, kBlendThreads, 0, st>>>(a, b, out, n_vec3, (long long)n_px);
  return check_cuda(cudaGetLastError(), "k_blend launch");
}

}  // namespace apap
