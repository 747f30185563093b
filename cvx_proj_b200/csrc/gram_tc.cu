// K1 on the tensor cores -- moving-DLT weights + Gram contraction (reference pyviz/apap.py:150-152,159)
// as tcgen05 (5th-generation tensor core) MMAs with the accumulators in tensor memory.
//
// The contraction  S_t(c) = sum_i w2(c, i) * P[i][t]  is a GEMM  [cells x N] . [N x 24]  whose A
// operand does not exist in memory: it is generated on the fly.  Per CTA (one 128-cell tile x one
// keypoint split; 10 warps, 3 CTAs resident per SM):
//   * warps 0-7 (producers; thread = cell = accumulator row = TMEM lane; warp w serves the lane
//     quarter w & 3, and the two warps of a quarter take alternate 16-keypoint steps, h = w >> 2)
//     compute the weights  w2 = max(2^-|s v - s x|, gamma^2)  of their step (packed FP32x2 adds / FMA,
//     MUFU.SQRT, then MUFU.EX2 for half of them and a degree-7 polynomial on the FMA pipe for the other
//     half -- see kPoly), split each into a TF32 head and tail (hi = w2 with the low 13 mantissa
//     bits cleared, lo = w2 - hi, exact) and store both straight into tensor memory (tcgen05.st, SASS
//     STTM) -- the A operand of the MMA is read from TMEM, so the weights never touch shared memory;
//   * warp 8 (one elected thread) issues, per 8-keypoint block, two TF32 MMAs (SASS UTCHMMA):
//     M128 x N64 x K8:  [D1 | D2] += hi . [Ph | Pl]   and   M128 x N32 x K8:  D2 += lo . Ph
//     (3xTF32: the product terms P are split into Ph + Pl on the host; the dropped lo . Pl term is
//     2^-22 relative).  The two cross terms accumulate in their own TMEM columns D2, so they never
//     re-round the big sums D1;
//   * warp 9 (one thread) streams the keypoint blocks -- the 64 x 8 tile [Ph | Pl] in the K-major
//     core-matrix layout of the MMA's shared-memory descriptor, and the 8 pre-scaled keypoint
//     coordinates -- by TMA bulk copies (cp.async.bulk + mbarrier, SASS UBLKCP) into a 4-stage ring;
//   * mbarriers connect the three roles: smem_full/smem_empty (TMA <-> producers + MMA),
//     a_full/a_empty (producers <-> MMA: two A slots in TMEM, slot h owned by the warps of parity h),
//     d_full/d_empty (segment drains).
//
// What bounds it (in-kernel trace of the lab build, profiles/r01_gram_tc_trace.txt).  2 MUFU per weight at
// 16 lanes/clk/SM make the XU pipe the bound; a warp issues the MUFU of its step in order (8 cycles of XU
// time each) and then spends ~600 cycles on work the XU does not see (split, STTM, tcgen05.wait::st,
// fences, mbarrier round trips of ~90 cycles each), while the rest of the step needs ~60 % of the issue
// slots of its scheduler -- XU, issue and latency are co-limiting and the XU ends up 65-80 % busy at the
// clock the SM really runs this kernel at (1.76 GHz by %globaltimer, not the 1.965 GHz nvidia-smi shows).
// Same-box A/B timings (profiles/r01_gram_variants.txt): two producer warps per lane quarter (3 CTAs x 8
// instead of 4 CTAs x 4) -3.5 %, the slot probe (mbarrier.test_wait) issued before the step's arithmetic
// and consumed after it -1 %, half of the 2^-t on the FMA pipe -4..6 %, truncating split instead of a
// rounding one -5 %; the depth of the A ring, of the shared-memory ring and the TMA latency do not matter.
// Round 2 (profiles/r02_gram_variants.txt; c2, same box per comparison): the kernel answers to its instruction count --
// a step of 16 keypoints was ~180 instructions per producer warp for 24 MUFU, and every 16 instructions taken out are
// ~4 % of the time.  The clamp dropped where apap_weight_bound proves it a no-op (-16 instructions, 139 -> 131 us), ring
// addresses as shared-window constants and one 16-column tcgen05.st per k-block (-9, -> 127 us), the producer loop
// unrolled 8x so that ring position and slot phase are immediates (-12, -> 125 us); the polynomial share stays at 2 of 4
// (1 of 4 and 3 of 4: +3 %); the MMA warp's own instruction count does not matter (-35 % of it: no change), nor does the
// number of keypoint splits (4 .. 8 at c2: 125 .. 127 us).  What is left between c2 (0.70 of the XU roofline) and c3
// (0.83, 28 waves): 1252 CTAs over 444 slots leave some SMs a ninth CTA while others have done their eight, and the last
// CTAs of an SM run alone at about half the rate of three.  Persistent CTAs would fix both but hold all the registers of
// the SM to the end, so K2 could no longer move in beside K1's last CTAs (its 9 us exposed tail would become 16).
//
// Accuracy.  The tensor core accumulates in FP32 and aligns/truncates the accumulator at every
// MMA, a drift proportional to the number of MMAs that touch a big accumulator.  So (a) only one
// MMA per keypoint block touches D1, and (b) every 256 keypoints (kSegKb blocks) the producers
// drain D1 + D2 from TMEM (tcgen05.ld, SASS LDTM) into FP32 sums in shared memory and the MMAs
// restart from zero; the per-split sums (<= 1024 keypoints, like the FFMA2 kernel) are written as
// the same partial-sum layout and combined in float64 by K2.  Measured against the float64 reference of
// tests/test_gram_reference.py, per partial entry and split, relative to its scale A = sum |w2 P_t| (B200, 1000 W,
// over every case there): 2.8e-7 mean / 2.9e-6 max (the FFMA2 kernel: 8.7e-8 mean / 1.0e-5 max), at most 0.18 of
// the test's bound (256 + 2 ln2 t) 2^-24 A.
#include <type_traits>

#include "common.cuh"

namespace apap {

// lab knobs (tools/variants.sh builds the library with -D...; the defaults are the product)
#ifndef APAP_TC_NOMUFU
#define APAP_TC_NOMUFU 0         // 1: diagnostic, weights without the two MUFU operations (wrong results)
#endif
#ifndef APAP_TC_SMEM_STAGES
#define APAP_TC_SMEM_STAGES 4
#endif
#ifndef APAP_TC_POLY
#define APAP_TC_POLY 2           // weight pairs per k-block (of 4) whose 2^-t runs on the FMA pipe when gamma^2 >= 1/4
#endif
#ifndef APAP_TC_UNROLL
#define APAP_TC_UNROLL 8          // producer loop unrolled over the ring positions and slot phases: addresses and parities are immediates (1: 131 us, 4: 128, 8: 125, 16: 126 at c2)
#endif
#ifndef APAP_TC_EARLY_PROBE
#define APAP_TC_EARLY_PROBE 1    // 0: wait for the A slot before the step's arithmetic (A/B timing)
#endif

constexpr int kKB = APAP_KP_BLOCK;                 // keypoints per k-block = K of one TF32 MMA
constexpr int kNT = 32;                            // accumulator columns (24 terms padded to the MMA N)
constexpr int kKbFloats = APAP_KP_BLOCK_FLOATS;    // [Ph | Pl] tile 512, s*kx[8], s*ky[8]
constexpr int kKbBytes = kKbFloats * 4;            // 2112
constexpr int kStepKb = 2;                         // k-blocks per producer/MMA hand-over ("step" = 16 keypoints)
constexpr int kStageKb = 4;                        // k-blocks per shared-memory stage (2 steps: one per producer parity)
constexpr int kStageBytesTc = kStageKb * kKbBytes; // 8448
constexpr int kSmemStages = APAP_TC_SMEM_STAGES;
constexpr int kUnroll = APAP_TC_UNROLL;
constexpr int kSlots = 2;                          // A slots in TMEM: slot h = steps of parity h, 2 k-blocks x (8 hi + 8 lo columns)
constexpr int kTmemCols = 128;                     // 32 (D1) + 32 (D2) + 2 * 32 (A)
constexpr int kSegKb = 32;                         // k-blocks per accumulation segment (256 keypoints)
constexpr int kSegSteps = kSegKb / kStepKb;
#ifndef APAP_TC_PARITIES
#define APAP_TC_PARITIES 2       // producer warps per lane quarter (1: 4 CTAs x 6 warps per SM, 2: 3 CTAs x 10 warps)
#endif
constexpr int kParities = APAP_TC_PARITIES;        // warps of a lane quarter take the steps s = h (mod kParities)
constexpr int kProducerWarps = 4 * kParities;
constexpr int kMmaWarp = kProducerWarps, kTmaWarp = kProducerWarps + 1;
constexpr int kTcThreads = (kProducerWarps + 2) * 32;
constexpr int kTcCtasPerSm = kParities == 1 ? 4 : 3;
static_assert(kParities == 2 && kParities == kSlots, "two producer warps per lane quarter, each with its own A slot");
static_assert((kSmemStages & (kSmemStages - 1)) == 0, "the ring position is a mask of the stage index");
static_assert(kKbFloats == 2 * kNT * kKB + 2 * kKB, "k-block layout");
static_assert((kChunk / kKB) % kStageKb == 0, "a split is a whole number of stages");
static_assert(kStageKb / kStepKb == kSlots && kSlots == 2, "one step per producer parity in a stage");

// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// non-blocking probe of a phase (the blocking form is mbar_try_wait)
__device__ __forceinline__ uint32_t mbar_test(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// the same on shared-window addresses (the producers' loop keeps them in registers)
__device__ __forceinline__ uint32_t mbar_test_at(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait_at(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_arrive_at(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(
          taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem descriptor], kind::tf32, M = 128, issued by one thread
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive when every MMA issued so far by this thread has retired (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// One lane of a converged warp: with elect.sync the compiler issues the single-thread tcgen05 instructions
// straight-line (behind `if (lane == 0)` it wraps every one of them in an ELECT loop).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// TF32 head of a positive finite float: the low 13 mantissa bits cleared (what the tensor core reads of
// it anyway); w - head is exact and has at most 13 significant bits.
__device__ __forceinline__ uint32_t tf32_head(float x) { return __float_as_uint(x) & 0xFFFFE000u; }
// Instruction descriptor: D = F32 (bit 4), A = B = TF32 (2 at bits 7 and 10), both K-major, N >> 3 at bit 17,
// M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// ------------------------------------------------------------------------------------------ lab trace
#ifdef APAP_TC_TRACE
__device__ long long g_trace[4][160][4];           // [role][step][mark] SM clock of CTA (APAP_TC_TRACE, 0, 0)
__device__ long long g_cta[8192][4];               // per CTA: SM id, globaltimer at entry, after the TMEM allocation, at exit
__device__ __forceinline__ long long gtimer() { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define TRACE(role, step, mark) do { if (blockIdx.y == APAP_TC_TRACE && blockIdx.x == 0 && (step) < 160) g_trace[role][step][mark] = clock64(); } while (0)
#else
#define TRACE(role, step, mark) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------ kernel
struct TcSmem {
  alignas(128) float stage[kSmemStages][kStageBytesTc / 4];
  float acc[kTerms][128];               // per-split sums of the producers' drains (thread = column: conflict-free)
  uint64_t smem_full[kSmemStages];      // TMA -> producers + MMA
  uint64_t smem_empty[kSmemStages];     // MMA (commit) -> TMA
  uint64_t a_full[kSlots];              // producers -> MMA (one arrival per producer warp of the slot's parity)
  uint64_t a_empty[kSlots];             // MMA (commit) -> producers
  uint64_t d_full;                      // MMA (commit) -> producers: a segment's sums are complete
  uint64_t d_empty;                     // producers -> MMA: the accumulators have been drained
  uint32_t tmem_base;
};
static_assert(sizeof(TcSmem) * kTcCtasPerSm <= 220 * 1024 && sizeof(TcSmem) <= 48 * 1024,
              "the resident CTAs fit the shared memory of an SM, one CTA the default dynamic limit");

// kPoly: weight pairs per k-block (of 4) that evaluate 2^-t with a polynomial on the FMA pipe instead of
// MUFU.EX2 -- the XU pipe is the kernel's bound and the FMA pipe has room.  The polynomial covers
// t in [0, 2], i.e. clamps gamma^2 >= 1/4 (the reference's gamma = 0.5, pyviz/apap.py:222); the launcher
// picks kPoly = 0 for smaller clamps.
template <int kPoly>
__global__ void __launch_bounds__(kTcThreads, kTcCtasPerSm) k_gram_tc(const float *__restrict__ kp_blocks,
                                                                      const float *__restrict__ anchors, int cells,
                                                                      int cells_padded, int n_kb, int kb_per_split,
                                                                      int k_splits, float gamma_sq,
                                                                      const float *__restrict__ t_bound,
                                                                      float *__restrict__ partials,
                                                                      int *__restrict__ tile_done) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  TcSmem &sm = *reinterpret_cast<TcSmem *>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // grid: x = split (fastest, so the CTAs of a tile run together and tiles complete progressively -- K2 can
  // start on finished tiles while the last CTAs of K1 are still running), y = cell tile, z = scene
  const int split = blockIdx.x, tile = blockIdx.y, scene = blockIdx.z;
  // programmatic dependent launch: the next kernel in the stream (K2, when launched for overlap) may be
  // scheduled once every CTA of this grid has got this far; it synchronises on tile_done, not on grid completion
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int kb0 = split * kb_per_split;
  const int nkb = min(n_kb, kb0 + kb_per_split) - kb0;            // k-blocks of this CTA: a multiple of kStageKb
  const int n_stage = nkb / kStageKb;
  const int n_step = nkb / kStepKb;                               // even
  const int n_seg = (n_step + kSegSteps - 1) / kSegSteps;
  kp_blocks += (size_t)scene * n_kb * kKbFloats;
  anchors += (size_t)scene * cells * 2;
  partials += (size_t)scene * k_splits * kTerms * cells_padded;

#ifdef APAP_TC_TRACE
  const int cta_lin = blockIdx.y * gridDim.x + blockIdx.x;   // launch order
  if (tid == 0 && cta_lin < 8192) {
    uint32_t smid; asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
    g_cta[cta_lin][0] = smid; g_cta[cta_lin][1] = gtimer();
  }
#endif
  if (tid == 0) {
    for (int s = 0; s < kSmemStages; ++s) { mbar_init(&sm.smem_full[s], 1); mbar_init(&sm.smem_empty[s], 1); }
    for (int s = 0; s < kSlots; ++s) { mbar_init(&sm.a_full[s], 4); mbar_init(&sm.a_empty[s], 1); }
    mbar_init(&sm.d_full, 1);
    mbar_init(&sm.d_empty, kProducerWarps);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(&sm.tmem_base, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
#ifdef APAP_TC_TRACE
  if (tid == 0 && cta_lin < 8192) g_cta[cta_lin][2] = gtimer();
#endif
  const uint32_t tmem = sm.tmem_base;
  const uint32_t tmem_d = tmem;                    // columns [0, 32): hi x Ph sums; [32, 64): the two cross terms
  const uint32_t tmem_a = tmem + 2 * kNT;          // columns [64, 128): slot h, k-block e -> hi at 32 h + 16 e, lo + 8

  if (warp < kProducerWarps) {
    // ================= producers: thread = cell of the tile = accumulator row = TMEM lane =====
    const int q = warp & 3, h = warp >> 2;         // lane quarter, step parity
    const int row = q * 32 + lane;                 // row of the tile
    const int c = tile * 128 + row;
    const float2 av = reinterpret_cast<const float2 *>(anchors)[min(c, cells - 1)];
    const float2 ax2 = make_float2(av.x, av.x), ay2 = make_float2(av.y, av.y);
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    // the terms this warp drains and writes: all 24, or half of them when two warps share the quarter
    const int t0 = kParities == 1 ? 0 : 16 * h, nt = kParities == 1 ? kTerms : (h ? kTerms - 16 : 16);
    const float t_max = fminf(-__log2f(gamma_sq), 2.f);   // 2^-t_max = the clamp (polynomial path)
    int seg_done = 0;
    auto drain = [&]() {                           // add the finished segment's TMEM sums into the split's sums
      mbar_wait(&sm.d_full, seg_done & 1);
      tc_fence_after();
#pragma unroll
      for (int half = 0; half < 2 / kParities; ++half) {
        uint32_t v[16], u[16];
        tmem_ld16(tmem_d + lane_base + t0 + 16 * half, v);
        tmem_ld16(tmem_d + lane_base + kNT + t0 + 16 * half, u);
        tmem_wait_ld();
#pragma unroll
        for (int t = 0; t < 16; ++t) {
          if (16 * half + t < nt) {
            const float add = __uint_as_float(v[t]) + __uint_as_float(u[t]);
            float &dst = sm.acc[t0 + 16 * half + t][row];
            dst = seg_done ? dst + add : add;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.d_empty);
      ++seg_done;
    };
    // The clamp max(w, gamma^2) costs 16 of the ~180 instructions of a step.  When the caller's bound on |s v - s x| over
    // the whole scene (apap_weight_bound) shows that no pair reaches it, the same loop runs without -- same bits, the
    // max and the min were no-ops (margin 0.1 % + 1e-3 on t against the 2^-22 of MUFU.EX2 and the 1.6e-7 of the polynomial).
    const bool no_clamp = t_bound && fmaf(__ldg(t_bound + scene), 1.001f, 1e-3f) < (kPoly > 0 ? t_max : -__log2f(gamma_sq));
    const uint32_t slot = tmem_a + lane_base + h * 32;
    const uint32_t bar_full0 = smem_u32(&sm.smem_full[0]);
    const uint32_t bar_a_empty = smem_u32(&sm.a_empty[h]), bar_a_full = smem_u32(&sm.a_full[h]);
    const uint32_t co0 = smem_u32(sm.stage[0]) + (2 * kNT * kKB + h * kStepKb * kKbFloats) * 4;   // the step's coordinates
    auto steps = [&](auto no_clamp_tag) {
    constexpr bool kNoClamp = decltype(no_clamp_tag)::value;
    // this warp's step of stage `it` is s = 2 it + h: slot h of the A ring is its own (kParities == kSlots), and every
    // shared-memory address of the loop is a constant plus a multiple of the ring position
#pragma unroll kUnroll
    for (int it = 0; it < n_stage; ++it) {
      const uint32_t ss = (uint32_t)it & (kSmemStages - 1);
      if (q == 0 && lane == 0) TRACE(h, it, 0);
      mbar_wait_at(bar_full0 + 8 * ss, ((uint32_t)it / kSmemStages) & 1);
      const uint32_t a_par = (it & 1) ^ 1;         // first use of the slot: free
#if APAP_TC_EARLY_PROBE
      const uint32_t slot_free = mbar_test_at(bar_a_empty, a_par);   // consumed after the arithmetic
#endif
      if (q == 0 && lane == 0) TRACE(h, it, 1);
      uint32_t co = co0 + ss * kStageBytesTc;
      float w[kStepKb * 8];
#pragma unroll
      for (int e = 0; e < kStepKb; ++e, co += kKbBytes) {
        const float4 x0 = lds128(co), x1 = lds128(co + 16), y0 = lds128(co + 32), y1 = lds128(co + 48);
        const float2 kx[4] = {make_float2(x0.x, x0.y), make_float2(x0.z, x0.w), make_float2(x1.x, x1.y),
                              make_float2(x1.z, x1.w)};
        const float2 ky[4] = {make_float2(y0.x, y0.y), make_float2(y0.z, y0.w), make_float2(y1.x, y1.y),
                              make_float2(y1.z, y1.w)};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 dx = __fadd2_rn(ax2, make_float2(-kx[k].x, -kx[k].y));
          const float2 dy = __fadd2_rn(ay2, make_float2(-ky[k].x, -ky[k].y));
          const float2 d2 = __ffma2_rn(dy, dy, __fmul2_rn(dx, dx));
#if APAP_TC_NOMUFU
          w[8 * e + 2 * k] = fmaxf(1.f - d2.x, gamma_sq);
          w[8 * e + 2 * k + 1] = fmaxf(1.f - d2.y, gamma_sq);
#else
          if (kPoly > 0 && k >= 4 - kPoly) {
            // 2^-min(t, t_max) by a degree-7 polynomial in u = t - 1 on [-1, 1] (max relative error 1.6e-7)
            const float2 u = __fadd2_rn(kNoClamp ? make_float2(sqrt_approx(d2.x), sqrt_approx(d2.y))
                                                        : make_float2(fminf(sqrt_approx(d2.x), t_max), fminf(sqrt_approx(d2.y), t_max)),
                                        make_float2(-1.f, -1.f));
            float2 pp = __ffma2_rn(make_float2(-7.525117780e-06f, -7.525117780e-06f), u, make_float2(7.831371477e-05f, 7.831371477e-05f));
            pp = __ffma2_rn(pp, u, make_float2(-6.669662544e-04f, -6.669662544e-04f));
            pp = __ffma2_rn(pp, u, make_float2(4.808282945e-03f, 4.808282945e-03f));
            pp = __ffma2_rn(pp, u, make_float2(-2.775189467e-02f, -2.775189467e-02f));
            pp = __ffma2_rn(pp, u, make_float2(1.201134026e-01f, 1.201134026e-01f));
            pp = __ffma2_rn(pp, u, make_float2(-3.465736210e-01f, -3.465736210e-01f));
            pp = __ffma2_rn(pp, u, make_float2(0.5f, 0.5f));
            w[8 * e + 2 * k] = pp.x;
            w[8 * e + 2 * k + 1] = pp.y;
          } else {
            w[8 * e + 2 * k] = kNoClamp ? ex2_approx(-sqrt_approx(d2.x)) : fmaxf(ex2_approx(-sqrt_approx(d2.x)), gamma_sq);
            w[8 * e + 2 * k + 1] = kNoClamp ? ex2_approx(-sqrt_approx(d2.y)) : fmaxf(ex2_approx(-sqrt_approx(d2.y)), gamma_sq);
          }
#endif
        }
      }
#if APAP_TC_EARLY_PROBE
      if (!slot_free) mbar_wait_at(bar_a_empty, a_par);
#else
      mbar_wait_at(bar_a_empty, a_par);
#endif
      tc_fence_after();
      if (q == 0 && lane == 0) TRACE(h, it, 2);
#pragma unroll
      for (int e = 0; e < kStepKb; ++e) {
        uint32_t hl[16];                               // TF32 heads, then tails: the 16 A columns of k-block e
#pragma unroll
        for (int k = 0; k < 8; k += 2) {               // lo = w - hi (exact), two at a time on the packed FP32x2 adder
          hl[k] = tf32_head(w[8 * e + k]);
          hl[k + 1] = tf32_head(w[8 * e + k + 1]);
          const float2 l = __fadd2_rn(make_float2(w[8 * e + k], w[8 * e + k + 1]),
                                      make_float2(-__uint_as_float(hl[k]), -__uint_as_float(hl[k + 1])));
          hl[8 + k] = __float_as_uint(l.x);
          hl[8 + k + 1] = __float_as_uint(l.y);
        }
        tmem_st16(slot + e * 16, hl);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_at(bar_a_full);
      if (q == 0 && lane == 0) TRACE(h, it, 3);
      // a segment behind: its MMAs have had a step's worth of time to retire
      if ((it & (kSegKb / kStageKb - 1)) == 0 && it) drain();
    }
    };
    if (no_clamp) steps(std::true_type{}); else steps(std::false_type{});
    while (seg_done < n_seg) drain();
    if (c < cells) {
      // partials[split][t][cell]: consecutive threads write consecutive cells (coalesced); a thread writes
      // the terms it accumulated itself
      float *dst = partials + (size_t)split * kTerms * cells_padded + c;
#pragma unroll
      for (int t = 0; t < kTerms; ++t)
        if (t < nt) dst[(size_t)(t0 + t) * cells_padded] = sm.acc[t0 + t][row];
    }
    __threadfence();                               // the partial sums are visible device-wide before the tile is counted
  } else if (warp == kMmaWarp) {
    // ================= MMA issuer (one elected thread; the warp stays converged around it) ====
    const uint32_t idesc64 = idesc_tf32(2 * kNT), idesc32 = idesc_tf32(kNT);
    // shared-memory matrix descriptor, K-major, no swizzle: a core matrix is 8 rows x 16 B; LBO (bits 16-29) =
    // bytes between the two 16-byte K chunks of a row = 1024, SBO (bits 32-45) = bytes between 8-row groups = 128,
    // bits 46-47 = descriptor version 1 (sm_100); the start address (>> 4) goes in bits 0-13
    const uint64_t desc_hi = ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)(1024 >> 4) << 16);
    // One elected thread runs the whole loop (no per-step ELECT / reconvergence), one stage = both A slots per round:
    // the two producer parities finish their steps within ~50 cycles of each other (profiles/r01_gram_tc_trace.txt),
    // and this warp shares its scheduler with the producers of lane quarter 0 -- every instruction it does not issue
    // is a slot for the quarter the other three wait for.
    if (elect_one()) {
      for (int st = 0; st < n_stage; ++st) {
        const int ss = st % kSmemStages;
        mbar_wait(&sm.smem_full[ss], (st / kSmemStages) & 1);
        mbar_wait(&sm.a_full[0], st & 1);
        const int step = st * kSlots;
        const int in_seg = step & (kSegSteps - 1);                 // kSegSteps is even: a segment starts on slot 0 ...
        if (in_seg == 0 && st > 0) mbar_wait(&sm.d_empty, ((step / kSegSteps) - 1) & 1);   // previous segment drained
        tc_fence_after();
        // B tile of a k-block: rows 0..31 = Ph, rows 32..63 = Pl
        uint64_t b = desc_hi | (uint64_t)((smem_u32(sm.stage[ss]) & 0x3FFFFu) >> 4);
#pragma unroll
        for (int g = 0; g < kSlots; ++g) {           // slot g = step parity
          if (g) {
            mbar_wait(&sm.a_full[g], st & 1);
            tc_fence_after();
          }
#pragma unroll
          for (int e = 0; e < kStepKb; ++e, b += kKbBytes >> 4) {
            const uint32_t a_hi = tmem_a + g * 32 + e * 16, a_lo = a_hi + 8;
            const uint32_t fresh = (in_seg == 0 && g == 0 && e == 0) ? 0u : 1u;
            // D[0:32] (+)= hi . Ph and D[32:64] (+)= hi . Pl in one N = 64 MMA, then D[32:64] += lo . Ph:
            // the cross terms never touch the columns of the big sums
            mma_tf32_ts(tmem_d, a_hi, b, idesc64, fresh);
            mma_tf32_ts(tmem_d + kNT, a_lo, b, idesc32, 1u);
          }
          mma_commit(&sm.a_empty[g]);                // the A columns are free when these retire
        }
        // ... and ends on slot 1
        if (in_seg == kSegSteps - kSlots || st == n_stage - 1) mma_commit(&sm.d_full);
        mma_commit(&sm.smem_empty[ss]);              // ... and so is the shared-memory stage
      }
    }
    __syncwarp();
  } else {
    // ================= TMA producer (one thread) =============================================
    if (lane == 0) {
      const char *src = reinterpret_cast<const char *>(kp_blocks) + (size_t)kb0 * kKbBytes;
      for (int st = 0; st < n_stage; ++st) {
        const int ss = st % kSmemStages;
        mbar_wait(&sm.smem_empty[ss], ((st / kSmemStages) & 1) ^ 1);   // first pass: free
        mbar_arrive_expect_tx(&sm.smem_full[ss], kStageBytesTc);
        bulk_g2s(sm.stage[ss], src + (size_t)st * kStageBytesTc, kStageBytesTc, &sm.smem_full[ss]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
  // one more split of this tile is complete (release: every writer fenced before the barrier above)
  if (tid == 0 && tile_done) atomicAdd(tile_done + (size_t)scene * gridDim.y + tile, 1);
#ifdef APAP_TC_TRACE
  if (tid == 0 && cta_lin < 8192) g_cta[cta_lin][3] = gtimer();
#endif
}

int launch_gram_tc(const float *kp_blocks, const float *anchors, int batch, int cells, int n_kp_padded, float gamma_sq,
                   const float *t_bound, float *partials, int *tile_done, cudaStream_t st) {
  const GramPlan p = make_gram_plan(cells, n_kp_padded, APAP_GRAM_TCGEN05);
  const int n_kb = n_kp_padded / kKB;
  const int kb_per_split = p.chunks_per_split * (kChunk / kKB);
  dim3 grid(p.k_splits, (cells + 127) / 128, batch);
  if (grid.y > 65535 || batch > 65535) return fail(APAP_E_TOOBIG, "gram: more than 65535 cell tiles (8.3 M cells) or scenes per launch");
  if (APAP_TC_POLY > 0 && gamma_sq >= 0.25f && gamma_sq <= 1.f)   // the polynomial covers 2^-t for t in [0, 2]
    k_gram_tc<APAP_TC_POLY><<<grid, kTcThreads, sizeof(TcSmem), st>>>(kp_blocks, anchors, cells, p.cells_padded, n_kb,
                                                                      kb_per_split, p.k_splits, gamma_sq, t_bound, partials, tile_done);
  else
    k_gram_tc<0><<<grid, kTcThreads, sizeof(TcSmem), st>>>(kp_blocks, anchors, cells, p.cells_padded, n_kb, kb_per_split,
                                                           p.k_splits, gamma_sq, t_bound, partials, tile_done);
  return check_cuda(cudaGetLastError(), "k_gram_tc launch");
}

#ifdef APAP_TC_TRACE
extern "C" int apap_lab_trace(long long *out) { return (int)cudaMemcpyFromSymbol(out, g_trace, sizeof(g_trace)); }
extern "C" int apap_lab_cta_trace(long long *out) { return (int)cudaMemcpyFromSymbol(out, g_cta, sizeof(g_cta)); }
#endif

}  // namespace apap
