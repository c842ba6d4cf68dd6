// AFT_BF16 path: the 6-layer post-norm transformer encoder (reference src/models/blocks/encoders.py:44-55,69 ->
// torch _transformer_encoder_layer_fwd) as ONE persistent kernel on the 5th-gen tensor cores.
//
// One CTA per SM; a CTA owns one 280-token sequence at a time and carries it through all layers.  The
// residual stream never leaves the SM: it lives in shared memory as the bf16 A-operand image of the next GEMM.
// Per sequence the only HBM traffic is the 72 KB input image and the 72 KB result image written over it; weights
// (256 KB bf16 per layer) are streamed from L2 by 1-D bulk copies (cp.async.bulk) into a small ring.
//
//   warps 0..15  : compute warps (4 warpgroups; warp w serves TMEM lane quadrant w % 4 = SM sub-partition w % 4, the four
//                  warps of a quadrant split every accumulator row by columns) -- TMEM -> registers epilogues (bias,
//                  softmax, 1/l, residual + LayerNorm, GELU), writing the next operand image (bf16) to shared memory /
//                  P to TMEM.  setmaxnreg 104.
//   warps 16..19 : control warpgroup (setmaxnreg 56): warp 18 = producer (bulk copies + expect_tx), warp 19 = MMA issuer
//                  (the warp runs the schedule converged, the elected lane issues every tcgen05.mma / commit and owns
//                  the TMEM allocation); warps 16, 17 idle.
//
// The MMA issuer and the compute warps each run a static program; they meet only through mbarriers
// (tcgen05.commit -> "done" barriers; one arrive per compute warp -> "ready/free" barriers), so tensor-core work
// for the next tile is in flight while the epilogue of the current one runs:  S(t+1) is issued as soon as S(t) is
// in registers, P.V(t) runs under the exponentials of tile t+1, the next head's projection is issued under the tail
// tile, and the layer boundary is handed over per row tile (out_proj -> LayerNorm1 -> FFN1, FFN2 -> LayerNorm2 -> next
// projection).  Protocol rules and the chaos build that tests them: DESIGN.md 4.1, tc_ptx.cuh (chaos_delay).
//
// GEMMs use M = 128 row tiles (3 per sequence; the rows past 280 of the third tile read whatever follows in shared
// memory -- rows of A are independent, the corresponding accumulator lanes are never read); the attention of the
// 24-row tail tile is sliced over the four lane quadrants (see "tail tile" below).
//
// Shared memory map (bytes, every region 1024-aligned; operand layouts in tc_layout.cuh):
//   O    [      0,  73728)  attention output image (A of out_proj)   | FFN: hidden images, 2 x 36864
//                           (padding rows 280..287 of the second chunk: second mbarrier block)
//   X    [  73728, 147456)  residual stream image (A of QKV / FFN1, residual of both LayerNorms)
//   QKV  [ 147456, 202752)  Q_g | K_g | V_g of the current head, 288 x 64 B each (SWIZZLE_64B); P of the tail tile
//                           | out_proj / FFN weight ring: 3 slots x 16384, then the layer's 4 KB vector block
//   W    [ 202752, 227328)  in_proj slice of one head: rows q_g | k_g | v_g (96 x K=128) | FFN: second K-chunk of a W1 pair
//   MISC [ 227328, 232448)  in_proj bias double buffer, mbarriers, TMEM base, softmax / LayerNorm exchange
// Tensor memory map (columns): S [0,288)  P [288,432) (bf16 pairs)  O_acc x2 [432,464) [464,496);
//   QKV accumulators alias S; out_proj / FFN2 accumulators [0,384); one FFN1 accumulator tile [384,512).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "tc_encoder.cuh"
#include "tc_layout.cuh"
#include "tc_ptx.cuh"
#include "tc_math.cuh"

namespace aft {

namespace {

using namespace ptx;
using namespace tcm;

// In the score tiles one pair of exponentials in kPolyExp is evaluated on the FMA pipe (packed fp32x2 Cody-Waite + cubic,
// 6 issue slots per value) instead of MUFU (8 pipe cycles per warp instruction), so that both pipes finish together.
constexpr int kPolyExp = 3;
constexpr int kParts = 4;   // threads per accumulator row = compute warpgroups (8 warps x 224 registers measured 7.6 % slower)
static_assert(kXImageBytes % (16 * 32 * 4 * kParts) == 0, "the copy-out of the result image assumes whole passes of the compute warps");
constexpr int kComputeWarps = 4 * kParts;
constexpr int kTcThreads = 32 * (kComputeWarps + 4);   // compute warpgroups + [idle, idle, producer, MMA]
constexpr int kProducerWarp = kComputeWarps + 2, kMmaWarp = kComputeWarps + 3;   // highest warp ids: favoured by the issue arbiter
constexpr int kRegsCtrl = 56;                          // setmaxnreg budget of the control warpgroup
constexpr int kRegsCompute = 104;                      // setmaxnreg budget of the compute warpgroups (pool = threads x launch regs)
// per-layer epilogue vectors (fp32, global): [4 heads][q32 | k32 | v32] in_proj bias (q part pre-scaled), then the
// 1024-float block  b_out 128 | b_l1 256 | b_l2 128 | n1_w | n1_b | n2_w | n2_b  that is staged in shared memory
constexpr int kVecPerLayer = 1408;
constexpr int kVecBlock = 384;       // offset of the 1024-float block inside a layer's vector
constexpr int kVecBOut = 0, kVecBL1 = 128, kVecBL2 = 384, kVecN1W = 512, kVecN1B = 640, kVecN2W = 768, kVecN2B = 896;   // inside the block
constexpr uint32_t kQkvBiasBytes = 96 * 4, kVecBlockBytes = 1024 * 4;

constexpr uint32_t OFF_O = 0, OFF_X = 73728, OFF_QKV = 147456, OFF_W = 202752, OFF_MISC = 227328;
constexpr uint32_t kQkvPart = 18432;            // 288 rows x 64 B
constexpr uint32_t kRingSlot = 16384;
constexpr uint32_t kHidBytes = 36864;           // 288 rows x 128 B
constexpr uint32_t kWInSlice = 24576;           // 2 chunks x 96 rows x 128 B
constexpr uint32_t kMiscBytes = 5120;
constexpr uint32_t kTcSmemBytes = OFF_MISC + kMiscBytes;          // = 232448, the whole 227 KB; the dynamic window must be 1024-aligned

// mbarriers (byte offsets inside MISC).  Protocol rule: a waiter tests phase parity, so no barrier may complete two
// phases ahead of its waiter; every barrier below is lag <= 1 by construction (per-buffer barriers where the consumer
// waits lazily: O accumulators, FFN1 accumulators, hidden buffers).  "commit" barriers have count 1 (tcgen05.commit or expect_tx),
// "warp" barriers have count 16 (lane 0 of every compute warp arrives).
constexpr uint32_t MISC_QKV_BIAS = 0;       // [2][96] f32: in_proj bias of the current / next head (bulk-copied with the slice)
constexpr uint32_t MISC_BARS = 768;         // mbarriers below are relative to MISC_BARS
constexpr uint32_t OFF_VEC = OFF_QKV + 3 * kRingSlot;   // 4 KB vector block: tail of the (dead) V image, FFN/LayerNorm phases only
enum : uint32_t {
  MB_X_FULL = 0,       // commit: sequence image landed
  MB_X_FREE = 8,       // warp  : last LayerNorm of the sequence done, X may be replaced
  MB_ATTN_DONE = 16,   // commit: last P.V of the layer done -> Q/K/V images dead, ring may overwrite them
  MB_W_FULL = 24,      // 4 x commit: [0] in_proj slot, [1..3] ring slots
  MB_W_EMPTY = 56,     // 4 x commit
  MB_QKV_DONE = 88,    // commit: QKV accumulators of head g complete
  MB_QKV_READY = 96,   // warp  : Q/K/V images of head g written (and the accumulators read out)
  MB_S_DONE = 104,     // commit: score tile complete
  MB_S_LOADED = 112,   // warp  : score tile is in registers, S columns free
  MB_P_READY = 120,    // warp  : P tile written to TMEM
  MB_PV_DONE = 128,    // commit: P.V complete (P columns free, O accumulator valid)
  MB_O_FREE = 136,     // 2 x warp : O accumulator buffer b read out, O image columns written
  MB_TAIL_MAX = 152,   // warp  : tail tile, partial row maxima of every compute warp published
                       // (160, 224: free -- the per-tile OUT_DONE / X1_READY / X2_READY barriers live in the second block)
  MB_F1_DONE = 168,    // commit: FFN1 accumulator tile (128 rows x 128 hidden units) complete
  MB_F1_FREE = 176,    // warp  : FFN1 accumulator tile read out
  MB_F2_DONE = 184,    // 3 x commit: FFN2 partial product of row tile t complete (hidden rows of the tile free / final result)
  MB_HID_READY = 208,  // 2 x warp : hidden image rows of FFN tile k (two 64-unit chunks) complete, barrier k & 1.  Two barriers:
                       // FFN1(k+1) is issued before the issuer waits for tile k, so a single barrier could collect a fast
                       // warp's arrival for tile k+1 while a slow warp still owes the one for tile k
  MB_VEC_FULL = 232,   // commit: per-layer vector block landed in shared memory
  MB_BIAS_FULL = 240,  // 2 x commit: in_proj bias of head g landed in buffer g & 1
  MB_COUNT_BYTES = 256,
};
constexpr uint32_t kXchgArray = 2048;   // bytes of one exchange array: [4][128] f32 (kParts <= 4 rows used)
constexpr uint32_t MISC_XMAX = 1024;    // exchange array 0 (softmax maxima / LayerNorm sums)
constexpr uint32_t MISC_TMEM_PTR = MISC_XMAX;   // start-up only: read by every thread before the exchange area is first used
constexpr uint32_t MISC_XSUM = MISC_XMAX + kXchgArray;   // exchange array 1 (softmax sums / LayerNorm sums of squares)

constexpr uint32_t TM_S = 0, TM_P = 288, TM_O = 432, TM_QKV = 0, TM_OUT = 0, TM_F1 = 384;
// Accumulator columns of the QKV projection of (head g, row tile t).  Head 0 follows LayerNorm2 tile by tile and uses
// columns t * 96 (inside the out_proj / FFN2 accumulators that LayerNorm2 has released up to that tile).  The tail
// scores of head g - 1 occupy all score columns, so for g > 0 tile 0 goes to the P columns -- free as soon as P.V of the
// second score tile has completed: the tail's P lives in shared memory -- and is issued BEFORE the tail's scores are
// read; tiles 1 and 2 follow in columns 0 and 96 while the tail's softmax runs.
__device__ __forceinline__ uint32_t qkv_col(int g, int t) {
  return g == 0 ? (uint32_t)(t * 96) : (t == 0 ? TM_P : (uint32_t)((t - 1) * 96));
}

constexpr uint32_t kIdescQkv = make_idesc_bf16(128, 96, false, false);
constexpr uint32_t kIdescS = make_idesc_bf16(128, 144, false, false);
constexpr uint32_t kIdescPV = make_idesc_bf16(128, 32, false, true);     // B = V, MN-major
constexpr uint32_t kIdescN128 = make_idesc_bf16(128, 128, false, false);
constexpr uint32_t kIdescS96 = make_idesc_bf16(128, 96, false, false), kIdescS64 = make_idesc_bf16(128, 64, false, false);   // tail: key slices
constexpr uint32_t kIdescPT = make_idesc_bf16(64, 32, false, true);    // tail: O = P (image, K-major, M = 64) . V (MN-major)
// The padding rows 280..287 of the O image's first chunk are unused; those of its second chunk hold the second mbarrier
// block (below).
// Second LayerNorm exchange area (2 x kXchgArray bytes), used by row tile 1: the start of the O region.  Both LayerNorms run
// when that region is dead (O image consumed by out_proj / hidden images consumed by FFN2, next writer behind a full
// X1_READY / X2_READY hand-shake).
constexpr uint32_t OFF_LN_XCHG = OFF_O;
// LayerNorm1 cannot use it: FFN1 of row tile 0 starts as soon as LayerNorm1 has released that tile, so fast warps may
// already store hidden rows into the O region while others are still in LayerNorm1.  Its second area is the tail of the
// in_proj slot: bytes [16 K, 24 K) are only written by the 24 KB head slices, which are not in flight between the last
// head's projection and the end of FFN1.
constexpr uint32_t OFF_LN1_XCHG = OFF_W + 16384;
// Second mbarrier block: the padding rows 280..287 of the O region's second chunk (never written: the epilogues skip
// padding rows, the tensor core only reads them into padding rows of its results).  Per-row-tile hand-offs:
constexpr uint32_t OFF_BAR2 = OFF_O + kXChunkBytes + 280 * 128;
constexpr uint32_t MB2_OUT_DONE = 0;    // 3 x commit: out_proj accumulators of row tile t complete
constexpr uint32_t MB2_X1_READY = 24;   // 3 x warp  : LayerNorm1 rows of tile t written to X
constexpr uint32_t MB2_X2_READY = 48;   // 3 x warp  : LayerNorm2 rows of tile t written to X, accumulator columns of the tile free



// =============================================================================================
// MMA issue helpers (called by the single issuing thread).  `sb` = 1024-aligned shared base address.
// =============================================================================================
// D (N cols at d_col) (+)= A(image with 128-B rows)[128 rows at a_base] . B(image at b_base)^T ; K = 16 * ksteps
__device__ __forceinline__ void issue_gemm_sw128(uint32_t tmem, uint32_t d_col, uint32_t a_base, uint32_t a_chunk_bytes,
                                                 uint32_t b_base, uint32_t b_chunk_bytes, int ksteps, uint32_t idesc,
                                                 bool accumulate_first, bool el = true) {
  // descriptor = (hi: SBO | version | swizzle, constant) : (lo: LBO | start address >> 4); the K step only moves `lo`
  constexpr uint32_t kHi = (uint32_t)(desc_k_sw128_const() >> 32);
  const uint32_t a_lo = (uint32_t)desc_k_sw128_const() | ((a_base >> 4) & 0x3FFF);
  const uint32_t b_lo = (uint32_t)desc_k_sw128_const() | ((b_base >> 4) & 0x3FFF);
  const uint32_t a_chunk = a_chunk_bytes >> 4, b_chunk = b_chunk_bytes >> 4;
#pragma unroll 4
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint32_t a = a_lo + (ks >> 2) * a_chunk + (ks & 3) * 2;
    const uint32_t b = b_lo + (ks >> 2) * b_chunk + (ks & 3) * 2;
    mma_ss(tmem + d_col, ((uint64_t)kHi << 32) | a, ((uint64_t)kHi << 32) | b, idesc, accumulate_first || ks > 0, el);
  }
}
// Descriptors of the attention operands: constant high word (SBO | version | swizzle), low word = LBO | address >> 4,
// so that stepping through an operand is one 32-bit add per MMA.
constexpr uint32_t kDescHiSw64 = (uint32_t)(((uint64_t)(512 >> 4)) | ((uint64_t)1 << 14) | ((uint64_t)kSwizzle64 << 29));
__device__ __forceinline__ uint32_t desc_lo_k64(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | ((16u >> 4) << 16); }     // K-major, LBO 16
__device__ __forceinline__ uint32_t desc_lo_mn64(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | ((512u >> 4) << 16); }   // MN-major, LBO 512
__device__ __forceinline__ uint64_t desc_sw64(uint32_t lo) { return ((uint64_t)kDescHiSw64 << 32) | lo; }
// S[tile t] = Q_g[tile t] . K_g^T   (two N = 144 halves, K = 32)
__device__ __forceinline__ void issue_scores(uint32_t tmem, uint32_t sb, int t, bool el = true) {
  const uint32_t q = desc_lo_k64(sb + OFF_QKV + t * 128 * 64);
  const uint32_t k = desc_lo_k64(sb + OFF_QKV + kQkvPart);
#pragma unroll
  for (int nh = 0; nh < 2; ++nh)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      mma_ss(tmem + TM_S + nh * 144, desc_sw64(q + ks * 2), desc_sw64(k + (nh * 144 * 64) / 16 + ks * 2), kIdescS, ks > 0, el);
}
// O_acc[buf] = P (TMEM, bf16 pairs) . V_g   (K = 288 keys = 18 steps, N = 32)
__device__ __forceinline__ void issue_pv(uint32_t tmem, uint32_t sb, int obuf, bool el = true) {
  const uint32_t v = desc_lo_mn64(sb + OFF_QKV + 2 * kQkvPart);
  const uint32_t d = tmem + TM_O + obuf * 32, a = tmem + TM_P;
#pragma unroll
  for (int ks = 0; ks < 18; ++ks) mma_ts(d, a + ks * 8, desc_sw64(v + ks * 64), kIdescPV, ks > 0, el);
}

// ---- tail tile (query rows 256..279), sliced over the lane quadrants.  TMEM lane quadrant w % 4 belongs to the warps
// of SM sub-partition w % 4, so a 128 x 288 score tile with 24 valid rows would keep a single sub-partition (one MUFU)
// busy while 12 of the 16 compute warps wait.  Row i of an M = 128 A operand lands on TMEM lane i, and the A operand
// is addressed by its first row: starting the Q image 32 q rows EARLIER puts the tail queries 256..279 on the lanes of
// quadrant q (rows in front of them are other queries, their results are never read).  The tail scores are issued as
// four such MMAs over disjoint key slices -- quadrant 0: keys [0, 96), quadrants 1..3: 64 keys each -- into the
// ordinary score columns, so that every sub-partition owns a quarter of the tail's exponentials in the ordinary
// row-major form (no cross-lane reductions).  P goes to shared memory as a K-major SWIZZLE_64B A-operand image over
// the dead Q image (nine 32-key chunks of 32 rows x 64 B; an MMA reads past its chunk into the following ones: only
// rows 0..23 matter), and O_tail = P . V runs as M = 64 MMAs into the usual accumulator columns.
__device__ __forceinline__ int tail_key0(int q) { return q == 0 ? 0 : 32 + 64 * q; }   // 0, 96, 160, 224
__device__ __forceinline__ void issue_scores_tail(uint32_t tmem, uint32_t sb, bool el = true) {
#pragma unroll
  for (int qq = 0; qq < 4; ++qq) {
    const int key0 = qq == 0 ? 0 : 32 + 64 * qq;
    const uint32_t a = desc_lo_k64(sb + OFF_QKV + (256 - 32 * qq) * 64);
    const uint32_t k = desc_lo_k64(sb + OFF_QKV + kQkvPart + key0 * 64);
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      mma_ss(tmem + TM_S + key0, desc_sw64(a + ks * 2), desc_sw64(k + ks * 2), qq == 0 ? kIdescS96 : kIdescS64, ks > 0, el);
  }
}
__device__ __forceinline__ void issue_pv_tail(uint32_t tmem, uint32_t sb, int obuf, bool el = true) {
  const uint32_t v = desc_lo_mn64(sb + OFF_QKV + 2 * kQkvPart);
  const uint32_t d = tmem + TM_O + obuf * 32;
#pragma unroll
  for (int ks = 0; ks < 18; ++ks)
    mma_ss(d, desc_sw64(desc_lo_k64(sb + OFF_QKV + (ks >> 1) * 2048) + (ks & 1) * 2), desc_sw64(v + ks * 64), kIdescPT, ks > 0, el);
}

// =============================================================================================
// compute-warp epilogues.  q = warp % 4 (TMEM lane quadrant), part = compute warpgroup (0 .. kParts-1): the kParts
// threads that own TMEM lane `rt` (one per warpgroup) split every accumulator row by columns.
// =============================================================================================

// QKV accumulators of (head g, row tile t) -> + bias -> bf16 -> Q_g / K_g / V_g images (SWIZZLE_64B rows of 64 B).
// The 96 accumulator columns [q_g | k_g | v_g] = 12 units of 8 columns, split evenly over the warpgroups.
constexpr int kQkvUnits = 12 / kParts;
// The thread's slice of the in_proj bias (the same 8 * kQkvUnits columns for every row tile): fetched before the
// accumulators are waited for, so that its shared-memory latency hides under that wait.
struct QkvBias { uint4 v[2 * kQkvUnits]; };
__device__ __forceinline__ QkvBias epi_qkv_bias(uint32_t bias96, int part) {
  QkvBias b;
#pragma unroll
  for (int i = 0; i < 2 * kQkvUnits; ++i) b.v[i] = ld_shared_v4(bias96 + (part * kQkvUnits * 2 + i) * 16);
  return b;
}
__device__ __forceinline__ void epi_qkv_store(uint32_t sb, const QkvBias& bias, int t, int q, int part, int lane, const uint32_t (&acc)[8 * kQkvUnits]) {
  const int r = t * 128 + q * 32 + lane;
  const int sw = (r >> 1) & 3;
#pragma unroll
  for (int i = 0; i < kQkvUnits; ++i) {
    const int u8 = part * kQkvUnits + i;     // unit index inside [q | k | v]
    const int mat = u8 >> 2, u = u8 & 3;     // which matrix, which 16-byte unit of its 64-byte row
    const uint4 b0 = bias.v[2 * i], b1 = bias.v[2 * i + 1];
    const uint32_t* a = acc + i * 8;
    auto sum = [](uint32_t x0, uint32_t x1, uint32_t y0, uint32_t y1) {
      return pack_bf16_pair(add2(pack2(__uint_as_float(x0), __uint_as_float(x1)), pack2(__uint_as_float(y0), __uint_as_float(y1))));
    };
    st_shared_v4(sb + OFF_QKV + mat * kQkvPart + r * 64 + ((u ^ sw) << 4), sum(a[0], a[1], b0.x, b0.y), sum(a[2], a[3], b0.z, b0.w),
                 sum(a[4], a[5], b1.x, b1.y), sum(a[6], a[7], b1.z, b1.w));
  }
}
__device__ __forceinline__ void epi_qkv(uint32_t tmem, uint32_t sb, const QkvBias& bias, int g, int t, int q, int part, int lane) {
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + qkv_col(g, t) + part * (8 * kQkvUnits);
  uint32_t acc[8 * kQkvUnits];
  tmem_ld_cols(taddr, acc);
  tmem_wait_ld();
  epi_qkv_store(sb, bias, t, q, part, lane, acc);
}
// row tiles 0 and 1 together: one TMEM round trip instead of two
__device__ __forceinline__ void epi_qkv_pair(uint32_t tmem, uint32_t sb, const QkvBias& bias, int g, int q, int part, int lane) {
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + part * (8 * kQkvUnits);
  uint32_t acc0[8 * kQkvUnits], acc1[8 * kQkvUnits];
  tmem_ld_cols(taddr + qkv_col(g, 0), acc0);
  tmem_ld_cols(taddr + qkv_col(g, 1), acc1);
  tmem_wait_ld();
  epi_qkv_store(sb, bias, 0, q, part, lane, acc0);
  epi_qkv_store(sb, bias, 1, q, part, lane, acc1);
}

constexpr int kSmCols = 288 / kParts;   // score columns per thread; the last warpgroup has 8 padding keys (280..287)

// Softmax of one score tile, in the pieces the barrier protocol needs.
// (1) load this thread's score columns and return their maximum
__device__ __forceinline__ float softmax_load(uint32_t tmem, int q, int part, float (&v)[kSmCols]) {
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + TM_S + part * kSmCols;
  uint32_t x[kSmCols];
  tmem_ld_cols(taddr, x);
  tmem_wait_ld();
#pragma unroll
  for (int j = 0; j < kSmCols; ++j) v[j] = __uint_as_float(x[j]);
  if (part == kParts - 1) {
#pragma unroll
    for (int j = kSmCols - (kSPad - kS); j < kSmCols; ++j) v[j] = -INFINITY;   // keys 280..287 are padding
  }
  float m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3];
#pragma unroll
  for (int j = 4; j < kSmCols; j += 4) {
    m0 = fmaxf(m0, v[j]); m1 = fmaxf(m1, v[j + 1]); m2 = fmaxf(m2, v[j + 2]); m3 = fmaxf(m3, v[j + 3]);
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}
// (2) exponentials in place (scores are in log2 units: q rows of in_proj pre-scaled by log2(e)/sqrt(dh)); returns the sum
__device__ __forceinline__ float softmax_exp(float (&v)[kSmCols], float m) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  // The exponentials are MUFU-bound (16 ex2 / clk / SM); every fourth one is computed on the FMA pipe instead.
#pragma unroll
  for (int j = 0; j < kSmCols; j += 4) {
    v[j] = ex2(v[j] - m); v[j + 1] = ex2(v[j + 1] - m); v[j + 2] = ex2(v[j + 2] - m);
    v[j + 3] = ex2_poly(v[j + 3] - m);
    s0 += v[j]; s1 += v[j + 1]; s2 += v[j + 2]; s3 += v[j + 3];
  }
  return (s0 + s1) + (s2 + s3);
}
// (2+3) exponentials and P store interleaved (16 columns at a time): the packing and the TMEM stores issue under the
// MUFU-bound exponentials instead of after them.  The caller has made sure that P.V(t-1) no longer reads P.
__device__ __forceinline__ float softmax_exp_store(uint32_t tmem, int q, int part, float (&v)[kSmCols], float m) {
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + TM_P + part * (kSmCols / 2);
  constexpr int kFull = kSmCols / 16;
  const f32x2 negm2 = pack2(-m, -m);
  f32x2 s2a = pack2(0.f, 0.f), s2b = pack2(0.f, 0.f);
  // one pair of columns: subtract the row maximum, exponentiate (MUFU, or the FMA pipe for every kPolyExp-th pair),
  // accumulate the row sum, return the packed bf16 pair
  auto exp_pair = [&](int gp) -> uint32_t {
    const f32x2 x2 = add2(pack2(v[2 * gp], v[2 * gp + 1]), negm2);
    f32x2 e2;
    if (gp % kPolyExp == kPolyExp - 1) {
      e2 = ex2_poly2(x2);
    } else {
      float a, b;
      unpack2(x2, a, b);
      e2 = pack2(ex2(a), ex2(b));
    }
    if (gp & 1) s2b = add2(s2b, e2); else s2a = add2(s2a, e2);
    return pack_bf16_pair(e2);
  };
#pragma unroll
  for (int i = 0; i < kFull; ++i) {
    uint32_t pk[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) pk[j] = exp_pair(i * 8 + j);
    tmem_st8(taddr + i * 8, pk);
  }
  if (kSmCols % 16) {
    uint32_t pk4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pk4[j] = exp_pair(kFull * 8 + j);
    tmem_st4(taddr + kFull * 8, pk4);
  }
  tmem_wait_st();
  float sa, sb2, sc, sd;
  unpack2(s2a, sa, sb2);
  unpack2(s2b, sc, sd);
  return (sa + sb2) + (sc + sd);
}
// (3) P tile -> TMEM as bf16 pairs (A operand of P.V): kSmCols / 2 packed columns per thread
__device__ __forceinline__ void softmax_store(uint32_t tmem, int q, int part, const float (&v)[kSmCols]) {
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + TM_P + part * (kSmCols / 2);
  constexpr int kFull = kSmCols / 16;
#pragma unroll
  for (int i = 0; i < kFull; ++i) {
    uint32_t pk[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) pk[j] = pack_bf16x2(v[i * 16 + 2 * j], v[i * 16 + 2 * j + 1]);
    tmem_st8(taddr + i * 8, pk);
  }
  if (kSmCols % 16) {
    uint32_t pk4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pk4[j] = pack_bf16x2(v[kFull * 16 + 2 * j], v[kFull * 16 + 2 * j + 1]);
    tmem_st4(taddr + kFull * 8, pk4);
  }
  tmem_wait_st();
}

// O accumulator (128 x 32) of (head g, tile t) -> / l -> bf16 -> O image columns g*32 .. g*32+31, split over the warpgroups
constexpr int kOCols = 32 / kParts;
__device__ __forceinline__ void epi_o_store(uint32_t sb, int g, int t, float inv_l, int q, int part, int lane, const uint32_t (&a)[kOCols]);
__device__ __forceinline__ void epi_o(uint32_t tmem, uint32_t sb, int g, int t, int obuf, float inv_l, int q, int part, int lane) {
  uint32_t a[kOCols];
  tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_O + obuf * 32 + part * kOCols, a);
  tmem_wait_ld();
  epi_o_store(sb, g, t, inv_l, q, part, lane, a);
}
// one O image row r: this thread's kOCols accumulator columns (warpgroup `part`) of head g, scaled by 1 / l
__device__ __forceinline__ void epi_o_store_row(uint32_t sb, int g, int r, float inv_l, int part, const uint32_t (&a)[kOCols]) {
  const uint32_t row = sb + OFF_O + (g >> 1) * kXChunkBytes + r * 128;
#pragma unroll
  for (int i = 0; i < kOCols / 8; ++i) {
    const int u = (g & 1) * 4 + part * (kOCols / 8) + i;
    const f32x2 il = pack2(inv_l, inv_l);
    auto sc = [&](int j) { return pack_bf16_pair(mul2(pack2(__uint_as_float(a[8 * i + j]), __uint_as_float(a[8 * i + j + 1])), il)); };
    st_shared_v4(row + ((u ^ (r & 7)) << 4), sc(0), sc(2), sc(4), sc(6));
  }
}
__device__ __forceinline__ void epi_o_store(uint32_t sb, int g, int t, float inv_l, int q, int part, int lane, const uint32_t (&a)[kOCols]) {
  epi_o_store_row(sb, g, t * 128 + q * 32 + lane, inv_l, part, a);
}

// ---- tail tile (see issue_scores_tail).  Thread (q, part, lane) owns tail query 256 + lane and NC keys:
// tail_key0(q) + part * NC ...  The 16 threads of a row (4 quadrants x 4 warpgroups) exchange their partial maxima /
// sums through the ordinary exchange arrays, each thread using the slot it also owns in the full tiles ([part][32 q +
// lane]): a warp only overwrites slots of its own quadrant, whose previous readers (the quadrant's warps, second named
// barrier of tile 1) are behind it, and the next full-tile writers are a whole QKV hand-shake away.
template <int NC>
__device__ __forceinline__ void softmax_tail_impl(uint32_t tmem, uint32_t sb, uint32_t miscb, uint32_t s_loaded_bar, uint32_t tail_bar, uint32_t tail_parity, int q, int part, int lane) {
  static_assert(NC % 8 == 0, "a thread's keys must be whole 16-byte units of the P image");
  const int key0 = tail_key0(q) + part * NC;
  float v[NC];
  {
    uint32_t x[NC];
    tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_S + key0, x);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < NC; ++j) v[j] = __uint_as_float(x[j]);
  }
  if (key0 + NC > kS) {   // keys 280..287 are padding (last warpgroup of quadrant 3)
#pragma unroll
    for (int j = 0; j < NC; ++j)
      if (key0 + j >= kS) v[j] = -INFINITY;
  }
  float m = fmaxf(v[0], v[1]);
#pragma unroll
  for (int j = 2; j < NC; j += 2) m = fmaxf(m, fmaxf(v[j], v[j + 1]));
  const uint32_t own = (uint32_t)(part * 512 + (q * 32 + lane) * 4);
  st_shared_f32(miscb + MISC_XMAX + own, m);
  tc_fence_before_sync();
  warp_arrive(s_loaded_bar, lane);
  // rendezvous of all compute warps (the 16 partial maxima of every row are published): an mbarrier rather than a named
  // barrier -- the two instantiations of this function are different call sites, which compute-sanitizer's synccheck
  // reports for bar.sync; sharing one call site instead cost 4 % of the kernel (the score registers had to survive a
  // merge of the two branches)
  warp_arrive(tail_bar, lane);
  mbar_wait(tail_bar, tail_parity);
#pragma unroll
  for (int pp = 0; pp < 4; ++pp)
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) m = fmaxf(m, ld_shared_f32(miscb + MISC_XMAX + pp * 512 + (qq * 32 + lane) * 4));
  const f32x2 negm2 = pack2(-m, -m);
  f32x2 s2 = pack2(0.f, 0.f);
  uint32_t pk[NC / 2];
#pragma unroll
  for (int j = 0; j < NC / 2; ++j) {
    const f32x2 x2 = add2(pack2(v[2 * j], v[2 * j + 1]), negm2);
    f32x2 e2;
    if (j % kPolyExp == kPolyExp - 1) {
      e2 = ex2_poly2(x2);
    } else {
      float a, b;
      unpack2(x2, a, b);
      e2 = pack2(ex2(a), ex2(b));
    }
    s2 = add2(s2, e2);
    pk[j] = pack_bf16_pair(e2);
  }
  // P row `lane`, keys key0 .. key0 + NC: 32-key chunks of 32 rows x 64 B (SWIZZLE_64B, 16-byte units of 8 keys)
#pragma unroll
  for (int u = 0; u < NC / 8; ++u) {
    const int key = key0 + 8 * u;
    st_shared_v4(sb + OFF_QKV + (key >> 5) * 2048 + lane * 64 + ((((key & 31) >> 3) ^ ((lane >> 1) & 3)) << 4), pk[4 * u], pk[4 * u + 1],
                 pk[4 * u + 2], pk[4 * u + 3]);
  }
  float sa, sb2;
  unpack2(s2, sa, sb2);
  st_shared_f32(miscb + MISC_XSUM + own, sa + sb2);
}
__device__ __forceinline__ void softmax_tail(uint32_t tmem, uint32_t sb, uint32_t miscb, uint32_t s_loaded_bar, uint32_t tail_bar,
                                             uint32_t tail_parity, int q, int part, int lane) {
  static_assert(kParts == 4, "the tail tile assumes four warpgroups");
  if (q == 0) softmax_tail_impl<24>(tmem, sb, miscb, s_loaded_bar, tail_bar, tail_parity, q, part, lane);
  else softmax_tail_impl<16>(tmem, sb, miscb, s_loaded_bar, tail_bar, tail_parity, q, part, lane);
}
// O_tail accumulator (M = 64: tail query i in lane i % 16 of quadrant i / 16) -> / l -> bf16 -> O image rows 256..279
__device__ __forceinline__ void epi_o_tail(uint32_t tmem, uint32_t sb, uint32_t miscb, int g, int obuf, int q, int part, int lane) {
  uint32_t a[kOCols];
  tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_O + obuf * 32 + part * kOCols, a);
  tmem_wait_ld();
  const int i = q * 16 + lane;
  if (lane < 16 && i < kS - 256) {
    float l = 0.f;
#pragma unroll
    for (int pp = 0; pp < 4; ++pp)
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) l += ld_shared_f32(miscb + MISC_XSUM + pp * 512 + (qq * 32 + i) * 4);
    epi_o_store_row(sb, g, 256 + i, rcp_approx(l), part, a);
  }
}

// out_proj / linear2 accumulators (tile t) + bias + residual (X image) -> LayerNorm -> X image in place (+ fp32 rows to
// h_out after the last layer).  A row is shared by the kParts threads that own TMEM lane `rt`; sum and sum of squares are
// combined through shared memory (one exchange, one named barrier of the quadrant's warps).
// `vec` = shared address of the layer's vector block; `xchg` = shared address of the exchange area.
constexpr int kLnCols = 128 / kParts, kLnUnits = kLnCols / 8;
__device__ __forceinline__ void epi_ln(uint32_t tmem, uint32_t sb, uint32_t vec, int which, int t, int q, int part, int lane,
                                       uint32_t xchg, char* x_images, int out_seq) {
  const int rt = q * 32 + lane, r = t * 128 + rt;
  const uint32_t bias = vec + 4 * ((which == 1 ? kVecBOut : kVecBL2) + part * kLnCols);
  const uint32_t gam = vec + 4 * ((which == 1 ? kVecN1W : kVecN2W) + part * kLnCols);
  const uint32_t bet = vec + 4 * ((which == 1 ? kVecN1B : kVecN2B) + part * kLnCols);
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + TM_OUT + t * 128 + part * kLnCols;
  const int c0 = part * kLnCols;                         // first column of this thread
  const uint32_t xrow = sb + OFF_X + (c0 >> 6) * kXChunkBytes + r * 128;
  const int u0 = (c0 & 63) >> 3;
  f32x2 v[kLnCols / 2];
  uint32_t acc[kLnCols];
  tmem_ld_cols(taddr, acc);
  tmem_wait_ld();
  f32x2 s2 = pack2(0.f, 0.f), q2 = pack2(0.f, 0.f);
#pragma unroll
  for (int u = 0; u < kLnUnits; ++u) {   // 16-byte unit = 8 columns
    const uint4 xr = ld_shared_v4(xrow + (((u0 + u) ^ (r & 7)) << 4));
    const uint4 b0 = ld_shared_v4(bias + u * 32), b1 = ld_shared_v4(bias + u * 32 + 16);
    const uint32_t xw[4] = {xr.x, xr.y, xr.z, xr.w};
    const f32x2 bb[4] = {pack2(__uint_as_float(b0.x), __uint_as_float(b0.y)), pack2(__uint_as_float(b0.z), __uint_as_float(b0.w)),
                         pack2(__uint_as_float(b1.x), __uint_as_float(b1.y)), pack2(__uint_as_float(b1.z), __uint_as_float(b1.w))};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const f32x2 a2 = pack2(__uint_as_float(acc[u * 8 + 2 * j]), __uint_as_float(acc[u * 8 + 2 * j + 1]));
      const f32x2 y = add2(add2(a2, bb[j]), bf16x2_to_f32x2(xw[j]));
      v[u * 4 + j] = y;
      s2 = add2(s2, y);
      q2 = fma2(y, y, q2);
    }
  }
  {
    float sa, sb2, qa, qb;
    unpack2(s2, sa, sb2);
    unpack2(q2, qa, qb);
    st_shared_f32(xchg + (part * 128 + rt) * 4, sa + sb2);
    st_shared_f32(xchg + kXchgArray + (part * 128 + rt) * 4, qa + qb);
  }
  named_bar_sync(1 + q, 32 * kParts);
  float sum = 0.f, sq = 0.f;
#pragma unroll
  for (int pp = 0; pp < kParts; ++pp) {
    sum += ld_shared_f32(xchg + (pp * 128 + rt) * 4);
    sq += ld_shared_f32(xchg + kXchgArray + (pp * 128 + rt) * 4);
  }
  const float mean = sum * (1.0f / 128.0f);
  const float var = fmaxf(fmaf(-mean, mean, sq * (1.0f / 128.0f)), 0.f);
  const float rstd = rsqrtf(var + 1e-5f);
  const float shift = -mean * rstd;
  const f32x2 rstd2 = pack2(rstd, rstd), shift2 = pack2(shift, shift);
#pragma unroll
  for (int u = 0; u < kLnUnits; ++u) {
    const uint4 g0 = ld_shared_v4(gam + u * 32), g1 = ld_shared_v4(gam + u * 32 + 16);
    const uint4 e0 = ld_shared_v4(bet + u * 32), e1 = ld_shared_v4(bet + u * 32 + 16);
    const f32x2 gg[4] = {pack2(__uint_as_float(g0.x), __uint_as_float(g0.y)), pack2(__uint_as_float(g0.z), __uint_as_float(g0.w)),
                         pack2(__uint_as_float(g1.x), __uint_as_float(g1.y)), pack2(__uint_as_float(g1.z), __uint_as_float(g1.w))};
    const f32x2 ee[4] = {pack2(__uint_as_float(e0.x), __uint_as_float(e0.y)), pack2(__uint_as_float(e0.z), __uint_as_float(e0.w)),
                         pack2(__uint_as_float(e1.x), __uint_as_float(e1.y)), pack2(__uint_as_float(e1.z), __uint_as_float(e1.w))};
    f32x2 o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = fma2(fma2(v[u * 4 + j], rstd2, shift2), gg[j], ee[j]);
    // padding rows 280..287 stay zero: their accumulators are fed by padding rows of the O region (which hold the second
    // mbarrier block) and must not leak non-finite values into the V image of the next layer
    if (r < kS) {
      const uint4 pk = make_uint4(pack_bf16_pair(o[0]), pack_bf16_pair(o[1]), pack_bf16_pair(o[2]), pack_bf16_pair(o[3]));
      const uint32_t off = r * 128 + (((u0 + u) ^ (r & 7)) << 4);
      st_shared_v4(sb + OFF_X + (c0 >> 6) * kXChunkBytes + off, pk.x, pk.y, pk.z, pk.w);
      // last layer: the same 16 bytes go to the sequence's image in global memory (the encoder output replaces its input)
      if (out_seq >= 0) *reinterpret_cast<uint4*>(x_images + out_seq * (int64_t)kXImageBytes + (c0 >> 6) * kXChunkBytes + off) = pk;
    }
  }
  // No trailing barrier: consecutive tiles alternate between two exchange areas (see the call sites), and a warp can only
  // reach tile t + 2 after every warp of its quadrant has passed the barrier of tile t + 1, i.e. finished reading tile t.
}

// FFN1 accumulators (pair pr = hidden units 128 pr .. 128 pr + 127, one row tile), split over the warpgroups: load + bias
constexpr int kActCols = 128 / kParts;
__device__ __forceinline__ void act_load(uint32_t tmem, uint32_t vec, int pr, int q, int part, f32x2 (&f)[kActCols / 2]) {
  const uint32_t bias = vec + 4 * (kVecBL1 + pr * 128 + part * kActCols);
  uint32_t a[kActCols];
  tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_F1 + part * kActCols, a);
  tmem_wait_ld();
#pragma unroll
  for (int u = 0; u < kActCols / 4; ++u) {
    const uint4 b = ld_shared_v4(bias + u * 16);
    f[u * 2] = add2(pack2(__uint_as_float(a[u * 4]), __uint_as_float(a[u * 4 + 1])), pack2(__uint_as_float(b.x), __uint_as_float(b.y)));
    f[u * 2 + 1] = add2(pack2(__uint_as_float(a[u * 4 + 2]), __uint_as_float(a[u * 4 + 3])), pack2(__uint_as_float(b.z), __uint_as_float(b.w)));
  }
}
// GELU / ReLU -> bf16 -> hidden images (K-chunks of FFN2's A operand): the pair's first 64 units go to buffer 0, the
// others to buffer 1.  Padding rows 280..287 are not written (the O region's padding rows hold scratch data).
__device__ __forceinline__ void act_store(uint32_t sb, int t, int act, int q, int part, int lane, f32x2 (&f)[kActCols / 2]) {
  const int r = t * 128 + q * 32 + lane;
  uint32_t pk[kActCols / 2];
  if (act == AFT_ACT_GELU) {
#pragma unroll
    for (int j = 0; j < kActCols / 2; ++j) pk[j] = pack_bf16_pair(gelu_tanh2(f[j]));
  } else {
#pragma unroll
    for (int j = 0; j < kActCols / 2; ++j) {
      float a, b;
      unpack2(f[j], a, b);
      pk[j] = pack_bf16x2(fmaxf(a, 0.f), fmaxf(b, 0.f));
    }
  }
  const int c0 = part * kActCols;                       // first column inside the 128-wide pair
  const uint32_t row = sb + OFF_O + (c0 >> 6) * kHidBytes + r * 128;
  const int u0 = (c0 & 63) >> 3;
  if (r < kS) {
#pragma unroll
    for (int u = 0; u < kActCols / 8; ++u)
      st_shared_v4(row + (((u0 + u) ^ (r & 7)) << 4), pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
  }
}

// =============================================================================================
// the persistent encoder kernel
// =============================================================================================
struct EncParams {
  char* x_images;             // [nseq][kXImageBytes]: residual stream images, replaced in place by the encoder output
  const TcLayer* layers;      // device table
  int num_layers;
  int activation;
  int64_t nseq;
  unsigned long long* timeline;   // diagnostics (device memory): (id << 48 | clock) records, 0-terminated; nullptr = off
};

// timeline events are recorded by block 0 only, for its second sequence, second layer (steady state): plain stores
// into device memory, MMA thread in slots [0,500), compute thread 0 in slots [500,1000)
__device__ __forceinline__ void tl_event(const EncParams& p, bool on, uint32_t id, uint32_t& n) {
#ifndef AFT_TC_TIMELINE
  (void)p; (void)on; (void)id; (void)n;   // compiled out: the bookkeeping costs registers the epilogues need
#else
  if (on) {
    unsigned long long* base = p.timeline + (id >= 200 ? 500 : 0);
    const unsigned long long t = clock64();
    ++n;                                        // register-resident count; slot 0 of each half mirrors it
    if (n < 500) { base[n] = ((unsigned long long)id << 48) | (t & 0xFFFFFFFFFFFFull); base[0] = n; }
  }
#endif
}
#ifdef AFT_TC_TIMELINE
#define AFT_TL_ON(expr) (expr)
#else
#define AFT_TL_ON(expr) false
#endif

// use counter of an mbarrier on one side of the protocol: wait()/done() walk the phases in order
struct Phase {
  uint32_t n = 0;
  __device__ __forceinline__ void wait(uint32_t bar) { mbar_wait(bar, n & 1); ++n; }
};

__global__ void __launch_bounds__(kTcThreads, 1) encoder_kernel(EncParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sb = smem_u32(smem_raw);
  if ((sb & 1023u) != 0) __trap();   // operand images need 1024-byte alignment and there is no room for slack
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t misc = sb + OFF_MISC + MISC_BARS;   // base of the mbarrier block
  const uint32_t miscb = sb + OFF_MISC;             // base of the MISC region (bias buffers, exchange arrays)

  if (threadIdx.x == 0) {
    const uint32_t commit_bars[] = {MB_VEC_FULL, MB_BIAS_FULL, MB_BIAS_FULL + 8, MB_X_FULL, MB_ATTN_DONE, MB_W_FULL, MB_W_FULL + 8, MB_W_FULL + 16, MB_W_FULL + 24,
                                    MB_W_EMPTY, MB_W_EMPTY + 8, MB_W_EMPTY + 16, MB_W_EMPTY + 24, MB_QKV_DONE, MB_S_DONE,
                                    MB_PV_DONE, MB_F1_DONE, MB_F2_DONE, MB_F2_DONE + 8, MB_F2_DONE + 16};
    const uint32_t warp_bars[] = {MB_X_FREE, MB_QKV_READY, MB_S_LOADED, MB_P_READY, MB_O_FREE, MB_O_FREE + 8,
                                  MB_F1_FREE, MB_HID_READY, MB_HID_READY + 8, MB_TAIL_MAX};
    for (uint32_t b : commit_bars) mbar_init(misc + b, 1);
    for (uint32_t b : warp_bars) mbar_init(misc + b, kComputeWarps);
    for (uint32_t t = 0; t < 3; ++t) {
      mbar_init(sb + OFF_BAR2 + MB2_OUT_DONE + 8 * t, 1);
      mbar_init(sb + OFF_BAR2 + MB2_X1_READY + 8 * t, kComputeWarps);
      mbar_init(sb + OFF_BAR2 + MB2_X2_READY + 8 * t, kComputeWarps);
    }
    fence_mbar_init();
  }
  if (warp == kMmaWarp) { tmem_alloc(miscb + MISC_TMEM_PTR, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(miscb + MISC_TMEM_PTR));
  __syncthreads();   // the pointer slot aliases the softmax exchange area

  const int L = p.num_layers;

  if (warp >= kComputeWarps) {
    setmaxnreg_dec<kRegsCtrl>();
    if (warp == kProducerWarp && lane == 0) {
      // ----------------------------------------------------------------------------- producer
      uint32_t n_in = 0, n_ring = 0, n_seq = 0, n_attn = 0;
      for (int64_t seq = blockIdx.x; seq < p.nseq; seq += gridDim.x, ++n_seq) {
        if (n_seq > 0) mbar_wait_relaxed(misc + MB_X_FREE, (n_seq - 1) & 1);
        mbar_arrive_expect_tx(misc + MB_X_FULL, kXImageBytes);
        bulk_g2s(sb + OFF_X, p.x_images + seq * (int64_t)kXImageBytes, kXImageBytes, misc + MB_X_FULL);
        // the image of this CTA's next sequence travels HBM -> L2 while this one is processed (the load above is exposed
        // at every sequence boundary: the residual image has no second buffer)
        if (seq + gridDim.x < p.nseq) bulk_prefetch_l2(p.x_images + (seq + gridDim.x) * (int64_t)kXImageBytes, kXImageBytes);
        for (int l = 0; l < L; ++l) {
          const TcLayer& W = p.layers[l];
          // the in_proj slot: four head slices per layer, then (FFN) the second K-chunk of each W1 pair
          auto fill_w = [&](const char* src, uint32_t bytes) {
            if (n_in > 0) mbar_wait_relaxed(misc + MB_W_EMPTY, (n_in - 1) & 1);
            mbar_arrive_expect_tx(misc + MB_W_FULL, bytes);
            bulk_g2s(sb + OFF_W, src, bytes, misc + MB_W_FULL);
            ++n_in;
          };
          auto fill_ring = [&](const char* src) {
            const int slot = n_ring % 3;
            const uint32_t fill = n_ring / 3;
            if (fill > 0) mbar_wait_relaxed(misc + MB_W_EMPTY + 8 * (1 + slot), (fill - 1) & 1);
            mbar_arrive_expect_tx(misc + MB_W_FULL + 8 * (1 + slot), kRingSlot);
            bulk_g2s(sb + OFF_QKV + slot * kRingSlot, src, kRingSlot, misc + MB_W_FULL + 8 * (1 + slot));
            ++n_ring;
          };
          for (int g = 0; g < 4; ++g) {
            fill_w(reinterpret_cast<const char*>(W.w_in) + g * kWInSlice, kWInSlice);
            // bias buffer g & 1 was last read by the epilogue of head g-2, which finished before QKV(g-1) was even issued
            mbar_arrive_expect_tx(misc + MB_BIAS_FULL + 8 * (g & 1), kQkvBiasBytes);
            bulk_g2s(miscb + MISC_QKV_BIAS + (g & 1) * kQkvBiasBytes, W.b_in + g * 96, kQkvBiasBytes, misc + MB_BIAS_FULL + 8 * (g & 1));
          }
          mbar_wait_relaxed(misc + MB_ATTN_DONE, n_attn & 1);   // Q/K/V images dead: the ring may overwrite them
          ++n_attn;
          mbar_arrive_expect_tx(misc + MB_VEC_FULL, kVecBlockBytes);
          bulk_g2s(sb + OFF_VEC, W.b_in + kVecBlock, kVecBlockBytes, misc + MB_VEC_FULL);
          // ring order: Wout k0, Wout k1 | W1 pair 0 k0 | W2 c0, W2 c1 | W1 pair 1 k0 | W2 c2, W2 c3; the k1 halves of
          // the W1 pairs go to the (idle) in_proj slot, so that a whole pair plus the W2 chunks in use are resident together
          const char* wout = reinterpret_cast<const char*>(W.w_out);
          const char* wl1 = reinterpret_cast<const char*>(W.w_l1);
          const char* wl2 = reinterpret_cast<const char*>(W.w_l2);
          fill_ring(wout);
          fill_ring(wout + kRingSlot);
          fill_ring(wl1);
          fill_w(wl1 + kRingSlot, kRingSlot);
          fill_ring(wl2);
          fill_ring(wl2 + kRingSlot);
          fill_ring(wl1 + 2 * kRingSlot);
          fill_w(wl1 + 3 * kRingSlot, kRingSlot);
          fill_ring(wl2 + 2 * kRingSlot);
          fill_ring(wl2 + 3 * kRingSlot);
        }
      }
    } else if (warp == kMmaWarp) {
      // ----------------------------------------------------------------------------- MMA issuer
      // The whole warp runs the schedule converged (all lanes poll the barriers, addresses stay warp-uniform and live in
      // uniform registers); only the tcgen05.mma / tcgen05.commit instructions are predicated on the elected lane.
      const bool el = elect_one();
      Phase x_full, qkv_ready, s_loaded, p_ready;
      const uint32_t bar2 = sb + OFF_BAR2;
      uint32_t n_in = 0, ring_base = 0, n_pv = 0, n_f1 = 0, n_layers_done = 0, tl_n = 0;
      // ring entry `idx` (global index): wait until it is resident, return its address; release = commit its empty barrier
      auto ring_wait = [&](uint32_t idx) -> uint32_t {
        mbar_wait(misc + MB_W_FULL + 8 * (1 + idx % 3), (idx / 3) & 1);
        tc_fence_after_sync();
        return sb + OFF_QKV + (idx % 3) * kRingSlot;
      };
      auto ring_release = [&](uint32_t idx) { mma_commit(misc + MB_W_EMPTY + 8 * (1 + idx % 3), el); };

      for (int64_t seq = blockIdx.x; seq < p.nseq; seq += gridDim.x) {
        x_full.wait(misc + MB_X_FULL);
        for (int l = 0; l < L; ++l, ++n_layers_done, ring_base += 8) {
          const bool tl = AFT_TL_ON(p.timeline != nullptr && blockIdx.x == 0 && seq == (int64_t)gridDim.x && l == 1 && lane == 0);
          // QKV projection of head g, row tiles [t0, t1); accumulators alias the S columns.  `first` waits for the weight
          // slice, `last` releases it and publishes the accumulators.
          auto issue_qkv = [&](int g, int t0, int t1, bool first, bool last) {
            if (first) {
              mbar_wait(misc + MB_W_FULL, n_in & 1);
              tc_fence_after_sync();
              tl_event(p, tl, 100 + g, tl_n);   // QKV(g) issue start
            }
            for (int t = t0; t < t1; ++t)
              issue_gemm_sw128(tmem, qkv_col(g, t), sb + OFF_X + t * 128 * 128, kXChunkBytes, sb + OFF_W, 96 * 128, 8, kIdescQkv, false, el);
            if (last) {
              mma_commit(misc + MB_W_EMPTY, el);
              mma_commit(misc + MB_QKV_DONE, el);
              tl_event(p, tl, 110 + g, tl_n);   // QKV(g) issued
              ++n_in;
            }
          };
          // Head 0: row tile t of X and the accumulator columns the tile's projection overwrites are free once the
          // previous LayerNorm2 has finished tiles 0..t (per-tile barriers, one completion per layer each).  Inside a
          // sequence the projection follows LayerNorm2 tile by tile; the first layer of a sequence starts from a new image.
          if (n_layers_done > 0 && l > 0) {
            for (int t = 0; t < 3; ++t) {
              mbar_wait(bar2 + MB2_X2_READY + 8 * t, (n_layers_done - 1) & 1);
              tc_fence_after_sync();
              issue_qkv(0, t, t + 1, t == 0, t == 2);
            }
          } else {
            if (n_layers_done > 0)
              for (int t = 0; t < 3; ++t) mbar_wait(bar2 + MB2_X2_READY + 8 * t, (n_layers_done - 1) & 1);
            tc_fence_after_sync();
            issue_qkv(0, 0, 3, true, true);
          }
          for (int g = 0; g < 4; ++g) {
            // ---- attention of head g
            qkv_ready.wait(misc + MB_QKV_READY);
            tc_fence_after_sync();
            tl_event(p, tl, 120 + g, tl_n);   // QKV_READY seen
            issue_scores(tmem, sb, 0, el);
            mma_commit(misc + MB_S_DONE, el);
            for (int t = 0; t < 3; ++t, ++n_pv) {
              s_loaded.wait(misc + MB_S_LOADED);      // S(t) is in registers
              tc_fence_after_sync();
              tl_event(p, tl, 130 + t, tl_n);   // S_LOADED(t) seen
              if (t == 0) { issue_scores(tmem, sb, 1, el); mma_commit(misc + MB_S_DONE, el); }
              else if (t == 1) { issue_scores_tail(tmem, sb, el); mma_commit(misc + MB_S_DONE, el); }
              // the tail scores fill all score columns: row tiles 1 and 2 of the next head's projection follow their
              // read-out and run under the tail's softmax (tile 0 was issued into the P columns, see below).  Measured:
              // holding tile 2 back until P.V of the tail has been issued is slower (57.5 vs 56.6 ms per 16384 estimates).
              else if (g < 3) issue_qkv(g + 1, 1, 3, false, true);
              p_ready.wait(misc + MB_P_READY);         // P(t) is in TMEM
              // O accumulator n_pv & 1 was last used by P.V #(n_pv - 2): its epilogue must have read it out
              if (n_pv >= 2) mbar_wait(misc + MB_O_FREE + 8 * (n_pv & 1), ((n_pv >> 1) - 1) & 1);
              tc_fence_after_sync();
              tl_event(p, tl, 140 + t, tl_n);   // P_READY(t) seen, P.V(t) issue start
              if (t == 2) issue_pv_tail(tmem, sb, n_pv & 1, el); else issue_pv(tmem, sb, n_pv & 1, el);
              mma_commit(misc + MB_PV_DONE, el);
              tl_event(p, tl, 150 + t, tl_n);   // P.V(t) issued
              if (t == 1 && g < 3) {
                // row tile 0 of the next head's projection -> P columns: P.V(1) (the last reader of P in TMEM for this head)
                // must have completed; nothing else is pending for this warp until the tail's scores have been read
                mbar_wait(misc + MB_PV_DONE, n_pv & 1);
                tc_fence_after_sync();
                issue_qkv(g + 1, 0, 1, true, false);
              }
              if (g == 3 && t == 2) mma_commit(misc + MB_ATTN_DONE, el);
            }
          }
          // ---- out_proj: needs every O epilogue of the layer (O image complete, P columns free)
          {
            // the epilogues of the last two P.V (#n_pv-2, #n_pv-1): O image complete, P columns free
            mbar_wait(misc + MB_O_FREE + 8 * (n_pv & 1), ((n_pv >> 1) - 1) & 1);
            mbar_wait(misc + MB_O_FREE + 8 * ((n_pv + 1) & 1), (((n_pv + 1) >> 1) - 1) & 1);
            tc_fence_after_sync();
            tl_event(p, tl, 160, tl_n);   // out_proj issue start
            const uint32_t w0 = ring_wait(ring_base + 0), w1 = ring_wait(ring_base + 1);
            for (int t = 0; t < 3; ++t) {   // tile-major: LayerNorm1 of tile 0 starts while tiles 1 and 2 are still in the pipe
              issue_gemm_sw128(tmem, TM_OUT + t * 128, sb + OFF_O + t * 128 * 128, 0, w0, 0, 4, kIdescN128, false, el);
              issue_gemm_sw128(tmem, TM_OUT + t * 128, sb + OFF_O + kXChunkBytes + t * 128 * 128, 0, w1, 0, 4, kIdescN128, true, el);
              mma_commit(bar2 + MB2_OUT_DONE + 8 * t, el);
            }
            ring_release(ring_base + 0);
            ring_release(ring_base + 1);
            tl_event(p, tl, 161, tl_n);   // out_proj issued
          }
          // ---- FFN.  FFN1 runs as N = 128 MMAs over pairs of hidden chunks (tile k = 3 pr + t, single accumulator tile in
          // TMEM); the FFN2 partial products of row tile t are issued as soon as the GELU of that tile is stored, right
          // behind the next FFN1 tile.  W1 pair: K-chunk 0 in a ring slot, K-chunk 1 in the in_proj slot.
          tl_event(p, tl, 170, tl_n);   // FFN start
          {
            constexpr uint32_t kHi = (uint32_t)(desc_k_sw128_const() >> 32);
            auto desc128 = [&](uint32_t saddr) -> uint32_t { return (uint32_t)desc_k_sw128_const() | ((saddr >> 4) & 0x3FFF); };
            auto issue_f2 = [&](int j) {   // FFN2 partial products of tile j % 3 over the two hidden chunks of pair j / 3
              const int pj = j / 3, tj = j - 3 * pj;
              // FFN tile J = 6 * layers_done + j of this CTA: barrier J & 1 (= j & 1), its completion number J >> 1
              mbar_wait(misc + MB_HID_READY + 8 * (j & 1), ((6 * n_layers_done + j) >> 1) & 1);
              tc_fence_after_sync();
              const uint32_t w2a = ring_wait(ring_base + 3 + 3 * pj), w2b = ring_wait(ring_base + 4 + 3 * pj);
              const uint32_t d = tmem + TM_OUT + tj * 128;
#pragma unroll
              for (int cc = 0; cc < 2; ++cc) {
                const uint32_t a_lo = desc128(sb + OFF_O + cc * kHidBytes + tj * 128 * 128), b_lo = desc128(cc == 0 ? w2a : w2b);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  mma_ss(d, ((uint64_t)kHi << 32) | (a_lo + ks * 2), ((uint64_t)kHi << 32) | (b_lo + ks * 2), kIdescN128,
                         pj > 0 || cc > 0 || ks > 0, el);
              }
              mma_commit(misc + MB_F2_DONE + 8 * tj, el);
              if (tj == 2) { ring_release(ring_base + 3 + 3 * pj); ring_release(ring_base + 4 + 3 * pj); }
              tl_event(p, tl, 190 + j, tl_n);   // FFN2(j) issued
            };
            uint32_t w1a = 0, w1b = 0;
            for (int k = 0; k < 6; ++k, ++n_f1) {
              const int pr = k / 3, t = k - 3 * pr;
              if (t == 0) {
                w1a = ring_wait(ring_base + 2 + 3 * pr);
                mbar_wait(misc + MB_W_FULL, n_in & 1);
                tc_fence_after_sync();
                w1b = sb + OFF_W;
              }
              if (pr == 0) mbar_wait(bar2 + MB2_X1_READY + 8 * t, n_layers_done & 1);   // LayerNorm1 rows of this tile are in X
              if (n_f1 >= 1) mbar_wait(misc + MB_F1_FREE, (n_f1 - 1) & 1);
              tc_fence_after_sync();
              const uint32_t a0 = desc128(sb + OFF_X + t * 128 * 128), a1 = desc128(sb + OFF_X + kXChunkBytes + t * 128 * 128);
              const uint32_t b0 = desc128(w1a), b1 = desc128(w1b);
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)
                mma_ss(tmem + TM_F1, ((uint64_t)kHi << 32) | ((ks < 4 ? a0 : a1) + (ks & 3) * 2),
                       ((uint64_t)kHi << 32) | ((ks < 4 ? b0 : b1) + (ks & 3) * 2), kIdescN128, ks > 0, el);
              mma_commit(misc + MB_F1_DONE, el);
              tl_event(p, tl, 180 + k, tl_n);   // FFN1(k) issued
              if (t == 2) {   // the pair's weights are free once these MMAs have completed
                ring_release(ring_base + 2 + 3 * pr);
                mma_commit(misc + MB_W_EMPTY, el);
                ++n_in;
              }
              if (k >= 1) issue_f2(k - 1);
            }
            issue_f2(5);
          }
        }
      }
    }
  } else {
    // ----------------------------------------------------------------------------- compute warps
    setmaxnreg_inc<kRegsCompute>();
    const int q = warp & 3, part = warp >> 2;
    const int rt = q * 32 + lane;                // row inside a 128-row tile
    const bool tile2_active = (q == 0);          // third row tile: only rows 256..287 exist
    // Barrier parities are derived from three counters (sequences, layers, heads done by this CTA): every barrier of the
    // protocol completes a fixed number of phases per head / layer / sequence.
    uint32_t n_seq = 0, n_layer = 0, n_head = 0, tl_n = 0;
    const uint32_t xmax_row = miscb + MISC_XMAX + rt * 4, xsum_row = miscb + MISC_XSUM + rt * 4;   // + part * 512 per warpgroup
    const uint32_t qkv_bias = miscb + MISC_QKV_BIAS;   // [2][96] f32
    const uint32_t vec = sb + OFF_VEC;                 // the layer's 1024-float vector block

    const int nseq = (int)p.nseq;   // one launch never carries more than 2^31 sequences (aft_api.cu chunks the batch)
#pragma unroll 1
    for (int seq = blockIdx.x; seq < nseq; seq += gridDim.x, ++n_seq) {
      mbar_wait(misc + MB_X_FULL, n_seq & 1);   // the residual image is read with generic loads by the LayerNorm epilogues
#pragma unroll 1
      for (int l = 0; l < L; ++l, ++n_layer) {
        const bool tl = AFT_TL_ON(p.timeline != nullptr && blockIdx.x == 0 && seq == (int)gridDim.x && l == 1 && threadIdx.x == 0);
#pragma unroll 1
        for (int g = 0; g < 4; ++g, ++n_head) {
          // ---- QKV epilogue of head g: P.V / score tile #k of this CTA has k = 3 * n_head + t, so k & 1 == (n_head + t) & 1
          tl_event(p, tl, 200 + g, tl_n);   // waiting QKV_DONE
          mbar_wait(misc + MB_BIAS_FULL + 8 * (g & 1), (n_head >> 1) & 1);   // in_proj bias of this head (buffer g & 1)
          const QkvBias qb = epi_qkv_bias(qkv_bias + (g & 1) * kQkvBiasBytes, part);
          mbar_wait(misc + MB_QKV_DONE, n_head & 1);
          tc_fence_after_sync();
          tl_event(p, tl, 210 + g, tl_n);   // QKV_DONE seen
          epi_qkv_pair(tmem, sb, qb, g, q, part, lane);
          if (tile2_active) epi_qkv(tmem, sb, qb, g, 2, q, part, lane);
          tc_fence_before_sync();
          fence_proxy_async_smem();
          warp_arrive(misc + MB_QKV_READY, lane);
          tl_event(p, tl, 220 + g, tl_n);   // QKV epilogue done
          // ---- softmax tiles; the O epilogue of tile t-1 runs after P(t) has been handed to the tensor core
          float inv_prev = 0.f;
#pragma unroll 1
          for (int t = 0; t < 4; ++t) {
            if (t < 2) {
              mbar_wait(misc + MB_S_DONE, (n_head + t) & 1);
              tc_fence_after_sync();
              tl_event(p, tl, 230 + t, tl_n);   // S_DONE(t) seen
              // the score row lives in registers from here to the P store: defined and consumed inside one block
              float v[kSmCols];
              float m = softmax_load(tmem, q, part, v);
              st_shared_f32(xmax_row + part * 512, m);
              tc_fence_before_sync();
              warp_arrive(misc + MB_S_LOADED, lane);
              tl_event(p, tl, 240 + t, tl_n);   // S(t) loaded
              named_bar_sync(1 + q, 32 * kParts);                          // exchange the partial row maxima
#pragma unroll
              for (int pp = 0; pp < kParts; ++pp) m = fmaxf(m, ld_shared_f32(xmax_row + pp * 512));
              // P.V(t-1) was issued a score load ago: it has all but always consumed P by now.  Its O accumulator is
              // fetched here and written out after the exponentials (the TMEM round trip hides under them).
              uint32_t oa[kOCols];
              if (t > 0) {
                mbar_wait(misc + MB_PV_DONE, (n_head + t - 1) & 1);
                tc_fence_after_sync();
                tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_O + ((n_head + t - 1) & 1) * 32 + part * kOCols, oa);
              }
              tl_event(p, tl, 260 + t, tl_n);   // PV_DONE(t-1) seen
              const float sum = softmax_exp_store(tmem, q, part, v, m);
              tl_event(p, tl, 250 + t, tl_n);   // exponentials done, P stored
              st_shared_f32(xsum_row + part * 512, sum);
              tc_fence_before_sync();
              warp_arrive(misc + MB_P_READY, lane);
              tl_event(p, tl, 270 + t, tl_n);   // P(t) stored
              if (t > 0) {
                tmem_wait_ld();
                epi_o_store(sb, g, t - 1, inv_prev, q, part, lane, oa);
              }
            } else if (t == 2) {
              mbar_wait(misc + MB_S_DONE, (n_head + 2) & 1);
              tc_fence_after_sync();
              tl_event(p, tl, 232, tl_n);       // tail S seen
              softmax_tail(tmem, sb, miscb, misc + MB_S_LOADED, misc + MB_TAIL_MAX, n_head & 1, q, part, lane);
              fence_proxy_async_smem();         // P is read by the tensor core
              // P.V(1) (long finished): waited for before the arrival so that the PV_DONE barrier can never run two
              // phases ahead of a waiter; its O accumulator is read out right below
              mbar_wait(misc + MB_PV_DONE, (n_head + 1) & 1);
              tc_fence_after_sync();
              warp_arrive(misc + MB_P_READY, lane);
              tl_event(p, tl, 272, tl_n);       // tail P stored
            } else {
              mbar_wait(misc + MB_PV_DONE, (n_head + 2) & 1);
              tc_fence_after_sync();
            }
            if (t > 0) {
              if (t == 2) epi_o(tmem, sb, g, 1, (n_head + 1) & 1, inv_prev, q, part, lane);
              else if (t == 3 && q < 2) epi_o_tail(tmem, sb, miscb, g, (n_head + 2) & 1, q, part, lane);
              tc_fence_before_sync();
              fence_proxy_async_smem();
              warp_arrive(misc + MB_O_FREE + 8 * ((n_head + t - 1) & 1), lane);
            }
            if (t < 2) {
              named_bar_sync(1 + q, 32 * kParts);                          // exchange the partial row sums
              float l_row = 0.f;
#pragma unroll
              for (int pp = 0; pp < kParts; ++pp) l_row += ld_shared_f32(xsum_row + pp * 512);
              inv_prev = rcp_approx(l_row);
            }
          }
        }
        // ---- out_proj epilogue: + bias + residual -> LayerNorm1 -> X
        tl_event(p, tl, 280, tl_n);   // waiting OUT_DONE
        mbar_wait(misc + MB_VEC_FULL, n_layer & 1);   // this layer's bias / LayerNorm vectors are in shared memory
#pragma unroll 1
        for (int t = 0; t < 3; ++t) {   // per row tile: out_proj accumulators in -> LayerNorm1 rows out (FFN1 of the tile may start)
          if (t < 2 || tile2_active) {
            mbar_wait(sb + OFF_BAR2 + MB2_OUT_DONE + 8 * t, n_layer & 1);
            tc_fence_after_sync();
            epi_ln(tmem, sb, vec, 1, t, q, part, lane, t == 1 ? sb + OFF_LN1_XCHG : miscb + MISC_XMAX, nullptr, -1);
          }
          tc_fence_before_sync();
          fence_proxy_async_smem();
          warp_arrive(sb + OFF_BAR2 + MB2_X1_READY + 8 * t, lane);
        }
        tl_event(p, tl, 282, tl_n);   // LayerNorm1 done
        // ---- FFN1 epilogues: bias + GELU -> hidden images.  Tile k = 3 pr + t of this layer: F1_DONE / F1_FREE / HID_READY
        // complete six times per layer (phase parity k & 1), F2_DONE[t] twice (pair 0: rows free again, pair 1: final).
#pragma unroll 1
        for (int k = 0; k < 6; ++k) {
          const int pr = k >= 3 ? 1 : 0, t = k - 3 * pr;
          const bool active = t < 2 || tile2_active;
          mbar_wait(misc + MB_F1_DONE, k & 1);
          tc_fence_after_sync();
          tl_event(p, tl, 300 + k, tl_n);   // F1_DONE(k) seen
          if (active) {   // accumulators defined and consumed inside one branch (see the softmax tiles)
            f32x2 f[kActCols / 2];
            act_load(tmem, vec, pr, q, part, f);
            tc_fence_before_sync();
            warp_arrive(misc + MB_F1_FREE, lane);
            // the hidden rows of this tile still feed the FFN2 partial products of pair 0
            if (pr == 1) mbar_wait(misc + MB_F2_DONE + 8 * t, 0);
            act_store(sb, t, p.activation, q, part, lane, f);
          } else {
            tc_fence_before_sync();
            warp_arrive(misc + MB_F1_FREE, lane);
          }
          tl_event(p, tl, 320 + k, tl_n);   // GELU(k) stored
          fence_proxy_async_smem();
          warp_arrive(misc + MB_HID_READY + 8 * (k & 1), lane);
        }
        // ---- linear2 epilogue: + bias + residual -> LayerNorm2 -> X (+ fp32 result after the last layer)
        tl_event(p, tl, 340, tl_n);   // LayerNorm2 start
#pragma unroll 1
        for (int t = 0; t < 3; ++t) {   // per row tile: second completion of the tile's F2_DONE in this layer = final accumulators
          if (t < 2 || tile2_active) {
            mbar_wait(misc + MB_F2_DONE + 8 * t, 1);
            tc_fence_after_sync();
            epi_ln(tmem, sb, vec, 2, t, q, part, lane, t == 1 ? sb + OFF_LN_XCHG : miscb + MISC_XMAX, nullptr, -1);
          }
          tc_fence_before_sync();
          fence_proxy_async_smem();
          warp_arrive(sb + OFF_BAR2 + MB2_X2_READY + 8 * t, lane);
        }
        if (l == L - 1) {
          // The encoder output replaces the sequence's input image in global memory: once every compute warp has written
          // its LayerNorm2 rows, the X image is copied out with fully coalesced 16-byte accesses (512 B per warp
          // instruction; storing from the LayerNorm registers would touch 32 different 128-byte lines per instruction).
          named_bar_sync(10, 32 * kComputeWarps);
          char* dst = p.x_images + seq * (int64_t)kXImageBytes;
#pragma unroll
          for (int i = 0; i < kXImageBytes / 16 / (32 * kComputeWarps); ++i) {
            const uint32_t off = (uint32_t)(i * 32 * kComputeWarps + threadIdx.x) * 16;
            *reinterpret_cast<uint4*>(dst + off) = ld_shared_v4(sb + OFF_X + off);
          }
          warp_arrive(misc + MB_X_FREE, lane);
        }
        tl_event(p, tl, 341, tl_n);   // LayerNorm2 done
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}

// =============================================================================================
// weight packing: fp32 [N, K] row-major -> bf16 operand image(s)
// =============================================================================================
// One thread per 16-byte unit.  The destination is a sequence of `nblocks` images, block b holding rows
// [row0 + b*row_stride, +rows) and columns [col0 + b*col_stride, +64*chunks) of the source; rows whose index
// (within the block) is < scale_rows are multiplied by `scale` (in_proj q rows).
__global__ void pack_image_kernel(const float* __restrict__ src, int ld, __nv_bfloat16* __restrict__ dst, int nblocks, int rows,
                                  int chunks, int row0, int row_stride, int col0, int col_stride, int scale_rows, float scale) {
  const int units_per_block = rows * chunks * 8;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nblocks * units_per_block) return;
  const int b = i / units_per_block, rem = i - b * units_per_block;
  const int chunk = rem / (rows * 8), rem2 = rem - chunk * rows * 8;
  const int r = rem2 >> 3, u = rem2 & 7;
  const float* s = src + (int64_t)(row0 + b * row_stride + r) * ld + col0 + b * col_stride + chunk * 64 + u * 8;
  const float sc = r < scale_rows ? scale : 1.0f;
  uint4 pk;
  pk.x = pack_bf16x2(s[0] * sc, s[1] * sc); pk.y = pack_bf16x2(s[2] * sc, s[3] * sc);
  pk.z = pack_bf16x2(s[4] * sc, s[5] * sc); pk.w = pack_bf16x2(s[6] * sc, s[7] * sc);
  char* d = reinterpret_cast<char*>(dst) + (int64_t)b * rows * chunks * 128 + image_offset(r, chunk * 64 + u * 8, rows);
  *reinterpret_cast<uint4*>(d) = pk;
}

// in_proj head slice g: rows [q_g | k_g | v_g] gathered from rows g*32, 128+g*32, 256+g*32
__global__ void pack_inproj_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, float qscale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // one 16-byte unit: 4 slices x 2 chunks x 96 rows x 8 units
  if (i >= 4 * 2 * 96 * 8) return;
  const int g = i / 1536, rem = i - g * 1536;
  const int chunk = rem / 768, rem2 = rem - chunk * 768;
  const int r = rem2 >> 3, u = rem2 & 7;
  const int part = r >> 5, rr = r & 31;
  const float* s = w + (int64_t)(part * 128 + g * 32 + rr) * kD + chunk * 64 + u * 8;
  const float sc = part == 0 ? qscale : 1.0f;
  uint4 pk;
  pk.x = pack_bf16x2(s[0] * sc, s[1] * sc); pk.y = pack_bf16x2(s[2] * sc, s[3] * sc);
  pk.z = pack_bf16x2(s[4] * sc, s[5] * sc); pk.w = pack_bf16x2(s[6] * sc, s[7] * sc);
  char* d = reinterpret_cast<char*>(dst) + (int64_t)g * kWInSlice + image_offset(r, chunk * 64 + u * 8, 96);
  *reinterpret_cast<uint4*>(d) = pk;
}

__global__ void pack_vec_kernel(LayerPackF32 L, float* __restrict__ dst, float qscale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kVecPerLayer) return;
  float v;
  if (i < kVecBlock) {            // [head g][q32 | k32 | v32]
    const int g = i / 96, j = i - g * 96, mat = j >> 5, c = j & 31;
    v = L.in_b[mat * 128 + g * 32 + c] * (mat == 0 ? qscale : 1.0f);
  } else {
    const int b = i - kVecBlock;
    if (b < kVecBL1) v = L.out_b[b - kVecBOut];
    else if (b < kVecBL2) v = L.l1_b[b - kVecBL1];
    else if (b < kVecN1W) v = L.l2_b[b - kVecBL2];
    else if (b < kVecN1B) v = L.n1_w[b - kVecN1W];
    else if (b < kVecN2W) v = L.n1_b[b - kVecN1B];
    else if (b < kVecN2B) v = L.n2_w[b - kVecN2W];
    else v = L.n2_b[b - kVecN2B];
  }
  dst[i] = v;
}

unsigned long long* g_timeline_dev = nullptr;   // diagnostics timeline buffer (device), armed by aft_selftest(102)
unsigned long long* g_timeline_arm = nullptr;
unsigned long long* g_timeline_host = nullptr;

constexpr size_t kLayerImageBytes = 4 * kWInSlice + 32768 + 65536 + 65536;   // 262,144

}  // namespace

// =============================================================================================
// host side
// =============================================================================================
bool tc_weights_alloc(TcWeights& w, int num_layers) {
  w.num_layers = num_layers;
  w.layers.assign(num_layers, TcLayer{});
  // arena: per layer the operand images + the epilogue vectors; then the device copy of the table
  const size_t per_layer = kLayerImageBytes + kVecPerLayer * sizeof(float);
  const size_t conv_bytes = (conv_tc_pack_bytes() + 255) / 256 * 256;
  w.arena_bytes = num_layers * per_layer + (num_layers * sizeof(TcLayer) + 255) / 256 * 256 + 2 * conv_bytes + 1024;
  if (cudaMalloc(&w.arena, w.arena_bytes) != cudaSuccess) {
    set_error("tc_weights_alloc: cudaMalloc(%zu) failed: %s", w.arena_bytes, cudaGetErrorString(cudaGetLastError()));
    w.arena = nullptr;
    return false;
  }
  char* base = static_cast<char*>(w.arena);
  for (int l = 0; l < num_layers; ++l) {
    char* p = base + l * kLayerImageBytes;
    TcLayer& T = w.layers[l];
    T.w_in = reinterpret_cast<const __nv_bfloat16*>(p);
    T.w_out = reinterpret_cast<const __nv_bfloat16*>(p + 4 * kWInSlice);
    T.w_l1 = reinterpret_cast<const __nv_bfloat16*>(p + 4 * kWInSlice + 32768);
    T.w_l2 = reinterpret_cast<const __nv_bfloat16*>(p + 4 * kWInSlice + 32768 + 65536);
    const float* v = reinterpret_cast<const float*>(base + num_layers * kLayerImageBytes) + l * kVecPerLayer;
    T.b_in = v;
    const float* blk = v + kVecBlock;
    T.b_out = blk + kVecBOut; T.b_l1 = blk + kVecBL1; T.b_l2 = blk + kVecBL2;
    T.n1_w = blk + kVecN1W; T.n1_b = blk + kVecN1B; T.n2_w = blk + kVecN2W; T.n2_b = blk + kVecN2B;
  }
  w.layers_dev = reinterpret_cast<TcLayer*>(base + num_layers * per_layer);
  w.conv_front = base + num_layers * per_layer + (num_layers * sizeof(TcLayer) + 255) / 256 * 256;
  w.conv_head = static_cast<char*>(w.conv_front) + conv_bytes;
  return true;
}

void tc_weights_free(TcWeights& w) {
  if (w.arena) cudaFree(w.arena);
  w.arena = nullptr;
}

bool tc_weights_pack(TcWeights& w, const std::vector<LayerPackF32>& src, const ConvPack& enh, const ConvPack& refine, cudaStream_t st) {
  if (!conv_tc_pack(enh, w.conv_front, st) || !conv_tc_pack(refine, w.conv_head, st)) return false;
  const float qscale = 1.4426950408889634f / sqrtf((float)kDh);   // log2(e) / sqrt(dh): softmax runs on exp2
  for (int l = 0; l < w.num_layers; ++l) {
    const LayerPackF32& S = src[l];
    const TcLayer& T = w.layers[l];
    auto bf = [](const __nv_bfloat16* p) { return const_cast<__nv_bfloat16*>(p); };
    pack_inproj_kernel<<<(4 * 2 * 96 * 8 + 255) / 256, 256, 0, st>>>(S.in_w, bf(T.w_in), qscale);
    // out_proj: one image, 128 rows, K = 128 (2 chunks)
    pack_image_kernel<<<(128 * 2 * 8 + 255) / 256, 256, 0, st>>>(S.out_w, kD, bf(T.w_out), 1, 128, 2, 0, 0, 0, 0, 0, 1.f);
    // linear1: 4 images of 64 rows, K = 128
    pack_image_kernel<<<(2 * 128 * 2 * 8 + 255) / 256, 256, 0, st>>>(S.l1_w, kD, bf(T.w_l1), 2, 128, 2, 0, 128, 0, 0, 0, 1.f);
    // linear2: 4 images of 128 rows, one K-chunk each (columns 64c .. 64c+63 of the [128, 256] matrix)
    pack_image_kernel<<<(4 * 128 * 1 * 8 + 255) / 256, 256, 0, st>>>(S.l2_w, kFF, bf(T.w_l2), 4, 128, 1, 0, 0, 0, 64, 0, 1.f);
    pack_vec_kernel<<<(kVecPerLayer + 255) / 256, 256, 0, st>>>(S, const_cast<float*>(T.b_in), qscale);
    count_launch(5);
  }
  if (cudaMemcpyAsync(w.layers_dev, w.layers.data(), w.num_layers * sizeof(TcLayer), cudaMemcpyHostToDevice, st) != cudaSuccess) {
    set_error("tc_weights_pack: table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    return false;
  }
  return check_launch("tc_weights_pack");
}

namespace {
size_t align_up_sz(size_t v, size_t a) { return (v + a - 1) / a * a; }
}

size_t tc_workspace_bytes(int64_t bc) {
  const size_t nseq = 2 * (size_t)bc;
  return align_up_sz(nseq * kPix * sizeof(float), 1024) + align_up_sz(nseq * (size_t)kXImageBytes, 1024) +
         align_up_sz((size_t)bc * 3 * 2 * kS * sizeof(float), 1024);   // enhanced images | X images | adaptive features
}

bool tc_forward_chunk(const TcWeights& w, const FrontPack& front, const HeadPack& head, int activation, int sm_count,
                      const float2* pilots, const float* snr, const float* ds, const float* dop, const OutDst& out,
                      int64_t nsamples, void* workspace, cudaStream_t st, TcProfileHook hook) {
  auto mark = [&]() { if (hook.mark) hook.mark(hook.ctx, st); };
  const int64_t nseq = 2 * nsamples;
  char* ws = static_cast<char*>(workspace);
  float* enh = reinterpret_cast<float*>(ws);
  char* ximg = ws + align_up_sz(nseq * kPix * sizeof(float), 1024);
  float* zbuf = reinterpret_cast<float*>(ximg + align_up_sz(nseq * (size_t)kXImageBytes, 1024));
  mark();
  if (!launch_frontend_tc(front, w.conv_front, pilots, snr, ds, dop, zbuf, enh, reinterpret_cast<__nv_bfloat16*>(ximg), nsamples, sm_count, st)) return false;
  if (cudaFuncSetAttribute(encoder_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes) != cudaSuccess) {
    set_error("encoder_kernel: cannot opt in to %u bytes of shared memory: %s", kTcSmemBytes, cudaGetErrorString(cudaGetLastError()));
    return false;
  }
  EncParams ep;
  ep.x_images = ximg;
  ep.layers = w.layers_dev;
  ep.num_layers = w.num_layers;
  ep.activation = activation;
  ep.nseq = nseq;
  ep.timeline = g_timeline_arm;
  const unsigned grid = (unsigned)(nseq < sm_count ? nseq : sm_count);
  mark();
  encoder_kernel<<<grid, kTcThreads, kTcSmemBytes, st>>>(ep);
  count_launch();
  if (!check_launch("encoder_kernel")) return false;
  mark();
  const bool ok = launch_head_tc(head, w.conv_head, ximg, enh, out, nsamples, sm_count, st);
  mark();
  return ok;
}

// =============================================================================================
// self tests of the tcgen05 building blocks (aft_selftest)
// =============================================================================================
namespace {

// which = 0: D[128,96] = A[128 rows of a 288-row X image, K=128] . B[96 rows, K=128]^T   (SW128 K-major both)
__global__ void __launch_bounds__(128, 1) selftest_gemm_kernel(const char* a_img, const char* b_img, float* d_out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar = sb + 110592, tptr = bar + 16, bar2 = bar + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_init(bar2, 1); fence_mbar_init(); }
  if (warp == 0) { tmem_alloc(tptr, 128); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(tptr));
  if (threadIdx.x == 0) {
    mbar_arrive_expect_tx(bar, kXImageBytes + kWInSlice);
    bulk_g2s(sb, a_img, kXImageBytes, bar);
    bulk_g2s(sb + kXImageBytes, b_img, kWInSlice, bar);
    mbar_wait(bar, 0);
    tc_fence_after_sync();
    // second row tile (rows 128..255) to exercise the tile offset
    issue_gemm_sw128(tmem, 0, sb + 128 * 128, kXChunkBytes, sb + kXImageBytes, 96 * 128, 8, kIdescQkv, false);
    mma_commit(bar2);
  }
  mbar_wait(bar2, 0);
  tc_fence_after_sync();
  const int row = warp * 32 + lane;
  for (int i = 0; i < 6; ++i) {
    uint32_t v[16];
    tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + i * 16, v);
    tmem_wait_ld();
    for (int j = 0; j < 16; ++j) d_out[row * 96 + i * 16 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

// which = 1, 2: one attention row tile with the production helpers: S = Q K^T (SW64), softmax -> P (TMEM), O = P V (MN-major)
__global__ void __launch_bounds__(kTcThreads, 1) selftest_attn_kernel(const char* qkv_img, float* s_out, float* o_out, int tile) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sb = smem_u32(smem_raw);
  if ((sb & 1023u) != 0) __trap();
  const uint32_t misc = sb + OFF_MISC + MISC_BARS, miscb = sb + OFF_MISC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(misc + MB_X_FULL, 1); mbar_init(misc + MB_S_DONE, 1); mbar_init(misc + MB_PV_DONE, 1);
    mbar_init(misc + MB_P_READY, kComputeWarps);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) { tmem_alloc(miscb + MISC_TMEM_PTR, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(miscb + MISC_TMEM_PTR));
  __syncthreads();
  if (warp >= kComputeWarps) {
    setmaxnreg_dec<kRegsCtrl>();
    if (warp == kMmaWarp && lane == 0) {
      mbar_arrive_expect_tx(misc + MB_X_FULL, 3 * kQkvPart);
      bulk_g2s(sb + OFF_QKV, qkv_img, 3 * kQkvPart, misc + MB_X_FULL);
      mbar_wait(misc + MB_X_FULL, 0);
      tc_fence_after_sync();
      issue_scores(tmem, sb, tile);
      mma_commit(misc + MB_S_DONE);
      mbar_wait(misc + MB_P_READY, 0);
      tc_fence_after_sync();
      issue_pv(tmem, sb, 1);
      mma_commit(misc + MB_PV_DONE);
    }
  } else {
    setmaxnreg_inc<kRegsCompute>();
    const int q = warp & 3, part = warp >> 2;
    const int rt = q * 32 + lane;
    const bool active = tile < 2 || q == 0;
    const uint32_t xmax_row = miscb + MISC_XMAX + rt * 4, xsum_row = miscb + MISC_XSUM + rt * 4;
    mbar_wait(misc + MB_S_DONE, 0);
    tc_fence_after_sync();
    float v[kSmCols];
    float m = 0.f, sum = 0.f;
    if (active) {
      m = softmax_load(tmem, q, part, v);
#pragma unroll
      for (int j = 0; j < kSmCols; ++j) s_out[rt * 288 + part * kSmCols + j] = v[j];   // raw scores (padding keys read -inf)
      st_shared_f32(xmax_row + part * 512, m);
    }
    named_bar_sync(1 + q, 32 * kParts);
    if (active) {
      for (int pp = 0; pp < kParts; ++pp) m = fmaxf(m, ld_shared_f32(xmax_row + pp * 512));
      sum = softmax_exp(v, m);
      softmax_store(tmem, q, part, v);
      st_shared_f32(xsum_row + part * 512, sum);
    }
    tc_fence_before_sync();
    warp_arrive(misc + MB_P_READY, lane);
    named_bar_sync(1 + q, 32 * kParts);
    mbar_wait(misc + MB_PV_DONE, 0);
    tc_fence_after_sync();
    if (active) {
      float l = 0.f;
      for (int pp = 0; pp < kParts; ++pp) l += ld_shared_f32(xsum_row + pp * 512);
      uint32_t a[kOCols];
      tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_O + 32 + part * kOCols, a);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < kOCols; ++j) o_out[rt * 32 + part * kOCols + j] = __uint_as_float(a[j]) / l;
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}

// which = 4: the tail tile (query rows 256..279) with the production helpers: S slices per lane quadrant, P image in
// shared memory, M = 64 P.V, store into the O image (head 0)
__global__ void __launch_bounds__(kTcThreads, 1) selftest_tail_kernel(const char* qkv_img, float* s_out, float* o_out) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sb = smem_u32(smem_raw);
  if ((sb & 1023u) != 0) __trap();
  const uint32_t misc = sb + OFF_MISC + MISC_BARS, miscb = sb + OFF_MISC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(misc + MB_X_FULL, 1); mbar_init(misc + MB_S_DONE, 1); mbar_init(misc + MB_PV_DONE, 1);
    mbar_init(misc + MB_P_READY, kComputeWarps); mbar_init(misc + MB_S_LOADED, kComputeWarps);
    mbar_init(misc + MB_TAIL_MAX, kComputeWarps);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) { tmem_alloc(miscb + MISC_TMEM_PTR, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(miscb + MISC_TMEM_PTR));
  __syncthreads();
  if (warp >= kComputeWarps) {
    setmaxnreg_dec<kRegsCtrl>();
    if (warp == kMmaWarp && lane == 0) {
      mbar_arrive_expect_tx(misc + MB_X_FULL, 3 * kQkvPart);
      bulk_g2s(sb + OFF_QKV, qkv_img, 3 * kQkvPart, misc + MB_X_FULL);
      mbar_wait(misc + MB_X_FULL, 0);
      tc_fence_after_sync();
      issue_scores_tail(tmem, sb);
      mma_commit(misc + MB_S_DONE);
      mbar_wait(misc + MB_P_READY, 0);
      tc_fence_after_sync();
      issue_pv_tail(tmem, sb, 1);
      mma_commit(misc + MB_PV_DONE);
    }
  } else {
    setmaxnreg_inc<kRegsCompute>();
    const int q = warp & 3, part = warp >> 2;
    mbar_wait(misc + MB_S_DONE, 0);
    tc_fence_after_sync();
    // raw scores: thread (q, part, lane) holds query 256 + lane and 16 or 24 keys of its quadrant's slice, 8 at a time
    const int nc = q == 0 ? 24 : 16, key0 = tail_key0(q) + part * nc;
    for (int c0 = 0; c0 < nc; c0 += 8) {
      uint32_t x[8];
      tmem_ld_cols(tmem + ((uint32_t)(q * 32) << 16) + TM_S + key0 + c0, x);
      tmem_wait_ld();
      for (int j = 0; j < 8; ++j) s_out[(key0 + c0 + j) * 32 + lane] = __uint_as_float(x[j]);
    }
    softmax_tail(tmem, sb, miscb, misc + MB_S_LOADED, misc + MB_TAIL_MAX, 0, q, part, lane);
    fence_proxy_async_smem();
    warp_arrive(misc + MB_P_READY, lane);
    mbar_wait(misc + MB_PV_DONE, 0);
    tc_fence_after_sync();
    if (q < 2) epi_o_tail(tmem, sb, miscb, 0, 1, q, part, lane);
    named_bar_sync(9, 32 * kComputeWarps);
    for (int i = threadIdx.x; i < 24 * 32; i += 32 * kComputeWarps) {
      const int r = 256 + i / 32, c = i % 32;
      unsigned short h;
      asm volatile("ld.shared.u16 %0, [%1];" : "=h"(h) : "r"(sb + OFF_O + r * 128 + (((c >> 3) ^ (r & 7)) << 4) + (c & 7) * 2));
      o_out[i] = __uint_as_float((uint32_t)h << 16);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}

float bf16_round_host(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u = (u + 0x7FFFu + ((u >> 16) & 1u)) & 0xFFFF0000u;
  float y;
  memcpy(&y, &u, 4);
  return y;
}
uint16_t bf16_bits_host(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
}
struct Lcg {
  uint64_t s;
  float next() {   // uniform in [-1, 1)
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    return (float)((s >> 40) & 0xFFFFFF) / 8388608.0f - 1.0f;
  }
};

}  // namespace

bool tc_selftest(int which, double* max_err, cudaStream_t st) {
  *max_err = -1.0;
  if (which >= 100) {
    // diagnostics: 100 = arm the wait-timeout channel (mapped host memory), 101 = print and clear its records
    static unsigned long long* host_buf = nullptr;
    if (which == 100) {
      if (!host_buf) {
        if (cudaHostAlloc(&host_buf, 64 * 16 * 8, cudaHostAllocMapped) != cudaSuccess) { set_error("diag: cudaHostAlloc failed"); return false; }
        memset(host_buf, 0, 64 * 16 * 8);
        unsigned long long* dev = nullptr;
        cudaHostGetDevicePointer(&dev, host_buf, 0);
        cudaMemcpyToSymbol(g_wait_diag, &dev, sizeof(dev));
      }
      *max_err = 0.0;
      return true;
    }
    if (which == 102) {   // arm the timeline (mapped host memory)
      if (!g_timeline_host) {
        g_timeline_host = static_cast<unsigned long long*>(malloc(1000 * 8));
        if (cudaMalloc(&g_timeline_dev, 1000 * 8) != cudaSuccess) { set_error("timeline: cudaMalloc failed"); return false; }
      }
      g_timeline_arm = g_timeline_dev;
      cudaMemset(g_timeline_dev, 0, 1000 * 8);
      *max_err = 0.0;
      return true;
    }
    if (which == 103) {   // dump "id clock" lines to stderr and disarm
      unsigned long long n_ev = 0;
      if (g_timeline_host && cudaMemcpy(g_timeline_host, g_timeline_dev, 1000 * 8, cudaMemcpyDeviceToHost) == cudaSuccess)
        for (int h = 0; h < 2; ++h)
          for (unsigned long long i = 1; i <= g_timeline_host[500 * h] && i < 500; ++i, ++n_ev)
            fprintf(stderr, "TL %llu %llu\n", g_timeline_host[500 * h + i] >> 48, g_timeline_host[500 * h + i] & 0xFFFFFFFFFFFFull);
      conv_tc_dump_timeline();
      g_timeline_arm = nullptr;
      *max_err = (double)n_ev;
      return true;
    }
    int n = 0;
    if (host_buf)
      for (int i = 0; i < 64 * 16; ++i)
        if (host_buf[i] >> 63) {
          const unsigned long long r = host_buf[i];
          if (n < 48)
            fprintf(stderr, "aft wait-timeout: block %llu thread %llu (warp %llu) parity %llu barrier@misc+%llu\n", (r >> 40) & 0x7FFFFF,
                    (r >> 24) & 0xFFFF, ((r >> 24) & 0xFFFF) >> 5, (r >> 16) & 0xFF, (r & 0xFFFF) & 1023);
          host_buf[i] = 0;
          ++n;
        }
    *max_err = n;
    return true;
  }
  Lcg rng{12345u + (uint64_t)which};
  if (which == 0) {
    std::vector<float> A(288 * 128), B(96 * 128);
    for (auto& v : A) v = bf16_round_host(rng.next());
    for (auto& v : B) v = bf16_round_host(rng.next());
    std::vector<uint16_t> ai(kXImageBytes / 2, 0), bi(kWInSlice / 2, 0);
    for (int r = 0; r < 288; ++r)
      for (int c = 0; c < 128; ++c) ai[(image_offset(r, c & ~7, kSPad) >> 1) + (c & 7)] = bf16_bits_host(A[r * 128 + c]);
    for (int r = 0; r < 96; ++r)
      for (int c = 0; c < 128; ++c) bi[(image_offset(r, c & ~7, 96) >> 1) + (c & 7)] = bf16_bits_host(B[r * 128 + c]);
    char *da = nullptr, *db = nullptr;
    float* dd = nullptr;
    if (cudaMalloc(&da, kXImageBytes) != cudaSuccess || cudaMalloc(&db, kWInSlice) != cudaSuccess ||
        cudaMalloc(&dd, 128 * 96 * sizeof(float)) != cudaSuccess) {
      set_error("selftest: cudaMalloc failed");
      return false;
    }
    cudaMemcpyAsync(da, ai.data(), kXImageBytes, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(db, bi.data(), kWInSlice, cudaMemcpyHostToDevice, st);
    const int smem = 110592 + 64 + 1024;
    cudaFuncSetAttribute(selftest_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    selftest_gemm_kernel<<<1, 128, smem, st>>>(da, db, dd);
    count_launch();
    std::vector<float> D(128 * 96);
    cudaMemcpyAsync(D.data(), dd, D.size() * sizeof(float), cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(da); cudaFree(db); cudaFree(dd);
    if (e != cudaSuccess) { set_error("selftest gemm: %s", cudaGetErrorString(e)); return false; }
    double worst = 0.0;
    for (int m = 0; m < 128; ++m)
      for (int n = 0; n < 96; ++n) {
        double ref = 0.0;
        for (int k = 0; k < 128; ++k) ref += (double)A[(128 + m) * 128 + k] * (double)B[n * 128 + k];
        worst = fmax(worst, fabs(ref - (double)D[m * 96 + n]));
      }
    *max_err = worst;
    return true;
  }
  if (which == 1 || which == 2) {
    const int tile = which == 1 ? 1 : 2;
    // Q, K, V [288][32] in SW64 images; values scaled so that scores spread over a few units (log2 domain)
    std::vector<float> Q(288 * 32), K(288 * 32), V(288 * 32);
    for (auto& v : Q) v = bf16_round_host(rng.next() * 1.5f);
    for (auto& v : K) v = bf16_round_host(rng.next() * 1.5f);
    for (auto& v : V) v = bf16_round_host(rng.next());
    std::vector<uint16_t> img(3 * kQkvPart / 2, 0);
    auto put = [&](int part, const std::vector<float>& M) {
      for (int r = 0; r < 288; ++r)
        for (int c = 0; c < 32; ++c) {
          const int u = c >> 3, sw = (r >> 1) & 3;
          img[(part * kQkvPart + r * 64 + ((u ^ sw) << 4)) / 2 + (c & 7)] = bf16_bits_host(M[r * 32 + c]);
        }
    };
    put(0, Q); put(1, K); put(2, V);
    char* di = nullptr;
    float *ds = nullptr, *dO = nullptr;
    if (cudaMalloc(&di, 3 * kQkvPart) != cudaSuccess || cudaMalloc(&ds, 128 * 288 * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&dO, 128 * 32 * sizeof(float)) != cudaSuccess) {
      set_error("selftest: cudaMalloc failed");
      return false;
    }
    cudaMemsetAsync(ds, 0, 128 * 288 * sizeof(float), st);
    cudaMemsetAsync(dO, 0, 128 * 32 * sizeof(float), st);
    cudaMemcpyAsync(di, img.data(), 3 * kQkvPart, cudaMemcpyHostToDevice, st);
    cudaFuncSetAttribute(selftest_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes);
    selftest_attn_kernel<<<1, kTcThreads, kTcSmemBytes, st>>>(di, ds, dO, tile);
    count_launch();
    std::vector<float> S(128 * 288), O(128 * 32);
    cudaMemcpyAsync(S.data(), ds, S.size() * sizeof(float), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(O.data(), dO, O.size() * sizeof(float), cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(di); cudaFree(ds); cudaFree(dO);
    if (e != cudaSuccess) { set_error("selftest attn: %s", cudaGetErrorString(e)); return false; }
    double worst_s = 0.0, worst_o = 0.0;
    const int rows = tile < 2 ? 128 : 24;
    for (int m = 0; m < rows; ++m) {
      const int qi = tile * 128 + m;
      std::vector<double> sc(280);
      double mx = -1e30;
      for (int j = 0; j < 280; ++j) {
        double s = 0.0;
        for (int c = 0; c < 32; ++c) s += (double)Q[qi * 32 + c] * (double)K[j * 32 + c];
        sc[j] = s;
        mx = fmax(mx, s);
        worst_s = fmax(worst_s, fabs(s - (double)S[m * 288 + j]));
      }
      double l = 0.0;
      std::vector<double> o(32, 0.0);
      for (int j = 0; j < 280; ++j) {
        const double pj = exp2(sc[j] - mx);
        l += pj;
        for (int c = 0; c < 32; ++c) o[c] += pj * (double)V[j * 32 + c];
      }
      for (int c = 0; c < 32; ++c) worst_o = fmax(worst_o, fabs(o[c] / l - (double)O[m * 32 + c]));
    }
    // scores must be exact to fp32 accumulation; outputs carry the bf16 rounding of P (~2^-9 relative)
    *max_err = fmax(worst_s, worst_o);
    if (worst_s > 1e-3) { set_error("selftest attn tile %d: scores off by %g (outputs %g)", tile, worst_s, worst_o); }
    return true;
  }
  if (which == 4) {
    std::vector<float> Q(288 * 32), K(288 * 32), V(288 * 32);
    for (auto& v : Q) v = bf16_round_host(rng.next() * 1.5f);
    for (auto& v : K) v = bf16_round_host(rng.next() * 1.5f);
    for (auto& v : V) v = bf16_round_host(rng.next());
    std::vector<uint16_t> img(3 * kQkvPart / 2, 0);
    auto put = [&](int part, const std::vector<float>& M) {
      for (int r = 0; r < 288; ++r)
        for (int c = 0; c < 32; ++c) {
          const int u = c >> 3, sw = (r >> 1) & 3;
          img[(part * kQkvPart + r * 64 + ((u ^ sw) << 4)) / 2 + (c & 7)] = bf16_bits_host(M[r * 32 + c]);
        }
    };
    put(0, Q); put(1, K); put(2, V);
    char* di = nullptr;
    float *ds = nullptr, *dO = nullptr;
    if (cudaMalloc(&di, 3 * kQkvPart) != cudaSuccess || cudaMalloc(&ds, 288 * 32 * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&dO, 24 * 32 * sizeof(float)) != cudaSuccess) {
      set_error("selftest: cudaMalloc failed");
      return false;
    }
    cudaMemsetAsync(ds, 0, 288 * 32 * sizeof(float), st);
    cudaMemsetAsync(dO, 0, 24 * 32 * sizeof(float), st);
    cudaMemcpyAsync(di, img.data(), 3 * kQkvPart, cudaMemcpyHostToDevice, st);
    cudaFuncSetAttribute(selftest_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes);
    selftest_tail_kernel<<<1, kTcThreads, kTcSmemBytes, st>>>(di, ds, dO);
    count_launch();
    std::vector<float> S(288 * 32), O(24 * 32);
    cudaMemcpyAsync(S.data(), ds, S.size() * sizeof(float), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(O.data(), dO, O.size() * sizeof(float), cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(di); cudaFree(ds); cudaFree(dO);
    if (e != cudaSuccess) { set_error("selftest tail: %s", cudaGetErrorString(e)); return false; }
    double worst_s = 0.0, worst_o = 0.0;
    for (int i = 0; i < 24; ++i) {
      const int qi = 256 + i;
      std::vector<double> sc(280);
      double mx = -1e30;
      for (int j = 0; j < 280; ++j) {
        double acc = 0.0;
        for (int c = 0; c < 32; ++c) acc += (double)Q[qi * 32 + c] * (double)K[j * 32 + c];
        sc[j] = acc;
        mx = fmax(mx, acc);
        worst_s = fmax(worst_s, fabs(acc - (double)S[j * 32 + i]));
      }
      double l = 0.0;
      std::vector<double> o(32, 0.0);
      for (int j = 0; j < 280; ++j) {
        const double pj = exp2(sc[j] - mx);
        l += pj;
        for (int c = 0; c < 32; ++c) o[c] += pj * (double)V[j * 32 + c];
      }
      for (int c = 0; c < 32; ++c) worst_o = fmax(worst_o, fabs(o[c] / l - (double)O[i * 32 + c]));
    }
    *max_err = fmax(worst_s, worst_o);
    if (worst_s > 1e-3 || worst_o > 2e-2) set_error("selftest tail: scores off by %g, outputs off by %g", worst_s, worst_o);
    return true;
  }
  set_error("aft_selftest: unknown test %d", which);
  return false;
}

}  // namespace aft
