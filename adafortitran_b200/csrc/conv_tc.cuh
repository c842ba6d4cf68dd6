// ConvEnhancer (reference src/models/blocks/enhancers.py:12-20) for the AFT_BF16 path: the two wide layers
// (8 -> 32 and 32 -> 8 channels, 92 % of the stack's FLOPs) run on the 5th-gen tensor cores as an implicit GEMM;
// the 1 -> 8 and 8 -> 1 layers stay on CUDA cores.
//
// Implicit GEMM by *shifted descriptors*: an activation map is stored in shared memory as K-major, NON-swizzled
// UMMA operand planes
//        plane[g][p][8 channels] (bf16, 16 bytes per position),   g = channel group of 8,
// over the zero-padded 122 x 16 position grid p = (row+1)*16 + (col+1).  Eight consecutive positions are one UMMA
// core matrix (8 rows x 16 bytes, contiguous), so the A operand "128 output positions starting at p0, as seen through
// filter tap (dy,dx)" is just the same plane addressed at p0 + (dy-1)*16 + (dx-1): one tcgen05.mma per (tap, 16 input
// channels) with a shifted start address -- no im2col copy.  M tiles run over padded positions (16 tiles of 128);
// results at border positions are discarded (written back as the zeros the next layer's padding needs).
//
//   conv2:  A = a1 plane, K 16 = 8 channels x 2 taps (the descriptor's LBO is the position offset between the two taps),
//           B = [32 cout][2 taps x 8 cin] per tap pair                                         ->  5 MMAs / tile, N = 32
//   conv3:  the three taps of a filter ROW go on N (N 32 = 3 dx x 8 cout + 8 zero), the rows on K: per tile 3 dy x 2
//           K-steps (32 channels) = 6 MMAs with A shifted by whole grid rows only; D[p][dx][co] is the contribution of
//           position p to output p - dx, and since p +- 1 are the neighbouring TMEM lanes of the same warp (the border
//           columns 0 and 15 of the 16-wide padded grid are never outputs) the epilogue adds the three with two warp
//           shuffles per channel.  6 instead of 18 MMAs per tile: the tensor pipe takes >= 40 clk per instruction
//           however narrow it is (tools/micro/mma_issue.cu), so the instruction count is the cost.
// Accumulators: conv2 and conv3 each fill all 512 TMEM columns (16 tiles x 32).
#pragma once

#include "aft_internal.cuh"
#include "tc_layout.cuh"
#include "tc_math.cuh"
#include "tc_ptx.cuh"

namespace aft {
namespace convtc {

using namespace ptx;

constexpr int kThreads = 512;                 // 16 warps; warps 0..3 also issue the MMAs (elected lane)
constexpr int kPosGuard = 32;                 // positions of slack before p = 0 (taps reach back 17 positions)
constexpr int kPosAlloc = 2112;               // 32 guard + 2048 (16 M-tiles) + 32 guard
constexpr int kPlaneBytes = kPosAlloc * 16;   // one 8-channel group: 33,792 bytes
constexpr int kTiles = 16;
constexpr int kIssuers = 4;                   // warps that issue the MMAs of a conv layer (stack_run), = count of its mbarriers
static_assert(kIssuers == 4, "a commit round (tiles 4 r .. 4 r + 3) must be the tiles one epilogue pass of the 16 warps reads");
// mbarriers of a stack run, byte offsets from the `bar` block (OFF_BAR): one per round of four tiles and layer
constexpr uint32_t kBarConv2 = 192, kBarConv3 = 224;
__device__ __forceinline__ void stack_bar_init(uint32_t bar) {
  for (int r = 0; r < 4; ++r) { ptx::mbar_init(bar + kBarConv2 + 8 * r, kIssuers); ptx::mbar_init(bar + kBarConv3 + 8 * r, kIssuers); }
}

// packed parameters of one conv stack (global memory, built by conv_tc_pack): byte offsets
constexpr int kPkW2 = 0;                      // 5 tap pairs x [2 taps][32 cout][8 cin] bf16 = 5 x 1024 (tap 9 = zeros)
constexpr int kPkW3 = 9216;                   // 6 (dy, kstep) x [2 halves][32 n = dx * 8 + cout, 24..31 zero][8] bf16 = 6 x 1024
constexpr int kPkF32 = 18432;                 // fp32: w0[9][8] | b0[8] | b1[32] | b2[8] | w3[9][8] | b3[1] (+pad) = 200 floats
constexpr int kPkBytes = 18432 + 800;         // 19,232
constexpr int kF_w0 = 0, kF_b0 = 72, kF_b1 = 80, kF_b2 = 112, kF_w3 = 120, kF_b3 = 192;

// shared-memory map of one conv-stack workspace (bytes, relative to a 1024-aligned base)
constexpr int OFF_A1 = 0;                               // 2 groups (second one zero) -- conv3's output a3 reuses group 0
constexpr int OFF_MID = 2 * kPlaneBytes;                // 4 groups
constexpr int OFF_PK = 6 * kPlaneBytes;                 // packed weights (kPkBytes)
constexpr int OFF_IN = OFF_PK + 19456;                  // fp32 padded input plane [122][16] (7,808 B); reused for the fp32 output
constexpr int OFF_BAR = OFF_IN + 7808;                  // callers' mbarriers (0..63: +16 = TMEM pointer) | 24 input floats | stack barriers (192..255)
constexpr int kStackSmemBytes = OFF_BAR + 256;          // 230,272
// After a stack has run, the mid planes are dead until the next conv2 epilogue rewrites positions [0, 2048) of every
// group; the fp32 result and the callers' scratch live there (behind the 512-byte front guard, which must stay zero).
constexpr int OFF_OUT = OFF_MID + kPosGuard * 16;                   // fp32 result, unpadded [1680]
constexpr int OFF_SCRATCH = OFF_MID + kPlaneBytes + kPosGuard * 16; // 32,768 bytes of caller scratch (group 1)
// The second a1 group is no longer an MMA operand (conv2 packs two taps into K instead of 8 channels + 8 zero channels):
// 33,792 bytes that stack_run never touches -- persistent caller scratch.
constexpr int OFF_KEEP = OFF_A1 + kPlaneBytes;

__device__ __forceinline__ uint64_t desc_k_none(uint32_t saddr, uint32_t lbo_bytes) {
  return make_smem_desc(saddr, lbo_bytes, 128, kSwizzleNone);   // SBO = 128: next 8 rows (positions / couts)
}
// the same split in a constant high word (SBO, version, layout) and a low word (LBO << 16 | address >> 4) so that the
// issue loops only add to the low word
constexpr uint32_t kDescHiNone = (128u >> 4) | (1u << 14);
__device__ __forceinline__ uint32_t desc_lo_none(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr >> 4) & 0x3FFF) | ((lbo_bytes >> 4) << 16); }
__device__ __forceinline__ uint64_t desc_join(uint32_t lo) { return ((uint64_t)kDescHiNone << 32) | lo; }

// diagnostics: phase stamps of one stack run (block 0, thread 0), only in -DAFT_TC_TIMELINE builds
#ifdef AFT_TC_TIMELINE
__device__ unsigned long long g_conv_tl[32];
#define AFT_CONV_STAMP(i) do { if (stamp_on && threadIdx.x == 0) g_conv_tl[i] = clock64(); } while (0)
#else
#define AFT_CONV_STAMP(i) do { } while (0)
#endif

constexpr uint32_t kIdescConv2 = make_idesc_bf16(128, 32, false, false);

__device__ __forceinline__ bool interior(int p) {   // padded position -> is it a real pixel?
  const int r = p >> 4, c = p & 15;
  return r >= 1 && r <= kGridH && c >= 1 && c <= kGridW;
}

// zero the activation planes once per CTA (guards and borders must stay zero; interiors are rewritten every image)
__device__ __forceinline__ void stack_init(uint8_t* smem, const uint8_t* __restrict__ pack) {
  uint4* z = reinterpret_cast<uint4*>(smem + OFF_A1);
  for (int i = threadIdx.x; i < 6 * kPlaneBytes / 16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
  const uint4* src = reinterpret_cast<const uint4*>(pack);
  uint4* dst = reinterpret_cast<uint4*>(smem + OFF_PK);
  for (int i = threadIdx.x; i < kPkBytes / 16; i += blockDim.x) dst[i] = src[i];
  float* in = reinterpret_cast<float*>(smem + OFF_IN);
  for (int i = threadIdx.x; i < kPlane; i += blockDim.x) in[i] = 0.f;
}

// Runs the stack on the fp32 padded plane at OFF_IN (interior filled by the caller, border zero) and leaves the fp32
// result, unpadded [1680], at OFF_OUT.  All kThreads threads call it.  `bar` = shared address of the barrier block
// (stack_bar_init), `phase` = number of stacks this CTA has run before (parity of its barriers).
__device__ __forceinline__ void stack_run(uint8_t* smem, uint32_t sb, uint32_t tmem, uint32_t bar, uint32_t phase) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool stamp_on = blockIdx.x == 0 && phase == 2; (void)stamp_on;
  AFT_CONV_STAMP(0);
  const float* fw = reinterpret_cast<const float*>(smem + OFF_PK + kPkF32);
  const float* in = reinterpret_cast<const float*>(smem + OFF_IN);

  // ---- conv1 (1 -> 8, ReLU) on CUDA cores: one interior position per thread iteration -> a1 group 0 (bf16).  The 72
  // weights stay in registers as packed fp32 pairs (FFMA2: same products, same order as the scalar form).
  {
    tcm::f32x2 w[9][4], b[4];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const float4 wa = *reinterpret_cast<const float4*>(fw + kF_w0 + t * 8), wb = *reinterpret_cast<const float4*>(fw + kF_w0 + t * 8 + 4);
      w[t][0] = tcm::pack2(wa.x, wa.y); w[t][1] = tcm::pack2(wa.z, wa.w); w[t][2] = tcm::pack2(wb.x, wb.y); w[t][3] = tcm::pack2(wb.z, wb.w);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = tcm::pack2(fw[kF_b0 + 2 * j], fw[kF_b0 + 2 * j + 1]);
    for (int px = tid; px < kPix; px += kThreads) {
      const int r = px / kGridW, c = px - r * kGridW;
      tcm::f32x2 acc[4] = {b[0], b[1], b[2], b[3]};
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const float a = in[(r + t / 3) * kPW + c + t % 3];
        const tcm::f32x2 aa = tcm::pack2(a, a);
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j] = tcm::fma2(aa, w[t][j], acc[j]);
      }
      const int p = (r + 1) * kPW + c + 1;
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float lo, hi;
        tcm::unpack2(acc[j], lo, hi);
        pk[j] = pack_bf16x2(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
      }
      *reinterpret_cast<uint4*>(smem + OFF_A1 + (kPosGuard + p) * 16) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
  }
  fence_proxy_async_smem();
  __syncthreads();
  AFT_CONV_STAMP(1);

  // ---- conv2 (8 -> 32) on the tensor core: 16 tiles x 5 tap pairs, K = 16 (8 channels x 2 taps)
  // Four issuing warps (tile i by warp i % 4; the tiles have disjoint accumulators): one thread issues one tcgen05.mma per
  // ~65 clk whatever its size, the tensor pipe takes these small ones every ~40 clk (tools/micro/mma_issue.cu) -- and the
  // 368 MMAs of a stack are half of its run time.  Each issuer commits to the same mbarrier (count kIssuers).
  if (warp < kIssuers) {   // converged warp, elected lane issues (keeps the descriptor math in uniform registers)
    const bool el = elect_one();
    tc_fence_after_sync();
    // K = 16 holds the 8 input channels of TWO taps: the second K half of the A descriptor (LBO) is the same plane seen
    // through the next tap, i.e. (shift(t1) - shift(t0)) positions further.  Five MMAs per tile (the ninth tap is paired
    // with zero weights) instead of nine.
    const uint32_t a_base = ((sb + OFF_A1 + kPosGuard * 16) >> 4) & 0x3FFF;   // + positions (16 B each == 1 address unit)
    const uint32_t b_lo = desc_lo_none(sb + OFF_PK + kPkW2, 512);
#pragma unroll 1
    for (int i = warp, r = 0; i < kTiles; i += kIssuers, ++r) {
#pragma unroll
      for (int pr = 0; pr < 5; ++pr) {
        const int t0 = 2 * pr, t1 = pr < 4 ? 2 * pr + 1 : 2 * pr;
        const int shift0 = (t0 / 3 - 1) * kPW + (t0 % 3 - 1), shift1 = (t1 / 3 - 1) * kPW + (t1 % 3 - 1);
        const uint32_t lbo = pr < 4 ? (uint32_t)(shift1 - shift0) : 1u;        // in 16-byte units
        mma_ss(tmem + i * 32, desc_join((a_base + i * 128 + shift0) | (lbo << 16)), desc_join(b_lo + pr * 64), kIdescConv2, pr > 0, el);
      }
      mma_commit(bar + kBarConv2 + 8 * r, el);   // round r = tiles 4 r .. 4 r + 3: its epilogue runs under the later rounds
    }
  }
  AFT_CONV_STAMP(2);
  AFT_CONV_STAMP(3);

  // ---- conv2 epilogue: + bias, ReLU, zero the border positions -> mid planes (4 groups of 8 channels, bf16)
  {
    const int q = warp & 3, part = warp >> 2;
    float b1[32];
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b = *reinterpret_cast<const float4*>(fw + kF_b1 + j);
      b1[j] = b.x; b1[j + 1] = b.y; b1[j + 2] = b.z; b1[j + 3] = b.w;
    }
#pragma unroll 2
    for (int i = part, r = 0; i < kTiles; i += 4, ++r) {
      mbar_wait(bar + kBarConv2 + 8 * r, phase & 1);
      tc_fence_after_sync();
      const int p = i * 128 + q * 32 + lane;
      uint32_t acc[32];
      tmem_ld16p(tmem + ((uint32_t)(q * 32) << 16) + i * 32, acc);
      tmem_ld16p(tmem + ((uint32_t)(q * 32) << 16) + i * 32 + 16, acc + 16);
      tmem_wait_ld();
      const bool in_img = interior(p);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float v0 = fmaxf(__uint_as_float(acc[g * 8 + 2 * j]) + b1[g * 8 + 2 * j], 0.f);
          const float v1 = fmaxf(__uint_as_float(acc[g * 8 + 2 * j + 1]) + b1[g * 8 + 2 * j + 1], 0.f);
          pk[j] = in_img ? pack_bf16x2(v0, v1) : 0u;
        }
        *reinterpret_cast<uint4*>(smem + OFF_MID + g * kPlaneBytes + (kPosGuard + p) * 16) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
    }
  }
  tc_fence_before_sync();
  fence_proxy_async_smem();
  __syncthreads();
  AFT_CONV_STAMP(4);

  // ---- conv3 (32 -> 8) on the tensor core: 16 tiles x 3 filter rows x 2 K-steps, N = 32 (3 dx x 8 cout + 8 zero columns)
  if (warp < kIssuers) {
    const bool el = elect_one();
    tc_fence_after_sync();
    const uint32_t a_lo = desc_lo_none(sb + OFF_MID + kPosGuard * 16, kPlaneBytes);
    const uint32_t b_lo = desc_lo_none(sb + OFF_PK + kPkW3, 512);
#pragma unroll 1
    for (int i = warp, r = 0; i < kTiles; i += kIssuers, ++r) {
#pragma unroll
      for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          mma_ss(tmem + i * 32, desc_join(a_lo + ks * (2 * kPlaneBytes / 16) + i * 128 + (dy - 1) * kPW), desc_join(b_lo + (dy * 2 + ks) * 64),
                 kIdescConv2, (dy | ks) != 0, el);
      mma_commit(bar + kBarConv3 + 8 * r, el);
    }
  }
  AFT_CONV_STAMP(5);
  AFT_CONV_STAMP(6);

  // ---- conv3 epilogue: out[p] = D[p-1][dx=-1] + D[p][dx=0] + D[p+1][dx=+1] (neighbouring lanes), + bias, ReLU, zero
  // borders -> a3 (bf16, reuses the a1 group-0 plane: conv2 has consumed it)
  {
    const int q = warp & 3, part = warp >> 2;
#pragma unroll 2
    for (int i = part, r = 0; i < kTiles; i += 4, ++r) {
      mbar_wait(bar + kBarConv3 + 8 * r, phase & 1);
      tc_fence_after_sync();
      const int p = i * 128 + q * 32 + lane;
      uint32_t acc[24];
      tmem_ld16p(tmem + ((uint32_t)(q * 32) << 16) + i * 32, acc);
      tmem_ld8p(tmem + ((uint32_t)(q * 32) << 16) + i * 32 + 16, acc + 16);
      tmem_wait_ld();
      const bool in_img = interior(p);
      float v[8];
#pragma unroll
      for (int co = 0; co < 8; ++co) {
        const float l = __shfl_up_sync(0xffffffffu, __uint_as_float(acc[co]), 1);
        const float r = __shfl_down_sync(0xffffffffu, __uint_as_float(acc[16 + co]), 1);
        v[co] = fmaxf((l + r) + (__uint_as_float(acc[8 + co]) + fw[kF_b2 + co]), 0.f);
      }
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) pk[j] = in_img ? pack_bf16x2(v[2 * j], v[2 * j + 1]) : 0u;
      *reinterpret_cast<uint4*>(smem + OFF_A1 + (kPosGuard + p) * 16) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  AFT_CONV_STAMP(7);

  // ---- conv4 (8 -> 1, no activation) on CUDA cores -> fp32 result, unpadded, at OFF_OUT.  Weights in registers as
  // packed pairs; four partial sums (two packed accumulators): short dependency chains, the order of the scalar form.
  {
    tcm::f32x2 w[9][4];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const float4 wa = *reinterpret_cast<const float4*>(fw + kF_w3 + t * 8), wb = *reinterpret_cast<const float4*>(fw + kF_w3 + t * 8 + 4);
      w[t][0] = tcm::pack2(wa.x, wa.y); w[t][1] = tcm::pack2(wa.z, wa.w); w[t][2] = tcm::pack2(wb.x, wb.y); w[t][3] = tcm::pack2(wb.z, wb.w);
    }
    const float b3 = fw[kF_b3];
    for (int px = tid; px < kPix; px += kThreads) {
      const int r = px / kGridW, c = px - r * kGridW;
      tcm::f32x2 acc01 = tcm::pack2(b3, 0.f), acc23 = tcm::pack2(0.f, 0.f);
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int p = (r + t / 3) * kPW + c + t % 3;
        const uint4 a = *reinterpret_cast<const uint4*>(smem + OFF_A1 + (kPosGuard + p) * 16);
        acc01 = tcm::fma2(tcm::bf16x2_to_f32x2(a.x), w[t][0], acc01);
        acc23 = tcm::fma2(tcm::bf16x2_to_f32x2(a.y), w[t][1], acc23);
        acc01 = tcm::fma2(tcm::bf16x2_to_f32x2(a.z), w[t][2], acc01);
        acc23 = tcm::fma2(tcm::bf16x2_to_f32x2(a.w), w[t][3], acc23);
      }
      float a0, a1, a2, a3;
      tcm::unpack2(acc01, a0, a1);
      tcm::unpack2(acc23, a2, a3);
      reinterpret_cast<float*>(smem + OFF_OUT)[px] = (a0 + a1) + (a2 + a3);
    }
  }
  __syncthreads();
  AFT_CONV_STAMP(8);
}

}  // namespace convtc
}  // namespace aft
