// AFT_BF16 path for grids other than the reference default -- in particular long sequences (BASELINE config 5: 3276 x 14
// grid, 7644 tokens per sequence): the 6-layer post-norm encoder (reference src/models/blocks/encoders.py:44-55,69 at
// max_seq_len >= S, positional_encodings.py:52,64) on the 5th-gen tensor cores with the sequence in GLOBAL memory.
//
// One sequence no longer fits an SM (K / V of one head: 478 KB), so the layer is cut in two kernels over 128-token row
// tiles (S is padded to T = ceil(S / 128) tiles; padding rows are zero tokens, padding keys are masked):
//
//   lin_block_kernel  (row-local part, one CTA per row tile, persistent):
//       [attention output tile] -> out_proj + residual + LayerNorm1 -> linear1 + GELU -> linear2 + residual + LayerNorm2
//       -> residual tile (bf16, in place)  [-> in_proj of the NEXT layer -> Q / K / V head tiles]
//     The first launch only runs the in_proj part (layer 0), the last one writes the fp32 rows the head reads.
//   attn_long_kernel  (one CTA per (sequence, head, 128-query tile), four CTAs per SM):
//       streaming attention over 64-key tiles of the head: S = Q K^T (tcgen05, accumulator in TMEM), online softmax
//       (running maximum / sum per row, one thread per query row, log2 domain), P (bf16) back to TMEM as the A operand
//       of P.V, output accumulator resident in TMEM and rescaled only when a maximum outgrows its reference by 2^8.
//       K / V tiles stream through a 4-stage ring of 1-D bulk copies; the next score tile is issued while the
//       exponentials of the current one run, and the other CTAs of the SM fill the tensor pipe / MUFU bubbles.
//
// Every operand lives in global memory as a byte-exact image of its shared-memory layout (tc_layout.cuh), per row tile:
//   residual / attention-output tile : K-major SWIZZLE_128B, 2 chunks x 128 rows x 128 B               = 32,768 B
//   Q / K / V tile of one head       : 128 rows x 64 B, SWIZZLE_64B (K-major for Q, K; the same bytes are V's MN-major
//                                      B operand)                                                        =  8,192 B
// Weights: the operand images and epilogue vectors of tc_encoder.cu (TcLayer), unchanged.
#include <cstdio>

#include "tc_encoder.cuh"
#include "tc_layout.cuh"
#include "tc_math.cuh"
#include "tc_ptx.cuh"

namespace aft {

namespace {

using namespace ptx;
using namespace tcm;

constexpr uint32_t kTileImg = 32768;      // residual / attention-output row tile image
constexpr uint32_t kChunk = 16384;        // one K-chunk (64 columns) of a 128-row image
constexpr uint32_t kHeadTile = 8192;      // Q / K / V tile of one head
constexpr int kVecPerLayerL = 1408, kVecBlockL = 384;   // layout of a layer's epilogue vector (tc_encoder.cu)
constexpr int kVBOut = 0, kVBL1 = 128, kVBL2 = 384, kVN1W = 512, kVN1B = 640, kVN2W = 768, kVN2B = 896;

constexpr uint32_t kDescHiSw64L = (uint32_t)(((uint64_t)(512 >> 4)) | ((uint64_t)1 << 14) | ((uint64_t)kSwizzle64 << 29));
__device__ __forceinline__ uint32_t dlo_k64(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | ((16u >> 4) << 16); }
__device__ __forceinline__ uint32_t dlo_mn64(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | ((512u >> 4) << 16); }
__device__ __forceinline__ uint64_t d64(uint32_t lo) { return ((uint64_t)kDescHiSw64L << 32) | lo; }
constexpr uint32_t kHi128 = (uint32_t)(desc_k_sw128_const() >> 32);
__device__ __forceinline__ uint64_t d128(uint32_t saddr, int ks) {
  return ((uint64_t)kHi128 << 32) | (((uint32_t)desc_k_sw128_const() | ((saddr >> 4) & 0x3FFF)) + (uint32_t)ks * 2);
}

// =============================================================================================
// fp32 rows [nseq * S][128] -> residual tile images (rows past S: zero tokens)
// =============================================================================================
__global__ void __launch_bounds__(256) f32_to_ximg_kernel(const float* __restrict__ h, char* __restrict__ ximg, int64_t nseq, int S, int T) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one 16-byte unit (8 columns)
  if (i >= nseq * T * 128 * 16) return;
  const int u = (int)(i & 15), r = (int)((i >> 4) & 127);
  const int64_t ti = i >> 11;
  const int64_t seq = ti / T;
  const int tok = (int)(ti - seq * T) * 128 + r;
  uint4 pk = make_uint4(0, 0, 0, 0);
  if (tok < S) {
    const float4 a = *reinterpret_cast<const float4*>(h + (seq * S + tok) * (int64_t)kD + u * 8);
    const float4 b = *reinterpret_cast<const float4*>(h + (seq * S + tok) * (int64_t)kD + u * 8 + 4);
    pk = make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
  }
  *reinterpret_cast<uint4*>(ximg + ti * (int64_t)kTileImg + image_offset(r, u * 8, 128)) = pk;
}

// =============================================================================================
// lin_block_kernel
// =============================================================================================
struct LinParams {
  char* ximg;              // [ntiles][32768] residual stream, replaced in place
  const char* aimg;        // [ntiles][32768] attention output of layer `layer_attn`
  char *q, *k, *v;         // [(seq * 4 + head) * T + tile][8192]
  float* h_out;            // fp32 [nseq * S][128] rows after the last layer (nullptr otherwise)
  const TcLayer* layers;
  int layer_attn;          // >= 0: out_proj / FFN of this layer run on the tile
  int layer_qkv;           // >= 0: in_proj of this layer runs on the (new) residual tile
  int activation;
  int64_t ntiles;
  int T, S;
};

constexpr int kLbCompute = 8, kLbThreads = 32 * (kLbCompute + 2);   // 8 compute warps (row quadrant x 2 column halves), producer, MMA
constexpr int kLbSlots = 5;
constexpr uint32_t LB_X = 0, LB_A = 32768, LB_H = 65536, LB_W = 98304, LB_VEC = LB_W + kLbSlots * kChunk,   // 180224
                   LB_BIAS = LB_VEC + 4096, LB_XCH = LB_BIAS + 1536, LB_BAR = LB_XCH + 2048, kLbSmem = LB_BAR + 256;
enum : uint32_t {
  LBB_IN = 0, LBB_VEC = 8, LBB_OUT_DONE = 16, LBB_F1_DONE = 24 /* 2 */, LBB_F2_DONE = 40, LBB_QKV_DONE = 48, LBB_X1_READY = 56,
  LBB_HID_READY = 64 /* 2 */, LBB_X2_READY = 80, LBB_QKV_READ = 88, LBB_TILE_DONE = 96, LBB_W_FULL = 104 /* 5 */, LBB_W_EMPTY = 144 /* 5 */,
  LBB_TMEM = 192
};
constexpr uint32_t kIdN128 = make_idesc_bf16(128, 128, false, false), kIdN96 = make_idesc_bf16(128, 96, false, false);

// 4 K-steps of one 64-column chunk: D (+)= A chunk (128 rows) . B piece^T
__device__ __forceinline__ void lb_issue_chunk(uint32_t d, uint32_t a, uint32_t b, uint32_t idesc, bool acc_first, bool el) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) mma_ss(d, d128(a, ks), d128(b, ks), idesc, acc_first || ks > 0, el);
}

__global__ void __launch_bounds__(kLbThreads, 1) lin_block_kernel(LinParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sb = smem_u32(smem_raw);
  if ((sb & 1023u) != 0) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar = sb + LB_BAR;
  const bool do_attn = p.layer_attn >= 0, do_qkv = p.layer_qkv >= 0;
  if (threadIdx.x == 0) {
    const uint32_t one[] = {LBB_IN, LBB_VEC, LBB_OUT_DONE, LBB_F1_DONE, LBB_F1_DONE + 8, LBB_F2_DONE, LBB_QKV_DONE, LBB_TILE_DONE};
    for (uint32_t b : one) mbar_init(bar + b, 1);
    for (int s = 0; s < kLbSlots; ++s) { mbar_init(bar + LBB_W_FULL + 8 * s, 1); mbar_init(bar + LBB_W_EMPTY + 8 * s, 1); }
    const uint32_t warps[] = {LBB_X1_READY, LBB_HID_READY, LBB_HID_READY + 8, LBB_X2_READY, LBB_QKV_READ};
    for (uint32_t b : warps) mbar_init(bar + b, kLbCompute);
    fence_mbar_init();
  }
  if (warp == kLbCompute + 1) { tmem_alloc(bar + LBB_TMEM, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(bar + LBB_TMEM));

  const TcLayer* LA = do_attn ? p.layers + p.layer_attn : nullptr;
  const TcLayer* LQ = do_qkv ? p.layers + p.layer_qkv : nullptr;

  if (warp == kLbCompute) {
    // ------------------------------------------------------------------------------------------- producer
    if (lane == 0) {
      // epilogue vectors: once per CTA
      mbar_arrive_expect_tx(bar + LBB_VEC, (do_attn ? 4096u : 0u) + (do_qkv ? 1536u : 0u));
      if (do_attn) bulk_g2s(sb + LB_VEC, LA->b_in + kVecBlockL, 4096, bar + LBB_VEC);
      if (do_qkv) bulk_g2s(sb + LB_BIAS, LQ->b_in, 1536, bar + LBB_VEC);
      uint32_t np = 0, n = 0;
      auto piece = [&](const void* src, uint32_t bytes) {
        const uint32_t s = np % kLbSlots;
        if (np >= kLbSlots) mbar_wait_relaxed(bar + LBB_W_EMPTY + 8 * s, ((np / kLbSlots) - 1) & 1);
        mbar_arrive_expect_tx(bar + LBB_W_FULL + 8 * s, bytes);
        bulk_g2s(sb + LB_W + s * kChunk, src, bytes, bar + LBB_W_FULL + 8 * s);
        ++np;
      };
      for (int64_t ti = blockIdx.x; ti < p.ntiles; ti += gridDim.x, ++n) {
        if (n > 0) mbar_wait_relaxed(bar + LBB_TILE_DONE, (n - 1) & 1);   // nobody reads the tile buffers any more
        mbar_arrive_expect_tx(bar + LBB_IN, kTileImg + (do_attn ? kTileImg : 0u));
        bulk_g2s(sb + LB_X, p.ximg + ti * (int64_t)kTileImg, kTileImg, bar + LBB_IN);
        if (do_attn) bulk_g2s(sb + LB_A, p.aimg + ti * (int64_t)kTileImg, kTileImg, bar + LBB_IN);
        if (ti + gridDim.x < p.ntiles) {
          bulk_prefetch_l2(p.ximg + (ti + gridDim.x) * (int64_t)kTileImg, kTileImg);
          if (do_attn) bulk_prefetch_l2(p.aimg + (ti + gridDim.x) * (int64_t)kTileImg, kTileImg);
        }
        if (do_attn) {
          const char* wo = reinterpret_cast<const char*>(LA->w_out);
          const char* w1 = reinterpret_cast<const char*>(LA->w_l1);
          const char* w2 = reinterpret_cast<const char*>(LA->w_l2);
          piece(wo, kChunk); piece(wo + kChunk, kChunk);
          for (int i = 0; i < 4; ++i) piece(w1 + i * kChunk, kChunk);
          for (int i = 0; i < 4; ++i) piece(w2 + i * kChunk, kChunk);
        }
        if (do_qkv) {
          const char* wi = reinterpret_cast<const char*>(LQ->w_in);
          for (int g = 0; g < 4; ++g) { piece(wi + g * 24576, 12288); piece(wi + g * 24576 + 12288, 12288); }
        }
      }
    }
  } else if (warp == kLbCompute + 1) {
    // ------------------------------------------------------------------------------------------- MMA issuer
    const bool el = elect_one();
    uint32_t np = 0, n = 0;
    auto piece_wait = [&]() -> uint32_t {
      const uint32_t s = np % kLbSlots;
      mbar_wait(bar + LBB_W_FULL + 8 * s, (np / kLbSlots) & 1);
      tc_fence_after_sync();
      return sb + LB_W + s * kChunk;
    };
    auto piece_done = [&]() { mma_commit(bar + LBB_W_EMPTY + 8 * (np % kLbSlots), el); ++np; };
    for (int64_t ti = blockIdx.x; ti < p.ntiles; ti += gridDim.x, ++n) {
      mbar_wait(bar + LBB_IN, n & 1);
      if (n > 0 && do_qkv) mbar_wait(bar + LBB_QKV_READ, (n - 1) & 1);   // accumulator columns of the previous tile read out
      tc_fence_after_sync();
      if (do_attn) {
        for (int c = 0; c < 2; ++c) {   // out_proj: A = attention-output tile
          const uint32_t w = piece_wait();
          lb_issue_chunk(tmem + 0, sb + LB_A + c * kChunk, w, kIdN128, c > 0, el);
          piece_done();
        }
        mma_commit(bar + LBB_OUT_DONE, el);
        mbar_wait(bar + LBB_X1_READY, n & 1);
        tc_fence_after_sync();
        for (int hf = 0; hf < 2; ++hf) {   // linear1: two halves of 128 hidden units
          for (int c = 0; c < 2; ++c) {
            const uint32_t w = piece_wait();
            lb_issue_chunk(tmem + 128 + hf * 128, sb + LB_X + c * kChunk, w, kIdN128, c > 0, el);
            piece_done();
          }
          mma_commit(bar + LBB_F1_DONE + 8 * hf, el);
        }
        mbar_wait(bar + LBB_HID_READY, n & 1);
        mbar_wait(bar + LBB_HID_READY + 8, n & 1);
        tc_fence_after_sync();
        for (int c = 0; c < 4; ++c) {   // linear2: A = hidden chunks (0, 1 over the attention tile, 2, 3 behind it)
          const uint32_t w = piece_wait();
          lb_issue_chunk(tmem + 0, sb + (c < 2 ? LB_A + c * kChunk : LB_H + (c - 2) * kChunk), w, kIdN128, c > 0, el);
          piece_done();
        }
        mma_commit(bar + LBB_F2_DONE, el);
        mbar_wait(bar + LBB_X2_READY, n & 1);
        tc_fence_after_sync();
      }
      if (do_qkv) {
        // the new residual tile goes back to global memory while the projection of the next layer reads it
        if (do_attn && lane == 0) bulk_s2g(p.ximg + ti * (int64_t)kTileImg, sb + LB_X, kTileImg);
        for (int g = 0; g < 4; ++g)
          for (int c = 0; c < 2; ++c) {
            const uint32_t w = piece_wait();
            lb_issue_chunk(tmem + g * 96, sb + LB_X + c * kChunk, w, kIdN96, c > 0, el);
            piece_done();
          }
        mma_commit(bar + LBB_QKV_DONE, el);
        if (do_attn && lane == 0) bulk_wait_read();
        __syncwarp();
      }
      mma_commit(bar + LBB_TILE_DONE, el);
    }
  } else {
    // ------------------------------------------------------------------------------------------- compute warps
    const int q = warp & 3, part = warp >> 2;    // TMEM lane quadrant, column half (= K-chunk of the images)
    const int rt = q * 32 + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const uint32_t vec = sb + LB_VEC, xch = sb + LB_XCH;
    const uint32_t xrow = sb + LB_X + part * kChunk + rt * 128;
    mbar_wait(bar + LBB_VEC, 0);
    uint32_t n = 0;
    // bias + residual + LayerNorm of this thread's 64 columns -> residual tile (bf16, in place); `which` 1 / 2
    auto layer_norm = [&](int which, float* out_row) {
      const uint32_t bias = vec + 4 * ((which == 1 ? kVBOut : kVBL2) + part * 64);
      const uint32_t gam = vec + 4 * ((which == 1 ? kVN1W : kVN2W) + part * 64);
      const uint32_t bet = vec + 4 * ((which == 1 ? kVN1B : kVN2B) + part * 64);
      f32x2 y[32];
      f32x2 s2 = pack2(0.f, 0.f), q2 = pack2(0.f, 0.f);
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t acc[32];
        tmem_ld_cols(lane_base + part * 64 + hf * 32, acc);
        tmem_wait_ld();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint4 xr = ld_shared_v4(xrow + (((hf * 4 + u) ^ (rt & 7)) << 4));
          const float4 b0 = lds_f4(bias + (hf * 4 + u) * 32), b1 = lds_f4(bias + (hf * 4 + u) * 32 + 16);
          const uint32_t xw[4] = {xr.x, xr.y, xr.z, xr.w};
          const f32x2 bb[4] = {pack2(b0.x, b0.y), pack2(b0.z, b0.w), pack2(b1.x, b1.y), pack2(b1.z, b1.w)};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const f32x2 a2 = pack2(__uint_as_float(acc[u * 8 + 2 * j]), __uint_as_float(acc[u * 8 + 2 * j + 1]));
            const f32x2 v = add2(add2(a2, bb[j]), bf16x2_to_f32x2(xw[j]));
            y[hf * 16 + u * 4 + j] = v;
            s2 = add2(s2, v);
            q2 = fma2(v, v, q2);
          }
        }
      }
      float sa, sb2, qa, qb;
      unpack2(s2, sa, sb2);
      unpack2(q2, qa, qb);
      st_shared_f32(xch + (part * 128 + rt) * 4, sa + sb2);
      st_shared_f32(xch + 1024 + (part * 128 + rt) * 4, qa + qb);
      named_bar_sync(1 + q, 64);
      const float sum = ld_shared_f32(xch + rt * 4) + ld_shared_f32(xch + (128 + rt) * 4);
      const float sq = ld_shared_f32(xch + 1024 + rt * 4) + ld_shared_f32(xch + 1024 + (128 + rt) * 4);
      named_bar_sync(1 + q, 64);   // both halves have read before the next use overwrites
      const float mean = sum * (1.0f / 128.0f);
      const float var = fmaxf(fmaf(-mean, mean, sq * (1.0f / 128.0f)), 0.f);
      const float rstd = rsqrtf(var + 1e-5f);
      const f32x2 rstd2 = pack2(rstd, rstd), shift2 = pack2(-mean * rstd, -mean * rstd);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 g0 = lds_f4(gam + u * 32), g1 = lds_f4(gam + u * 32 + 16), e0 = lds_f4(bet + u * 32), e1 = lds_f4(bet + u * 32 + 16);
        const f32x2 gg[4] = {pack2(g0.x, g0.y), pack2(g0.z, g0.w), pack2(g1.x, g1.y), pack2(g1.z, g1.w)};
        const f32x2 ee[4] = {pack2(e0.x, e0.y), pack2(e0.z, e0.w), pack2(e1.x, e1.y), pack2(e1.z, e1.w)};
        f32x2 o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = fma2(fma2(y[u * 4 + j], rstd2, shift2), gg[j], ee[j]);
        st_shared_v4(xrow + ((u ^ (rt & 7)) << 4), pack_bf16_pair(o[0]), pack_bf16_pair(o[1]), pack_bf16_pair(o[2]), pack_bf16_pair(o[3]));
        if (out_row != nullptr) {
          float a, b, c, d, e, f, g, h;
          unpack2(o[0], a, b); unpack2(o[1], c, d); unpack2(o[2], e, f); unpack2(o[3], g, h);
          *reinterpret_cast<float4*>(out_row + part * 64 + u * 8) = make_float4(a, b, c, d);
          *reinterpret_cast<float4*>(out_row + part * 64 + u * 8 + 4) = make_float4(e, f, g, h);
        }
      }
    };
    for (int64_t ti = blockIdx.x; ti < p.ntiles; ti += gridDim.x, ++n) {
      const int64_t seq = ti / p.T;
      const int tile = (int)(ti - seq * p.T);
      mbar_wait(bar + LBB_IN, n & 1);
      if (do_attn) {
        mbar_wait(bar + LBB_OUT_DONE, n & 1);
        tc_fence_after_sync();
        layer_norm(1, nullptr);
        tc_fence_before_sync();
        fence_proxy_async_smem();
        warp_arrive(bar + LBB_X1_READY, lane);
        for (int hf = 0; hf < 2; ++hf) {   // hidden units 128 hf + 64 part ... -> hidden chunk 2 hf + part
          mbar_wait(bar + LBB_F1_DONE + 8 * hf, n & 1);
          tc_fence_after_sync();
          const uint32_t bias = vec + 4 * (kVBL1 + hf * 128 + part * 64);
          const int c = 2 * hf + part;
          const uint32_t hrow = sb + (c < 2 ? LB_A + c * kChunk : LB_H + (c - 2) * kChunk) + rt * 128;
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            uint32_t acc[32];
            tmem_ld_cols(lane_base + 128 + hf * 128 + part * 64 + h2 * 32, acc);
            tmem_wait_ld();
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float4 b0 = lds_f4(bias + (h2 * 4 + u) * 32), b1 = lds_f4(bias + (h2 * 4 + u) * 32 + 16);
              const f32x2 bb[4] = {pack2(b0.x, b0.y), pack2(b0.z, b0.w), pack2(b1.x, b1.y), pack2(b1.z, b1.w)};
              uint32_t pk[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const f32x2 f = add2(pack2(__uint_as_float(acc[u * 8 + 2 * j]), __uint_as_float(acc[u * 8 + 2 * j + 1])), bb[j]);
                if (p.activation == AFT_ACT_GELU) {
                  pk[j] = pack_bf16_pair(gelu_tanh2(f));
                } else {
                  float a, b;
                  unpack2(f, a, b);
                  pk[j] = pack_bf16x2(fmaxf(a, 0.f), fmaxf(b, 0.f));
                }
              }
              st_shared_v4(hrow + (((h2 * 4 + u) ^ (rt & 7)) << 4), pk[0], pk[1], pk[2], pk[3]);
            }
          }
          tc_fence_before_sync();
          fence_proxy_async_smem();
          warp_arrive(bar + LBB_HID_READY + 8 * hf, lane);
        }
        mbar_wait(bar + LBB_F2_DONE, n & 1);
        tc_fence_after_sync();
        const int tok = tile * 128 + rt;
        layer_norm(2, (p.h_out != nullptr && tok < p.S) ? p.h_out + (seq * p.S + tok) * (int64_t)kD : nullptr);
        tc_fence_before_sync();
        fence_proxy_async_smem();
        warp_arrive(bar + LBB_X2_READY, lane);
      }
      if (do_qkv) {
        mbar_wait(bar + LBB_QKV_DONE, n & 1);
        tc_fence_after_sync();
        const int sw = (rt >> 1) & 3;
#pragma unroll 1
        for (int g = 0; g < 4; ++g) {
          // 96 columns [q_g | k_g | v_g] = 12 units of 8: this half owns units 6 part .. 6 part + 5
          uint32_t acc[48];
          tmem_ld_cols(lane_base + g * 96 + part * 48, acc);
          tmem_wait_ld();
          const int64_t tbase = ((seq * 4 + g) * p.T + tile) * (int64_t)kHeadTile + rt * 64;
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            const int u8 = part * 6 + i, mat = u8 >> 2, u = u8 & 3;
            const float4 b0 = lds_f4(sb + LB_BIAS + (g * 96 + u8 * 8) * 4), b1 = lds_f4(sb + LB_BIAS + (g * 96 + u8 * 8) * 4 + 16);
            const uint32_t* a = acc + i * 8;
            auto sum = [](uint32_t x0, uint32_t x1, float y0, float y1) {
              return pack_bf16_pair(add2(pack2(__uint_as_float(x0), __uint_as_float(x1)), pack2(y0, y1)));
            };
            char* dst = (mat == 0 ? p.q : (mat == 1 ? p.k : p.v)) + tbase + ((u ^ sw) << 4);
            *reinterpret_cast<uint4*>(dst) = make_uint4(sum(a[0], a[1], b0.x, b0.y), sum(a[2], a[3], b0.z, b0.w), sum(a[4], a[5], b1.x, b1.y),
                                                         sum(a[6], a[7], b1.z, b1.w));
          }
        }
        tc_fence_before_sync();
        warp_arrive(bar + LBB_QKV_READ, lane);
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kLbCompute + 1) tmem_dealloc(tmem, 512);
}

// =============================================================================================
// attn_long_kernel
// =============================================================================================
// One CTA = one 128-query tile of one (sequence, head); FOUR CTAs per SM (128 TMEM columns, 41 KB of shared memory and
// 64 K / 4 registers each), so that sixteen softmax warps per SM are in different phases of their key loops: the loop is
// bound by the exponentials (MUFU, 16 / clk / SM), and a first version with two CTAs of four warps (one 128-key tile per
// step, P.V products accumulated in registers) kept the MUFU pipe only 66 % busy.
//   key tile = 64 keys: S [128 x 64] (2 MMAs) -> one thread per query row: running maximum, exponentials, P (bf16) -> TMEM
//   -> O += P . V (4 MMAs, accumulator stays in TMEM across the key loop).
// The accumulator is only rescaled when a row maximum has grown by more than 2^8 since the last rescale (the scores are
// in log2 units; in between P is computed against the stale maximum, i.e. P <= 256, exact in bf16's exponent range), so
// the common path has no TMEM round trip of O -- the scheme of FlashAttention-4's correction step.
struct AttnParams {
  const char *q, *k, *v;   // head tiles
  char* aimg;              // attention output tiles (out_proj operand images)
  int T, S;
};
constexpr int kAtThreads = 256;   // warps 0..3: one thread per query row; warp 4: MMA issuer; warp 5: producer; 6, 7 idle
constexpr int kAtStages = 4, kKeyTile = 64;
constexpr uint32_t kKvStage = 8192;                      // K (4 KB) | V (4 KB) of one 64-key tile
constexpr uint32_t AT_Q = 0, AT_KV = 8192, AT_BAR = AT_KV + kAtStages * kKvStage, kAtSmem = AT_BAR + 256;   // 41,216
enum : uint32_t {
  ATB_Q = 0, ATB_S_DONE = 8, ATB_S_LOADED = 16, ATB_P_READY = 24, ATB_PV_DONE = 32, ATB_KV_FULL = 40 /* 4 */, ATB_KV_EMPTY = 72 /* 4 */,
  ATB_TMEM = 112
};
constexpr uint32_t ATM_S = 0, ATM_P = 64, ATM_O = 96;
constexpr uint32_t kIdS = make_idesc_bf16(128, 64, false, false), kIdPV = make_idesc_bf16(128, 32, false, true);
constexpr int kAtRegsCompute = 104, kAtRegsCtrl = 24;
constexpr float kRescaleThreshold = 8.0f;
constexpr int kLongPoly = 4;   // one pair of exponentials in kLongPoly runs on the FMA pipe (packed Cody-Waite + cubic, tc_math.cuh)

__global__ void __launch_bounds__(kAtThreads, 4) attn_long_kernel(AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sb = smem_u32(smem_raw);
  if ((sb & 1023u) != 0) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar = sb + AT_BAR;
  const int T = p.T, qt = blockIdx.x, g = blockIdx.y;
  const int nkt = (p.S + kKeyTile - 1) / kKeyTile;        // 64-key tiles (the last one may be partly padding)
  const int64_t seq = blockIdx.z;
  const int64_t head_base = ((seq * 4 + g) * T) * (int64_t)kHeadTile;
  if (threadIdx.x == 0) {
    mbar_init(bar + ATB_Q, 1); mbar_init(bar + ATB_S_DONE, 1); mbar_init(bar + ATB_PV_DONE, 1);
    mbar_init(bar + ATB_S_LOADED, 4); mbar_init(bar + ATB_P_READY, 4);
    for (int s = 0; s < kAtStages; ++s) { mbar_init(bar + ATB_KV_FULL + 8 * s, 1); mbar_init(bar + ATB_KV_EMPTY + 8 * s, 1); }
    fence_mbar_init();
  }
  if (warp == 4) { tmem_alloc(bar + ATB_TMEM, 128); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(bar + ATB_TMEM));

  if (warp >= 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kAtRegsCtrl));
    if (warp == 5 && lane == 0) {
      // --------------------------------------------------------------------------------------- producer
      mbar_arrive_expect_tx(bar + ATB_Q, kHeadTile);
      bulk_g2s(sb + AT_Q, p.q + head_base + qt * (int64_t)kHeadTile, kHeadTile, bar + ATB_Q);
      for (int j = 0; j < nkt; ++j) {
        const int s = j % kAtStages;
        if (j >= kAtStages) mbar_wait_relaxed(bar + ATB_KV_EMPTY + 8 * s, ((j / kAtStages) - 1) & 1);
        mbar_arrive_expect_tx(bar + ATB_KV_FULL + 8 * s, kKvStage);
        // 64 keys = half of a 128-row head tile image (rows 64 (j & 1) ...: 4 KB, whole swizzle atoms)
        bulk_g2s(sb + AT_KV + s * kKvStage, p.k + head_base + j * 4096ll, 4096, bar + ATB_KV_FULL + 8 * s);
        bulk_g2s(sb + AT_KV + s * kKvStage + 4096, p.v + head_base + j * 4096ll, 4096, bar + ATB_KV_FULL + 8 * s);
      }
    } else if (warp == 4) {
      // --------------------------------------------------------------------------------------- MMA issuer
      const bool el = elect_one();
      const uint32_t qd = dlo_k64(sb + AT_Q);
      auto issue_s = [&](int j) {
        const uint32_t kd = dlo_k64(sb + AT_KV + (j % kAtStages) * kKvStage);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) mma_ss(tmem + ATM_S, d64(qd + ks * 2), d64(kd + ks * 2), kIdS, ks > 0, el);
        mma_commit(bar + ATB_S_DONE, el);
      };
      mbar_wait(bar + ATB_Q, 0);
      mbar_wait(bar + ATB_KV_FULL, 0);
      tc_fence_after_sync();
      issue_s(0);
      for (int j = 0; j < nkt; ++j) {
        if (j + 1 < nkt) {
          mbar_wait(bar + ATB_KV_FULL + 8 * ((j + 1) % kAtStages), ((j + 1) / kAtStages) & 1);
          mbar_wait(bar + ATB_S_LOADED, j & 1);          // score tile j is in registers
          tc_fence_after_sync();
          issue_s(j + 1);
        }
        mbar_wait(bar + ATB_P_READY, j & 1);             // P(j) in TMEM, accumulator rescaled if it had to be
        tc_fence_after_sync();
        const uint32_t vd = dlo_mn64(sb + AT_KV + (j % kAtStages) * kKvStage + 4096);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) mma_ts(tmem + ATM_O, tmem + ATM_P + ks * 8, d64(vd + ks * 64), kIdPV, j > 0 || ks > 0, el);
        mma_commit(bar + ATB_PV_DONE, el);
        mma_commit(bar + ATB_KV_EMPTY + 8 * (j % kAtStages), el);
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------- softmax: one row per thread
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kAtRegsCompute));
    const int rt = warp * 32 + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    float m_ref = -INFINITY;   // maximum the accumulator and the row sum are currently scaled to
    float l = 0.f;
#pragma unroll 1
    for (int j = 0; j < nkt; ++j) {
      mbar_wait(bar + ATB_S_DONE, j & 1);
      tc_fence_after_sync();
      float v[kKeyTile];
      {
        uint32_t x[kKeyTile];
        tmem_ld_cols(lane_base + ATM_S, x);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < kKeyTile; ++c) v[c] = __uint_as_float(x[c]);
      }
      tc_fence_before_sync();
      warp_arrive(bar + ATB_S_LOADED, lane);
      if (j == nkt - 1) {   // keys past the sequence are padding
        const int nvalid = p.S - j * kKeyTile;
#pragma unroll
        for (int c = 0; c < kKeyTile; ++c)
          if (c >= nvalid) v[c] = -INFINITY;
      }
      float m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3];
#pragma unroll
      for (int c = 4; c < kKeyTile; c += 4) { m0 = fmaxf(m0, v[c]); m1 = fmaxf(m1, v[c + 1]); m2 = fmaxf(m2, v[c + 2]); m3 = fmaxf(m3, v[c + 3]); }
      const float mt = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
      // P.V(j-1) must be complete before P is overwritten (and before the accumulator may be touched)
      if (j > 0) {
        mbar_wait(bar + ATB_PV_DONE, (j - 1) & 1);
        tc_fence_after_sync();
      }
      // rescale (whole warp, per-row factors) only when some row's maximum outgrew its reference by more than the threshold
      const bool grow = mt > m_ref + kRescaleThreshold;
      if (__any_sync(0xFFFFFFFFu, grow)) {
        const float mn = fmaxf(m_ref, mt);
        const float f = ex2(m_ref - mn);   // first tile: exp2(-inf) = 0, the accumulator is not read (j == 0)
        if (j > 0) {
          uint32_t a[32];
          tmem_ld_cols(lane_base + ATM_O, a);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) a[i] = __float_as_uint(__uint_as_float(a[i]) * f);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t (&a8)[8] = *reinterpret_cast<const uint32_t (*)[8]>(a + 8 * i);
            tmem_st8(lane_base + ATM_O + i * 8, a8);
          }
        }
        l *= f;
        m_ref = mn;
      }
      // exponentials against the reference maximum -> P (bf16 pairs) -> TMEM
      const f32x2 negm2 = pack2(-m_ref, -m_ref);
      f32x2 s2a = pack2(0.f, 0.f), s2b = pack2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < kKeyTile / 16; ++i) {
        uint32_t pk[8];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int c = i * 16 + 2 * jj;
          const f32x2 x2 = add2(pack2(v[c], v[c + 1]), negm2);
          f32x2 e2;
          if (jj % kLongPoly == kLongPoly - 1) {
            e2 = ex2_poly2(x2);   // a share of the exponentials on the FMA pipe
          } else {
            float a, b;
            unpack2(x2, a, b);
            e2 = pack2(ex2(a), ex2(b));
          }
          if (jj & 1) s2b = add2(s2b, e2); else s2a = add2(s2a, e2);
          pk[jj] = pack_bf16_pair(e2);
        }
        tmem_st8(lane_base + ATM_P + i * 8, pk);
      }
      tmem_wait_st();
      float sa, sb2, sc, sd;
      unpack2(s2a, sa, sb2);
      unpack2(s2b, sc, sd);
      l += (sa + sb2) + (sc + sd);
      tc_fence_before_sync();
      warp_arrive(bar + ATB_P_READY, lane);
    }
    mbar_wait(bar + ATB_PV_DONE, (nkt - 1) & 1);
    tc_fence_after_sync();
    uint32_t a[32];
    tmem_ld_cols(lane_base + ATM_O, a);
    tmem_wait_ld();
    const float inv = 1.0f / l;
    const f32x2 inv2 = pack2(inv, inv);
    char* row = p.aimg + (seq * T + qt) * (int64_t)kTileImg + (g >> 1) * kChunk + rt * 128;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      auto sc2 = [&](int i) { return pack_bf16_pair(mul2(pack2(__uint_as_float(a[8 * u + i]), __uint_as_float(a[8 * u + i + 1])), inv2)); };
      *reinterpret_cast<uint4*>(row + ((((g & 1) * 4 + u) ^ (rt & 7)) << 4)) = make_uint4(sc2(0), sc2(2), sc2(4), sc2(6));
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, 128);
}

size_t align_up_l(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

// =============================================================================================
// host side
// =============================================================================================
size_t tc_long_workspace_bytes(int64_t nseq, int S) {
  const size_t T = (size_t)(S + 127) / 128, tiles = (size_t)nseq * T;
  return 2 * align_up_l(tiles * kTileImg, 1024) + 3 * align_up_l(tiles * 4 * kHeadTile, 1024);
}

bool tc_long_encoder(const TcWeights& w, int activation, int sm_count, const float* h_in, float* h_out, int64_t nseq, int S,
                     void* workspace, cudaStream_t st) {
  const int T = (S + 127) / 128;
  const int64_t tiles = nseq * T;
  char* ws = static_cast<char*>(workspace);
  char* ximg = ws;
  char* aimg = ximg + align_up_l((size_t)tiles * kTileImg, 1024);
  char* q = aimg + align_up_l((size_t)tiles * kTileImg, 1024);
  char* k = q + align_up_l((size_t)tiles * 4 * kHeadTile, 1024);
  char* v = k + align_up_l((size_t)tiles * 4 * kHeadTile, 1024);
  if (cudaFuncSetAttribute(lin_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLbSmem) != cudaSuccess ||
      cudaFuncSetAttribute(attn_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAtSmem) != cudaSuccess) {
    set_error("tc_long: cannot opt in to the shared-memory sizes: %s", cudaGetErrorString(cudaGetLastError()));
    return false;
  }
  {
    const int64_t units = tiles * 128 * 16;
    f32_to_ximg_kernel<<<(unsigned)((units + 255) / 256), 256, 0, st>>>(h_in, ximg, nseq, S, T);
    count_launch();
    if (!check_launch("f32_to_ximg_kernel")) return false;
  }
  LinParams lp;
  lp.ximg = ximg; lp.aimg = aimg; lp.q = q; lp.k = k; lp.v = v;
  lp.layers = w.layers_dev; lp.activation = activation; lp.ntiles = tiles; lp.T = T; lp.S = S;
  const unsigned lgrid = (unsigned)(tiles < sm_count ? tiles : sm_count);
  AttnParams ap;
  ap.q = q; ap.k = k; ap.v = v; ap.aimg = aimg; ap.T = T; ap.S = S;
  for (int l = -1; l < w.num_layers; ++l) {
    if (l >= 0) {
      attn_long_kernel<<<dim3((unsigned)T, 4, (unsigned)nseq), kAtThreads, kAtSmem, st>>>(ap);
      count_launch();
      if (!check_launch("attn_long_kernel")) return false;
    }
    lp.layer_attn = l;
    lp.layer_qkv = l + 1 < w.num_layers ? l + 1 : -1;
    lp.h_out = l == w.num_layers - 1 ? h_out : nullptr;
    lin_block_kernel<<<lgrid, kLbThreads, kLbSmem, st>>>(lp);
    count_launch();
    if (!check_launch("lin_block_kernel")) return false;
  }
  return true;
}

}  // namespace aft
