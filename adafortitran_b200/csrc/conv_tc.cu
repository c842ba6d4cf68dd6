// Frontend and head of the AFT_BF16 path with the ConvEnhancer stacks on the tensor cores (conv_tc.cuh).
//   frontend_tc : pilots -> Linear(24,1680) -> ConvEnhancer -> Unfold(3x2) [+ ChannelAdapter] -> linear_1 + pos -> X image
//   head_tc     : linear_2 -> Fold -> + conv_enhanced -> ConvEnhancer -> complex64
// Same math and reference citations as frontend.cu / head.cu; persistent CTAs (the zero-padded activation planes,
// the packed weights and the TMEM allocation are set up once per CTA).
#include <cstdio>

#include "conv_tc.cuh"

namespace aft {

using namespace convtc;

namespace {

// One item = (token row t, 4 consecutive model columns): 288 x 32 items = 18 per thread.  A thread keeps the same four
// columns for all its items (512 threads = 16 rows x 32 column groups per pass), so its IN_DIM x 4 weights stay in
// registers as packed fp32 pairs and an item costs IN_DIM / 4 shared loads of the token row (one row per warp: broadcast)
// + IN_DIM * 2 FFMA2.  Items go three at a time so that the reads of the positional table (L2 resident, 143 KB) of a
// batch are in flight together.  Same products in the same order as the scalar fmaf form.
template <int IN_DIM>
__device__ __forceinline__ void linear1_image(const float* __restrict__ posb, const float* tok, const float* __restrict__ w1t, char* base) {
  constexpr int kItems = kSPad * (kD / 4), kPerThread = kItems / kThreads;   // 9216 / 512 = 18
  static_assert(kItems % kThreads == 0 && kPerThread % 3 == 0 && kThreads % (kD / 4) == 0, "item count must split evenly");
  const int tid = threadIdx.x, c4 = (tid & 31) * 4, t0 = tid >> 5;
  tcm::f32x2 w[IN_DIM][2];
#pragma unroll
  for (int k = 0; k < IN_DIM; ++k) {
    const float4 wv = *reinterpret_cast<const float4*>(w1t + k * kD + c4);
    w[k][0] = tcm::pack2(wv.x, wv.y); w[k][1] = tcm::pack2(wv.z, wv.w);
  }
  const int chunk_off = (c4 >> 6) * kXChunkBytes, unit = (c4 & 63) >> 3, sub = (c4 & 4) * 2;   // ximage_offset(t, c4), split
#pragma unroll 1
  for (int b0 = 0; b0 < kPerThread; b0 += 3) {
    float4 pa[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int t = t0 + (b0 + j) * (kThreads / 32);
      const int tt = t < kS ? t : 0;   // rows 280..287 are zero padding (computed on a valid row, stored as zeros)
      pa[j] = *reinterpret_cast<const float4*>(posb + tt * kD + c4);
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int t = t0 + (b0 + j) * (kThreads / 32);
      const int tt = t < kS ? t : 0;
      tcm::f32x2 acc0 = tcm::pack2(pa[j].x, pa[j].y), acc1 = tcm::pack2(pa[j].z, pa[j].w);
      float a[IN_DIM];
      if (IN_DIM % 4 == 0) {
#pragma unroll
        for (int k = 0; k < IN_DIM; k += 4) {
          const float4 v = *reinterpret_cast<const float4*>(tok + tt * IN_DIM + k);
          a[k] = v.x; a[k + 1] = v.y; a[k + 2] = v.z; a[k + 3] = v.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < IN_DIM; k += 2) {
          const float2 v = *reinterpret_cast<const float2*>(tok + tt * IN_DIM + k);
          a[k] = v.x; a[k + 1] = v.y;
        }
      }
#pragma unroll
      for (int k = 0; k < IN_DIM; ++k) {
        const tcm::f32x2 aa = tcm::pack2(a[k], a[k]);
        acc0 = tcm::fma2(aa, w[k][0], acc0);
        acc1 = tcm::fma2(aa, w[k][1], acc1);
      }
      uint2 pk = make_uint2(tcm::pack_bf16_pair(acc0), tcm::pack_bf16_pair(acc1));
      if (t >= kS) pk = make_uint2(0, 0);
      *reinterpret_cast<uint2*>(base + chunk_off + t * kChunkRowBytes + (((unit ^ (t & 7)) << 4) | sub)) = pk;
    }
  }
}

// ChannelAdapter (reference blocks/channel_adaptivity.py:34-40,59-63), once per SAMPLE (the reference evaluates it in both
// the real and the imaginary pass): z[sample][m][j], m = snr / delay spread / Doppler, j < 2 S.  The last layer
// (42 x 560 weights per condition, 94 KB) is held in registers -- thread j keeps column j -- and the CTA streams its
// samples past them, instead of every sequence re-reading 282 KB of weights from L2 inside the frontend kernel.
constexpr int kAdaThreads = 576;     // >= 2 S = 560 outputs of one encoder
constexpr int kAdaGroup = 32;        // samples per pass of a CTA
__global__ void __launch_bounds__(kAdaThreads, 1)
adapter_kernel(FrontPack p, const float* __restrict__ snr, const float* __restrict__ ds, const float* __restrict__ dop,
               float* __restrict__ z, int64_t nsamples) {
  __shared__ float hid2[kAdaGroup][kMaxAdaHidden];
  const int j = threadIdx.x;
  const bool live = j < 2 * kS;
  for (int i = threadIdx.x; i < kAdaGroup * kMaxAdaHidden; i += kAdaThreads) (&hid2[0][0])[i] = 0.f;   // units >= h2 stay zero
  for (int m = 0; m < 3; ++m) {
    const MlpPack& mp = p.mlp[m];
    const float* cond = m == 0 ? snr : (m == 1 ? ds : dop);
    float w[kMaxAdaHidden];
#pragma unroll
    for (int k = 0; k < kMaxAdaHidden; ++k) w[k] = (live && k < p.h2) ? mp.w2t[k * 2 * kS + j] : 0.f;
    const float b2 = live ? mp.b2[j] : 0.f;
    for (int64_t s0 = (int64_t)blockIdx.x * kAdaGroup; s0 < nsamples; s0 += (int64_t)gridDim.x * kAdaGroup) {
      const int ns = (int)(nsamples - s0 < kAdaGroup ? nsamples - s0 : kAdaGroup);
      __syncthreads();   // the previous group's hidden activations have been consumed
      // hidden layers of the group's samples: thread (sample, unit) pairs
      for (int i = threadIdx.x; i < ns * p.h2; i += kAdaThreads) {
        const int s = i / p.h2, u = i - s * p.h2;
        const float c = cond[s0 + s];
        float acc = mp.b1[u];
        for (int k = 0; k < p.h1; ++k) acc = fmaf(mp.w1[u * p.h1 + k], fmaxf(fmaf(mp.w0[k], c, mp.b0[k]), 0.f), acc);
        hid2[s][u] = fmaxf(acc, 0.f);
      }
      __syncthreads();
      if (live) {
        for (int s = 0; s < ns; ++s) {
          float acc = b2;
#pragma unroll
          for (int k = 0; k < kMaxAdaHidden; ++k) acc = fmaf(w[k], hid2[s][k], acc);   // units >= h2: zero weights
          z[((s0 + s) * 3 + m) * (int64_t)(2 * kS) + j] = acc;
        }
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kThreads, 1)
frontend_tc_kernel(FrontPack p, const uint8_t* __restrict__ pack, const float2* __restrict__ pilots, const float* __restrict__ zin,
                   float* __restrict__ enh_out, __nv_bfloat16* __restrict__ hb_out, int64_t nseq) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sb = smem_u32(smem);
  if ((sb & 1023u) != 0) __trap();
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar = sb + OFF_BAR;
  float* xin = reinterpret_cast<float*>(smem + OFF_BAR + 64);   // [24]
  if (tid == 0) { stack_bar_init(bar); fence_mbar_init(); }
  if (warp == 1) { tmem_alloc(bar + 16, 512); tmem_relinquish(); }
  stack_init(smem, pack);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(bar + 16));

  float* in = reinterpret_cast<float*>(smem + OFF_IN);
  const float* enh = reinterpret_cast<const float*>(smem + OFF_OUT);
  float* tok = reinterpret_cast<float*>(smem + OFF_SCRATCH);   // [280][in_dim]
  float* z = tok + 3360;                                       // [3][560]
  const int in_dim = p.in_dim;
  uint32_t n_run = 0;

  for (int64_t seq = blockIdx.x; seq < nseq; seq += gridDim.x, ++n_run) {
    const int64_t sample = seq >> 1;
    if (tid < kPilots) {
      const float2 v = pilots[sample * kPilots + tid];
      xin[tid] = (seq & 1) ? v.y : v.x;
    }
    __syncthreads();
#ifdef AFT_TC_TIMELINE
    const bool st_on = blockIdx.x == 0 && n_run == 2 && tid == 0;
    if (st_on) g_conv_tl[10] = clock64();
#endif
    // upsample (fortitran.py:203) into the padded fp32 plane
    // four consecutive pixels per thread: the 161 KB weight matrix (L2 resident) is read with 16-byte loads, a quarter
    // of the load instructions of the one-pixel form (same products, same order per pixel)
    static_assert(kPix % 4 == 0, "four pixels per thread");
    for (int q4 = tid; q4 < kPix / 4; q4 += kThreads) {
      const int pix = 4 * q4;
      float4 wv[kPilots];
#pragma unroll
      for (int k = 0; k < kPilots; ++k) wv[k] = *reinterpret_cast<const float4*>(p.up_wt + k * kPix + pix);
      float4 acc = *reinterpret_cast<const float4*>(p.up_b + pix);
#pragma unroll
      for (int k = 0; k < kPilots; ++k) {
        const float xk = xin[k];
        acc.x = fmaf(wv[k].x, xk, acc.x); acc.y = fmaf(wv[k].y, xk, acc.y);
        acc.z = fmaf(wv[k].z, xk, acc.z); acc.w = fmaf(wv[k].w, xk, acc.w);
      }
      const float a4[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = (pix + j) / kGridW, c = (pix + j) - r * kGridW;
        in[(r + 1) * kPW + c + 1] = a4[j];
      }
    }
    __syncthreads();
#ifdef AFT_TC_TIMELINE
    if (st_on) g_conv_tl[11] = clock64();
#endif
    stack_run(smem, sb, tmem, bar, n_run);                      // fortitran.py:209
#ifdef AFT_TC_TIMELINE
    if (st_on) g_conv_tl[12] = clock64();
#endif
    for (int i = tid; i < kPix / 4; i += kThreads)   // 16-byte stores
      reinterpret_cast<float4*>(enh_out + seq * kPix)[i] = reinterpret_cast<const float4*>(enh)[i];

    // tokens = [patch(6) | adaptive(6)]  (fortitran.py:212-217)
    for (int i = tid; i < kS * kPatchLen; i += kThreads) {
      const int t = i / kPatchLen, f = i - t * kPatchLen;
      const int pi = t / kTokW, pj = t - pi * kTokW;
      const int a = f / kPatchW, b = f - a * kPatchW;
      tok[t * in_dim + f] = enh[(kPatchH * pi + a) * kGridW + kPatchW * pj + b];
    }
    if (p.adaptive) {
      // adaptive features (fortitran.py:216): computed once per sample by adapter_kernel, 3 x 560 floats
      const float* zs = zin + sample * (int64_t)(3 * 2 * kS);
      for (int i = tid; i < 3 * 2 * kS; i += kThreads) z[i] = zs[i];
      __syncthreads();
      for (int i = tid; i < kS * kAda; i += kThreads) {
        const int t = i / kAda, f = i - t * kAda;
        tok[t * in_dim + kPatchLen + f] = z[(f >> 1) * 2 * kS + 2 * t + (f & 1)];
      }
    }
    __syncthreads();
#ifdef AFT_TC_TIMELINE
    if (st_on) g_conv_tl[13] = clock64();
#endif
    // h = tok . W1^T + b1 + pos (encoders.py:67-68) -> bf16 operand image of the residual stream
    if (in_dim == kPatchLen) linear1_image<kPatchLen>(p.posb, tok, p.l1_wt, reinterpret_cast<char*>(hb_out) + seq * (int64_t)kXImageBytes);
    else linear1_image<kPatchLen + kAda>(p.posb, tok, p.l1_wt, reinterpret_cast<char*>(hb_out) + seq * (int64_t)kXImageBytes);
    __syncthreads();   // scratch / result are overwritten by the next image
#ifdef AFT_TC_TIMELINE
    if (st_on) g_conv_tl[14] = clock64();
#endif
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

__global__ void __launch_bounds__(kThreads, 1)
head_tc_kernel(HeadPack p, const uint8_t* __restrict__ pack, const uint8_t* __restrict__ himg, const float* __restrict__ enh,
               OutDst out /* complex64 destinations, see aft_internal.cuh */, int64_t nsamples) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sb = smem_u32(smem);
  if ((sb & 1023u) != 0) __trap();
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar = sb + OFF_BAR;
  if (tid == 0) { stack_bar_init(bar); mbar_init(bar + 32, 1); mbar_init(bar + 40, 3); fence_mbar_init(); }
  if (warp == 1) { tmem_alloc(bar + 16, 512); tmem_relinquish(); }
  stack_init(smem, pack);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(bar + 16));

  float* in = reinterpret_cast<float*>(smem + OFF_IN);
  const float* res = reinterpret_cast<const float*>(smem + OFF_OUT);
  // persistent scratch (second a1 group): W2 image 0..4095 | enhanced image 4096.. | real part 12288.. | complex64 staging row
  constexpr uint32_t kStageOff = OFF_KEEP + 19456;
  static_assert(12288 + kPix * 4 <= 19456 && 19456 + kPix * 8 <= kPlaneBytes, "staging row must fit behind the real part");
  // linear_2 on the tensor core.  The encoder's output image (2 K-chunks x 288 rows x 128 B, SWIZZLE_128B) is staged as ONE
  // contiguous 73,728-byte block starting 1024-aligned inside mid group 1 and running through groups 2 and 3 (dead between
  // two stack runs): it is then directly the A operand of  D[token, 16] = X[token, 128] . W2^T  (three M = 128 row tiles,
  // N = 16: six real outputs + zero rows).  The block covers the zero guards between the groups; they are re-zeroed
  // before the conv stack runs.  W2 lives as a 4 KB bf16 operand image at the start of the persistent scratch.
  constexpr uint32_t kImgOff = OFF_MID + kPlaneBytes + 1024;
  static_assert(kImgOff % 1024 == 0 && kImgOff + kXImageBytes <= OFF_MID + 4 * kPlaneBytes, "image staging must be aligned and inside the mid planes");
  const float* es = reinterpret_cast<const float*>(smem + OFF_KEEP + 4096);
  float* re_keep = reinterpret_cast<float*>(smem + OFF_KEEP + 12288);   // real part of the sample (result of the first pass), [1680]
  for (int i = tid; i < 2 * 16 * 8; i += kThreads) {   // 16-byte units of the W2 image: [chunk][row 0..15][unit]
    const int c = i >> 7, r = (i >> 3) & 15, u = i & 7;
    uint4 pk = make_uint4(0, 0, 0, 0);
    if (r < kPatchLen) {
      const float* w = p.l2_w + r * kD + c * 64 + u * 8;
      pk = make_uint4(pack_bf16x2(w[0], w[1]), pack_bf16x2(w[2], w[3]), pack_bf16x2(w[4], w[5]), pack_bf16x2(w[6], w[7]));
    }
    *reinterpret_cast<uint4*>(smem + OFF_KEEP + c * 2048 + r * 128 + ((u ^ (r & 7)) << 4)) = pk;
  }
  float l2b[kPatchLen];
#pragma unroll
  for (int f = 0; f < kPatchLen; ++f) l2b[f] = p.l2_b[f];
  fence_proxy_async_smem();
  __syncthreads();
  uint32_t n_run = 0;
  constexpr uint32_t kIdescL2 = make_idesc_bf16(128, 16, false, false);

  for (int64_t sample = blockIdx.x; sample < nsamples; sample += gridDim.x) {
    for (int part = 0; part < 2; ++part, ++n_run) {
      const int64_t seq = 2 * sample + part;
      const uint8_t* hs = himg + seq * (int64_t)kXImageBytes;   // encoder output: bf16 operand image (tc_layout.cuh)
#ifdef AFT_TC_TIMELINE
      const bool st_on = blockIdx.x == 0 && n_run == 2 && tid == 0;
      if (st_on) g_conv_tl[20] = clock64();
#endif
      if (warp == 0) {
        const bool el = elect_one();
        if (el) {
          // (the previous part ended with a __syncthreads: nobody reads the mid planes or the enhanced image any more)
          mbar_arrive_expect_tx(bar + 32, kXImageBytes + kPix * sizeof(float));
          bulk_g2s(sb + kImgOff, hs, kXImageBytes, bar + 32);
          bulk_g2s(sb + OFF_KEEP + 4096, enh + seq * (int64_t)kPix, kPix * sizeof(float), bar + 32);
          // the next part's inputs travel HBM -> L2 while this part's conv stack runs
          const int64_t nseq2 = part == 0 ? seq + 1 : 2 * (sample + gridDim.x);
          if (nseq2 < 2 * nsamples) {
            bulk_prefetch_l2(himg + nseq2 * (int64_t)kXImageBytes, kXImageBytes);
            bulk_prefetch_l2(enh + nseq2 * (int64_t)kPix, kPix * sizeof(float));
          }
        }
      }
      if (warp < 3) {   // linear_2: one issuing warp per row tile (an issuing thread manages one MMA per ~65 clk)
        const bool el = elect_one();
        const int t = warp;
        mbar_wait(bar + 32, n_run & 1);
        tc_fence_after_sync();
        constexpr uint32_t kHi = (uint32_t)(desc_k_sw128_const() >> 32);
        const uint32_t lo = (uint32_t)desc_k_sw128_const();
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t a = lo | (((sb + kImgOff + c * kXChunkBytes + t * 128 * 128) >> 4) & 0x3FFF);
            const uint32_t b = lo | (((sb + OFF_KEEP + c * 2048) >> 4) & 0x3FFF);
            mma_ss(tmem + t * 16, ((uint64_t)kHi << 32) | (a + ks * 2), ((uint64_t)kHi << 32) | (b + ks * 2), kIdescL2, (c | ks) != 0, el);
          }
        mma_commit(bar + 40, el);
      }
      mbar_wait(bar + 32, n_run & 1);   // the enhanced image is read with generic loads below
      mbar_wait(bar + 40, n_run & 1);
      tc_fence_after_sync();
      // linear_2 epilogue (encoders.py:70), Fold (patch_processors.py:69-71) and the residual (fortitran.py:228): one
      // thread per token (warps 0..11: row tile warp / 4, lane quadrant warp % 4)
      if (warp < 12) {
        const int t = (warp >> 2) * 128 + (warp & 3) * 32 + (tid & 31);
        uint32_t acc[8];
        tmem_ld8p(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (warp >> 2) * 16, acc);
        tmem_wait_ld();
        if (t < kS) {
          const int pi = t / kTokW, pj = t - pi * kTokW;
#pragma unroll
          for (int f = 0; f < kPatchLen; ++f) {
            const int a = f / kPatchW, b = f - a * kPatchW;
            const int r = kPatchH * pi + a, c = kPatchW * pj + b;
            in[(r + 1) * kPW + c + 1] = __uint_as_float(acc[f]) + l2b[f] + es[r * kGridW + c];
          }
        }
      }
      // the staged image overwrote the zero guards between mid groups 1 | 2 and 2 | 3: the conv stack reads them as padding
      for (int i = tid; i < 2 * 64; i += kThreads) {
        const int g = i >> 6;   // boundary between groups g + 1 and g + 2: back guard of the first + front guard of the second = 1024 bytes
        *reinterpret_cast<uint4*>(smem + OFF_MID + (g + 2) * kPlaneBytes - kPosGuard * 16 + (i & 63) * 16) = make_uint4(0, 0, 0, 0);
      }
      tc_fence_before_sync();
      __syncthreads();
#ifdef AFT_TC_TIMELINE
      if (st_on) g_conv_tl[21] = clock64();
#endif
      stack_run(smem, sb, tmem, bar, n_run);                    // fortitran.py:231
#ifdef AFT_TC_TIMELINE
      if (st_on) g_conv_tl[22] = clock64();
#endif
      // torch.complex (fortitran.py:180): the real pass parks its result in shared memory; the imaginary pass interleaves
      // both as complex64 in a shared staging row (13,440 bytes), which one thread then hands to the copy engine: one
      // bulk copy per destination (the caller's buffer and, in the fused all-gather, the peers' gather buffers over
      // NVLink).  The stores to up to eight GPUs no longer occupy the SM's store path: they drain while the next sample
      // is computed, and the staging row is only rewritten a whole sample later (bulk_wait_read at the start of a part 1).
      if (part == 0) {
        for (int i = tid; i < kPix; i += kThreads) re_keep[i] = res[i];
        if (tid == 0) bulk_wait_read();   // the previous sample's copies have read the staging row (ordered before the
                                          // staging writes below by the barriers of the next stack run)
      } else {
        for (int i = tid; i < kPix / 2; i += kThreads) {
          const float2 re2 = reinterpret_cast<const float2*>(re_keep)[i], im2 = reinterpret_cast<const float2*>(res)[i];
          reinterpret_cast<float4*>(smem + kStageOff)[i] = make_float4(re2.x, im2.x, re2.y, im2.y);
        }
        fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0)
          for (int d = 0; d < out.n; ++d) bulk_s2g(out.ptr[d] + sample * kPix, sb + kStageOff, kPix * sizeof(float2));
      }
      __syncthreads();
#ifdef AFT_TC_TIMELINE
      if (st_on) g_conv_tl[23] = clock64();
#endif
    }
  }
  if (tid == 0) bulk_wait_all();   // the last estimates have left
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// fp32 ConvEnhancer parameters (SIMT packing, ConvPack) -> tensor-core pack (conv_tc.cuh layout)
__global__ void conv_tc_pack_kernel(ConvPack src, uint8_t* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  __nv_bfloat16* w2 = reinterpret_cast<__nv_bfloat16*>(dst + kPkW2);
  __nv_bfloat16* w3 = reinterpret_cast<__nv_bfloat16*>(dst + kPkW3);
  float* f = reinterpret_cast<float*>(dst + kPkF32);
  if (i < 5 * 512) {           // conv2: [tap pair][half = tap of the pair][cout 32][cin 8]; the tenth tap is zero
    const int pr = i / 512, rem = i % 512, half = rem / 256, co = (rem % 256) / 8, j = rem % 8;
    const int t = 2 * pr + half;
    w2[i] = __float2bfloat16(t < 9 ? src.w1[(t * 8 + j) * 32 + co] : 0.f);   // src.w1 is [tap][cin 8][cout 32]
  }
  if (i < 6 * 512) {           // conv3: [dy][kstep][half][n 32 = dx * 8 + cout][8]; n >= 24 is zero
    const int dk = i / 512, rem = i % 512, half = rem / 256, n = (rem % 256) / 8, j = rem % 8;
    const int dy = dk >> 1, ks = dk & 1, ci = ks * 16 + half * 8 + j, dx = n >> 3, co = n & 7;
    w3[i] = __float2bfloat16(n < 24 ? src.w2[((dy * 3 + dx) * 32 + ci) * 8 + co] : 0.f);   // src.w2 is [tap][cin 32][cout 8]
  }
  if (i < 72) { f[kF_w0 + i] = src.w0[i]; f[kF_w3 + i] = src.w3[i]; }
  if (i < 8) { f[kF_b0 + i] = src.b0[i]; f[kF_b2 + i] = src.b2[i]; }
  if (i < 32) f[kF_b1 + i] = src.b1[i];
  if (i == 0) f[kF_b3] = src.b3[0];
}

}  // namespace

size_t conv_tc_pack_bytes() { return kPkBytes; }

// diagnostics (-DAFT_TC_TIMELINE builds): prints the phase durations of the stamped stack run
void conv_tc_dump_timeline() {
#ifdef AFT_TC_TIMELINE
  unsigned long long t[32];
  if (cudaMemcpyFromSymbol(t, g_conv_tl, sizeof(t)) != cudaSuccess) return;
  const char* names[] = {"conv1", "conv2 issue", "conv2 wait", "conv2 epilogue", "conv3 issue", "conv3 wait", "conv3 epilogue", "conv4"};
  for (int i = 0; i < 8; ++i) fprintf(stderr, "CONV %-15s %llu\n", names[i], t[i + 1] - t[i]);
  fprintf(stderr, "CONV head: linear_2+fold %llu | stack %llu | store %llu\n", t[21] - t[20], t[22] - t[21], t[23] - t[22]);
  fprintf(stderr, "CONV frontend: upsample %llu | stack %llu | enh store+tokens %llu | linear_1 %llu\n", t[11] - t[10], t[12] - t[11], t[13] - t[12], t[14] - t[13]);
#endif
}

bool conv_tc_pack(const ConvPack& src, void* dst, cudaStream_t st) {
  conv_tc_pack_kernel<<<(9 * 512 + 255) / 256, 256, 0, st>>>(src, static_cast<uint8_t*>(dst));
  count_launch();
  return check_launch("conv_tc_pack_kernel");
}

bool launch_frontend_tc(const FrontPack& p, const void* pack, const float2* pilots, const float* snr, const float* ds,
                        const float* dop, float* zbuf, float* enh, __nv_bfloat16* hb, int64_t nsamples, int sm_count, cudaStream_t st) {
  if (cudaFuncSetAttribute(frontend_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStackSmemBytes) != cudaSuccess) {
    set_error("frontend_tc: cannot opt in to %d bytes of shared memory: %s", kStackSmemBytes, cudaGetErrorString(cudaGetLastError()));
    return false;
  }
  if (nsamples <= 0) return true;
  const int64_t nseq = 2 * nsamples;
  if (p.adaptive) {
    if (p.h1 > kMaxAdaHidden || p.h2 > kMaxAdaHidden) { set_error("adapter hidden sizes exceed %d", kMaxAdaHidden); return false; }
    const int64_t groups = (nsamples + kAdaGroup - 1) / kAdaGroup;
    adapter_kernel<<<(unsigned)(groups < sm_count ? groups : sm_count), kAdaThreads, 0, st>>>(p, snr, ds, dop, zbuf, nsamples);
    count_launch();
    if (!check_launch("adapter_kernel")) return false;
  }
  frontend_tc_kernel<<<(unsigned)(nseq < sm_count ? nseq : sm_count), kThreads, kStackSmemBytes, st>>>(
      p, static_cast<const uint8_t*>(pack), pilots, zbuf, enh, hb, nseq);
  count_launch();
  return check_launch("frontend_tc_kernel");
}

bool launch_head_tc(const HeadPack& p, const void* pack, const void* himg, const float* enh, const OutDst& out, int64_t nsamples,
                    int sm_count, cudaStream_t st) {
  if (cudaFuncSetAttribute(head_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStackSmemBytes) != cudaSuccess) {
    set_error("head_tc: cannot opt in to %d bytes of shared memory: %s", kStackSmemBytes, cudaGetErrorString(cudaGetLastError()));
    return false;
  }
  if (nsamples <= 0) return true;
  head_tc_kernel<<<(unsigned)(nsamples < sm_count ? nsamples : sm_count), kThreads, kStackSmemBytes, st>>>(
      p, static_cast<const uint8_t*>(pack), static_cast<const uint8_t*>(himg), enh, out, nsamples);
  count_launch();
  return check_launch("head_tc_kernel");
}

}  // namespace aft
