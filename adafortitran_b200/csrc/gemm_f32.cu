// fp32 CUDA-core GEMM of the AFT_FP32 path:  C[M,N] = A[M,K] . W[N,K]^T + bias  with the epilogues the
// post-norm encoder layer needs (reference: torch _transformer_encoder_layer_fwd as used by
// src/models/blocks/encoders.py:69):
//   kEpiBias       : QKV projection
//   kEpiBiasAct    : FFN linear1 + GELU(erf) / ReLU
//   kEpiBiasResLn  : out_proj / linear2 + residual + LayerNorm (N == 128 == one tile, statistics tile-local)
// and the two epilogues of the training forward (train.cuh), which add dropout and keep the pre-LN sum / the
// pre-activation for the backward; with p = 0 they compute exactly what kEpiBiasResLn / kEpiBiasAct compute.
// Plain FMA accumulation (no TF32): the fp32 parity gate is 1e-4 normwise.
#include "train.cuh"

namespace aft {

namespace {

constexpr int BM = 128, BN = 128, BK = 16, PITCH = BM + 4;

template <int EPI>
__global__ void __launch_bounds__(256)
gemm_f32_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ bias,
                float* C, int64_t M, int N, int K, int act, const float* residual,
                const float* __restrict__ gamma, const float* __restrict__ beta, TrainEpi te) {
  constexpr bool kResLn = EPI == kEpiBiasResLn || EPI == kEpiTrainResLn;
  __shared__ __align__(16) float As[BK][PITCH];
  __shared__ __align__(16) float Bs[BK][PITCH];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int col0 = blockIdx.y * BN;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = tid + i * 256;
      const int r = idx >> 2, kq = (idx & 3) * 4;
      float4 va = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row0 + r < M) va = *reinterpret_cast<const float4*>(A + (row0 + r) * K + k0 + kq);
      As[kq + 0][r] = va.x; As[kq + 1][r] = va.y; As[kq + 2][r] = va.z; As[kq + 3][r] = va.w;
      const float4 vb = *reinterpret_cast<const float4*>(W + (int64_t)(col0 + r) * K + k0 + kq);
      Bs[kq + 0][r] = vb.x; Bs[kq + 1][r] = vb.y; Bs[kq + 2][r] = vb.z; Bs[kq + 3][r] = vb.w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

  // thread's columns: col0 + tx*4 + {0..3} and col0 + 64 + tx*4 + {0..3}
  const int cA = col0 + tx * 4, cB = col0 + 64 + tx * 4;
  const float4 biasA = *reinterpret_cast<const float4*>(bias + cA);
  const float4 biasB = *reinterpret_cast<const float4*>(bias + cB);
  const float bv[8] = {biasA.x, biasA.y, biasA.z, biasA.w, biasB.x, biasB.y, biasB.z, biasB.w};
  float gv[8], be[8];
  if (kResLn) {
    const float4 gA = *reinterpret_cast<const float4*>(gamma + cA), gB = *reinterpret_cast<const float4*>(gamma + cB);
    const float4 eA = *reinterpret_cast<const float4*>(beta + cA), eB = *reinterpret_cast<const float4*>(beta + cB);
    gv[0] = gA.x; gv[1] = gA.y; gv[2] = gA.z; gv[3] = gA.w; gv[4] = gB.x; gv[5] = gB.y; gv[6] = gB.z; gv[7] = gB.w;
    be[0] = eA.x; be[1] = eA.y; be[2] = eA.z; be[3] = eA.w; be[4] = eB.x; be[5] = eB.y; be[6] = eB.z; be[7] = eB.w;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = row0 + ty * 8 + i;
    const bool live = m < M;   // warp-uniform per half-warp; shuffles below are executed by all lanes
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = acc[i][j] + bv[j];
    if (EPI == kEpiTrainAct && live) {
      *reinterpret_cast<float4*>(te.aux + m * N + cA) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(te.aux + m * N + cB) = make_float4(v[4], v[5], v[6], v[7]);
    }
    if (EPI == kEpiBiasAct || EPI == kEpiTrainAct) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = act == AFT_ACT_GELU ? gelu_erf(v[j]) : fmaxf(v[j], 0.f);
    }
    if ((EPI == kEpiTrainAct || EPI == kEpiTrainResLn) && te.drop.thresh != 0u) {
      // element index row * N + col within the sequence; cA and cB are multiples of 4: one Philox call each
      const uint32_t seq = (uint32_t)(m / kS), row = (uint32_t)(m - (int64_t)seq * kS);
      const float4 ka = te.drop.mult4((row * N + cA) >> 2, seq, te.layer_site);
      const float4 kb = te.drop.mult4((row * N + cB) >> 2, seq, te.layer_site);
      v[0] *= ka.x; v[1] *= ka.y; v[2] *= ka.z; v[3] *= ka.w;
      v[4] *= kb.x; v[5] *= kb.y; v[6] *= kb.z; v[7] *= kb.w;
    }
    if (kResLn) {
      if (live) {
        const float4 rA = *reinterpret_cast<const float4*>(residual + m * N + cA);
        const float4 rB = *reinterpret_cast<const float4*>(residual + m * N + cB);
        v[0] += rA.x; v[1] += rA.y; v[2] += rA.z; v[3] += rA.w;
        v[4] += rB.x; v[5] += rB.y; v[6] += rB.z; v[7] += rB.w;
        if (EPI == kEpiTrainResLn) {
          *reinterpret_cast<float4*>(te.aux + m * N + cA) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(te.aux + m * N + cB) = make_float4(v[4], v[5], v[6], v[7]);
        }
      }
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[j];
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
      const float mean = s * (1.0f / BN);
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float d = v[j] - mean; q = fmaf(d, d, q); }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) q += __shfl_xor_sync(0xffffffffu, q, off);
      const float rstd = rsqrtf(q * (1.0f / BN) + 1e-5f);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (v[j] - mean) * rstd * gv[j] + be[j];
    }
    if (live) {
      *reinterpret_cast<float4*>(C + m * N + cA) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(C + m * N + cB) = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

// The same tiling for arbitrary N and K (bias epilogue only): guarded scalar loads / stores at the edges.  Used by the
// shape-generic frontend for the pilot upsampler Linear(P, H*W) (reference src/models/fortitran.py:86,203), whose extents
// follow the grid (BASELINE config 5: 3276 -> 45864).
__global__ void __launch_bounds__(256)
gemm_f32_edge_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ bias, float* C, int64_t M, int N, int K) {
  __shared__ __align__(16) float As[BK][PITCH];
  __shared__ __align__(16) float Bs[BK][PITCH];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int col0 = blockIdx.y * BN;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {   // 128 rows x 16 k per operand, k fastest: consecutive threads read consecutive k
      const int idx = tid + i * 256;
      const int r = idx >> 4, kk = idx & 15;
      const bool kin = k0 + kk < K;
      As[kk][r] = (kin && row0 + r < M) ? A[(row0 + r) * K + k0 + kk] : 0.f;
      Bs[kk][r] = (kin && col0 + r < N) ? W[(int64_t)(col0 + r) * K + k0 + kk] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = row0 + ty * 8 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = col0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + j - 4);
      if (c < N) C[m * N + c] = acc[i][j] + bias[c];
    }
  }
}

}  // namespace

bool launch_gemm_f32_any(const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K, cudaStream_t st) {
  if (M <= 0) return true;
  const dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN));
  gemm_f32_edge_kernel<<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K);
  count_launch();
  return check_launch("gemm_f32_edge_kernel");
}

bool launch_gemm_f32(int epi, const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K,
                     int act, const float* residual, const float* gamma, const float* beta, cudaStream_t st) {
  if (M <= 0) return true;
  if (N % BN != 0 || K % BK != 0 || (epi == kEpiBiasResLn && N != BN)) {
    set_error("gemm_f32: unsupported shape N=%d K=%d epi=%d", N, K, epi);
    return false;
  }
  const dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)(N / BN));
  const TrainEpi none{};
  switch (epi) {
    case kEpiBias:
      gemm_f32_kernel<kEpiBias><<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K, act, residual, gamma, beta, none);
      break;
    case kEpiBiasAct:
      gemm_f32_kernel<kEpiBiasAct><<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K, act, residual, gamma, beta, none);
      break;
    default:
      gemm_f32_kernel<kEpiBiasResLn><<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K, act, residual, gamma, beta, none);
      break;
  }
  count_launch();
  return check_launch("gemm_f32_kernel");
}

bool launch_gemm_f32_train(int epi, const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K,
                           int act, const float* residual, const float* gamma, const float* beta, const TrainEpi& te,
                           cudaStream_t st) {
  if (M <= 0) return true;
  if (N % BN != 0 || K % BK != 0 || (epi == kEpiTrainResLn && N != BN) || (epi != kEpiTrainResLn && epi != kEpiTrainAct)) {
    set_error("gemm_f32_train: unsupported shape N=%d K=%d epi=%d", N, K, epi);
    return false;
  }
  const dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)(N / BN));
  if (epi == kEpiTrainResLn)
    gemm_f32_kernel<kEpiTrainResLn><<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K, act, residual, gamma, beta, te);
  else
    gemm_f32_kernel<kEpiTrainAct><<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K, act, residual, gamma, beta, te);
  count_launch();
  return check_launch("gemm_f32_kernel");
}

}  // namespace aft
