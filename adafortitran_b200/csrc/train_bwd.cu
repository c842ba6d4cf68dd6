// Backward of the AFT_FP32 training path (reference default geometry): gradients of every parameter for
// grad_out = dL/d(out), written into one flat fp32 buffer in the order of include/aft.h.
//
// Reverse order over the real and imaginary sequences of the batch together (they share the weights, so their
// contributions sum):  head (final_refiner conv stack, fold, linear_2)  ->  encoder layers L-1 .. 0  ->  front
// (linear_1 + positional table, unfold, initial_enhancer, pilot up-sampler, channel adapter).  The ConvEnhancer
// activations, the up-sampled image, the tokens and the adapter MLP activations are recomputed here; the encoder
// activations come from the workspace the training forward filled (train.cuh).
//
// Determinism: no float atomics.  Every weight / bias gradient is a sum over rows (tokens or sequences) computed as
// per-chunk partials in the workspace and then summed over the chunks in a fixed order, so the same inputs and seed
// give bit-identical gradients.  The long scalar sums (bias, conv, small-matrix gradients) and the sums over chunks
// accumulate in fp64; the GEMM tiles accumulate in fp32.
#include "train.cuh"

namespace aft {

namespace {

constexpr int BM = 128, BN = 128, BK = 16, PITCH = BM + 4;

unsigned blocks(int64_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

// ---------------------------------------------------------------------------------------------
// GEMMs of the backward (fp32 FMA, the 128x128x16 tiling of gemm_f32.cu)
//   MODE 0:  C[M][Nc] (+)= A[M][R] . B[R][Nc]                 dX = dY . W
//   MODE 1:  P[z][Nr][Nc] = sum_{m in chunk z} A[m][Nr] B[m][Nc]   dW = dY^T . X  (partials, one per row chunk)
// ---------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256)
bwd_gemm_kernel(const float* __restrict__ A, const float* __restrict__ B, float* C, int64_t M, int R, int Nr, int Nc,
                int64_t chunk_rows, int accumulate) {
  __shared__ __align__(16) float As[BK][PITCH];
  __shared__ __align__(16) float Bs[BK][PITCH];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * BM;   // MODE 0: rows of A / C; MODE 1: rows of dW (columns of A)
  const int col0 = blockIdx.y * BN;
  int64_t k_begin = 0, k_end = R;
  if (MODE == 1) {
    k_begin = (int64_t)blockIdx.z * chunk_rows;
    k_end = k_begin + chunk_rows < M ? k_begin + chunk_rows : M;
  }
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  for (int64_t k0 = k_begin; k0 < k_end; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = tid + i * 256;
      if (MODE == 0) {
        const int r = idx >> 2, kq = (idx & 3) * 4;
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + r < M) va = *reinterpret_cast<const float4*>(A + (row0 + r) * R + k0 + kq);
        As[kq + 0][r] = va.x; As[kq + 1][r] = va.y; As[kq + 2][r] = va.z; As[kq + 3][r] = va.w;
      } else {
        const int kk = idx >> 5, c4 = (idx & 31) * 4;
        *reinterpret_cast<float4*>(&As[kk][c4]) = *reinterpret_cast<const float4*>(A + (k0 + kk) * Nr + row0 + c4);
      }
      const int kk = idx >> 5, c4 = (idx & 31) * 4;
      *reinterpret_cast<float4*>(&Bs[kk][c4]) = *reinterpret_cast<const float4*>(B + (k0 + kk) * Nc + col0 + c4);
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
  const int cA = col0 + tx * 4, cB = col0 + 64 + tx * 4;
  float* out = MODE == 1 ? C + (int64_t)blockIdx.z * Nr * Nc : C;
  const int64_t rows = MODE == 1 ? Nr : M;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = row0 + ty * 8 + i;
    if (m >= rows) continue;
    float4 va = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    float4 vb = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
    float* pa = out + m * Nc + cA;
    float* pb = out + m * Nc + cB;
    if (MODE == 0 && accumulate) {
      const float4 oa = *reinterpret_cast<const float4*>(pa), ob = *reinterpret_cast<const float4*>(pb);
      va.x += oa.x; va.y += oa.y; va.z += oa.z; va.w += oa.w;
      vb.x += ob.x; vb.y += ob.y; vb.z += ob.z; vb.w += ob.w;
    }
    *reinterpret_cast<float4*>(pa) = va;
    *reinterpret_cast<float4*>(pb) = vb;
  }
}

// out[i] = sum_z part[z * stride + i], z in increasing order
__global__ void k_reduce(const float* __restrict__ part, int nz, int64_t stride, int64_t count, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double s = 0.0;
  for (int z = 0; z < nz; ++z) s += part[z * stride + i];
  out[i] = (float)s;
}

// part[z][n*K + k] = sum_{m in chunk z} A[m*lda + n] * (B ? B[m*ldb + k] : 1)   (small weight / bias gradients)
__global__ void k_wgrad_rows(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, int N, int K,
                             int64_t M, int64_t rows, float* __restrict__ part) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (int64_t)N * K) return;
  const int n = (int)(o / K), k = (int)(o - (int64_t)n * K);
  const int64_t m0 = (int64_t)blockIdx.y * rows;
  const int64_t m1 = m0 + rows < M ? m0 + rows : M;
  double acc = 0.0;   // long sums with cancellation: accumulated in fp64, stored as fp32 partials
  if (B) {
    for (int64_t m = m0; m < m1; ++m) acc = fma((double)A[m * lda + n], (double)B[m * ldb + k], acc);
  } else {
    for (int64_t m = m0; m < m1; ++m) acc += A[m * lda + n];
  }
  part[(int64_t)blockIdx.y * N * K + o] = (float)acc;
}

// ---------------------------------------------------------------------------------------------
// ConvEnhancer pieces on [nseq][c][120][14] planes in global memory; weights in the packed [tap][cin][cout] layout
// ---------------------------------------------------------------------------------------------
__global__ void k_conv_fwd(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ b, float* __restrict__ Y,
                           int cin, int cout, int relu, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nseq * cout * kPix) return;
  const int p = (int)(i % kPix);
  const int64_t sc = i / kPix;
  const int co = (int)(sc % cout);
  const int64_t seq = sc / cout;
  const int r = p / kGridW, c = p - r * kGridW;
  float acc = b[co];
  const float* xs = X + seq * cin * kPix;
  for (int ci = 0; ci < cin; ++ci)
    for (int t = 0; t < 9; ++t) {
      const int rr = r + t / 3 - 1, cc = c + t % 3 - 1;
      if (rr < 0 || rr >= kGridH || cc < 0 || cc >= kGridW) continue;
      acc = fmaf(W[(t * cin + ci) * cout + co], xs[ci * kPix + rr * kGridW + cc], acc);
    }
  Y[i] = relu ? fmaxf(acc, 0.f) : acc;
}

// dX[seq][ci][p] = (sum_co sum_tap W . dY shifted) * (mask ? [mask > 0] : 1)
__global__ void k_conv_dgrad(const float* __restrict__ dY, const float* __restrict__ W, const float* __restrict__ mask,
                             float* __restrict__ dX, int cin, int cout, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nseq * cin * kPix) return;
  const int p = (int)(i % kPix);
  const int64_t sc = i / kPix;
  const int ci = (int)(sc % cin);
  const int64_t seq = sc / cin;
  if (mask && !(mask[i] > 0.f)) { dX[i] = 0.f; return; }
  const int r = p / kGridW, c = p - r * kGridW;
  const float* ds = dY + seq * cout * kPix;
  float acc = 0.f;
  for (int t = 0; t < 9; ++t) {
    const int rr = r - t / 3 + 1, cc = c - t % 3 + 1;
    if (rr < 0 || rr >= kGridH || cc < 0 || cc >= kGridW) continue;
    const float* w = W + (t * cin + ci) * cout;
    for (int co = 0; co < cout; ++co) acc = fmaf(w[co], ds[co * kPix + rr * kGridW + cc], acc);
  }
  dX[i] = acc;
}

// part[z][o]: o < cout*cin*9 -> weight gradient in torch layout [co][ci][3][3]; o >= -> bias gradient of co
__global__ void k_conv_wgrad(const float* __restrict__ dY, const float* __restrict__ X, int cin, int cout, int64_t nseq,
                             int64_t spc, float* __restrict__ part) {
  const int nw = cout * cin * 9, n = nw + cout;
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n) return;
  const int64_t s0 = (int64_t)blockIdx.y * spc;
  const int64_t s1 = s0 + spc < nseq ? s0 + spc : nseq;
  double acc = 0.0;   // sums over whole images with cancellation: accumulated in fp64
  if (o < nw) {
    const int co = o / (cin * 9), ci = (o / 9) % cin, t = o % 9;
    const int dy = t / 3 - 1, dx = t % 3 - 1;
    const int r0 = dy < 0 ? 1 : 0, r1 = dy > 0 ? kGridH - 1 : kGridH;
    const int c0 = dx < 0 ? 1 : 0, c1 = dx > 0 ? kGridW - 1 : kGridW;
    for (int64_t s = s0; s < s1; ++s) {
      const float* g = dY + (s * cout + co) * kPix;
      const float* x = X + (s * cin + ci) * kPix;
      for (int r = r0; r < r1; ++r)
        for (int c = c0; c < c1; ++c) acc = fma((double)g[r * kGridW + c], (double)x[(r + dy) * kGridW + c + dx], acc);
    }
  } else {
    const int co = o - nw;
    for (int64_t s = s0; s < s1; ++s) {
      const float* g = dY + (s * cout + co) * kPix;
      for (int p = 0; p < kPix; ++p) acc += g[p];
    }
  }
  part[(int64_t)blockIdx.y * n + o] = (float)acc;
}

// ---------------------------------------------------------------------------------------------
// head / front element-wise pieces
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int pix_of(int t, int f) {   // token t, patch element f -> grid pixel (Unfold / Fold 3x2)
  const int pi = t / kTokW, pj = t - pi * kTokW;
  const int a = f / kPatchW, b = f - a * kPatchW;
  return (kPatchH * pi + a) * kGridW + kPatchW * pj + b;
}

__global__ void k_split_grad(const float2* __restrict__ g, float* __restrict__ out, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // (seq, pix)
  if (i >= nseq * kPix) return;
  const int64_t seq = i / kPix;
  const int p = (int)(i - seq * kPix);
  const float2 v = g[(seq >> 1) * kPix + p];
  out[i] = (seq & 1) ? v.y : v.x;
}

// z = enh + Fold(h . l2_w^T + l2_b): the input of final_refiner
__global__ void k_head_input(const float* __restrict__ h, const float* __restrict__ enh, const float* __restrict__ l2w,
                             const float* __restrict__ l2b, float* __restrict__ z, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // (seq, token, f)
  if (i >= nseq * kS * kPatchLen) return;
  const int f = (int)(i % kPatchLen);
  const int64_t m = i / kPatchLen;
  const int t = (int)(m % kS);
  const int64_t seq = m / kS;
  float acc = 0.f;
  for (int c = 0; c < kD; ++c) acc = fmaf(h[m * kD + c], l2w[f * kD + c], acc);
  const int p = pix_of(t, f);
  z[seq * kPix + p] = enh[seq * kPix + p] + (acc + l2b[f]);
}

// dl2[m][f] = dz[seq][pix(t, f)]
__global__ void k_unfold(const float* __restrict__ dz, float* __restrict__ dl2, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nseq * kS * kPatchLen) return;
  const int f = (int)(i % kPatchLen);
  const int64_t m = i / kPatchLen;
  const int t = (int)(m % kS);
  dl2[i] = dz[(m / kS) * kPix + pix_of(t, f)];
}

// dh[m][c] = sum_f dl2[m][f] l2_w[f][c]
__global__ void k_dh_from_l2(const float* __restrict__ dl2, const float* __restrict__ l2w, float* __restrict__ dh, int64_t M) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * kD) return;
  const int64_t m = i / kD;
  const int c = (int)(i - m * kD);
  float acc = 0.f;
#pragma unroll
  for (int f = 0; f < kPatchLen; ++f) acc = fmaf(dl2[m * kPatchLen + f], l2w[f * kD + c], acc);
  dh[i] = acc;
}

// LayerNorm backward (one warp per row) with the dropout mask of the branch that entered the residual add:
//   s = res + drop(f),  y = LN(s):   dres = ds,  dproj = ds * mult,  tmp = dy * xhat  (for d gamma)
__global__ void k_ln_bwd(const float* __restrict__ dy, const float* __restrict__ s, const float* __restrict__ gamma,
                         float* __restrict__ dres, float* __restrict__ dproj, float* __restrict__ tmp, int64_t M, DropCfg drop,
                         uint32_t layer_site) {
  const int64_t m = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (m >= M) return;
  const float4 sv = *reinterpret_cast<const float4*>(s + m * kD + lane * 4);
  const float4 gv = *reinterpret_cast<const float4*>(dy + m * kD + lane * 4);
  const float4 wv = *reinterpret_cast<const float4*>(gamma + lane * 4);
  const float x[4] = {sv.x, sv.y, sv.z, sv.w}, d[4] = {gv.x, gv.y, gv.z, gv.w}, w[4] = {wv.x, wv.y, wv.z, wv.w};
  float sum = x[0] + x[1] + x[2] + x[3];
  for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
  const float mean = sum * (1.0f / kD);
  float q = 0.f;
  for (int j = 0; j < 4; ++j) { const float t = x[j] - mean; q = fmaf(t, t, q); }
  for (int off = 16; off > 0; off >>= 1) q += __shfl_xor_sync(0xffffffffu, q, off);
  const float rstd = rsqrtf(q * (1.0f / kD) + 1e-5f);
  float xh[4], g[4], sg = 0.f, sgx = 0.f;
  for (int j = 0; j < 4; ++j) {
    xh[j] = (x[j] - mean) * rstd;
    g[j] = d[j] * w[j];
    sg += g[j];
    sgx = fmaf(g[j], xh[j], sgx);
  }
  for (int off = 16; off > 0; off >>= 1) {
    sg += __shfl_xor_sync(0xffffffffu, sg, off);
    sgx += __shfl_xor_sync(0xffffffffu, sgx, off);
  }
  sg *= (1.0f / kD);
  sgx *= (1.0f / kD);
  float o[4];
  for (int j = 0; j < 4; ++j) o[j] = rstd * (g[j] - sg - xh[j] * sgx);
  *reinterpret_cast<float4*>(dres + m * kD + lane * 4) = make_float4(o[0], o[1], o[2], o[3]);
  *reinterpret_cast<float4*>(tmp + m * kD + lane * 4) = make_float4(d[0] * xh[0], d[1] * xh[1], d[2] * xh[2], d[3] * xh[3]);
  float4 k = make_float4(1.f, 1.f, 1.f, 1.f);
  if (drop.thresh != 0u) {
    const uint32_t seq = (uint32_t)(m / kS), row = (uint32_t)(m % kS);
    k = drop.mult4((row * kD + lane * 4) >> 2, seq, layer_site);
  }
  *reinterpret_cast<float4*>(dproj + m * kD + lane * 4) = make_float4(o[0] * k.x, o[1] * k.y, o[2] * k.z, o[3] * k.w);
}

__device__ __forceinline__ float act_fwd(float x, int act) { return act == AFT_ACT_GELU ? gelu_erf(x) : fmaxf(x, 0.f); }
__device__ __forceinline__ float act_grad(float x, int act) {
  if (act != AFT_ACT_GELU) return x > 0.f ? 1.f : 0.f;
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * 0.39894228040143267794f * expf(-0.5f * x * x);
}

// mode 0: a = drop(act(u))  (the linear2 input of the forward);  mode 1: da <- da * mult * act'(u)  (in place)
__global__ void k_act(const float* __restrict__ u, float* __restrict__ io, int64_t M, int act, int mode, DropCfg drop,
                      uint32_t layer_site) {
  const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // 4 consecutive elements of a row
  if (i4 >= M * kFF / 4) return;
  const int64_t m = i4 / (kFF / 4);
  const int c = (int)(i4 - m * (kFF / 4)) * 4;
  float4 k = make_float4(1.f, 1.f, 1.f, 1.f);
  if (drop.thresh != 0u) {
    const uint32_t seq = (uint32_t)(m / kS), row = (uint32_t)(m % kS);
    k = drop.mult4((row * kFF + c) >> 2, seq, layer_site);
  }
  const float4 uv = *reinterpret_cast<const float4*>(u + i4 * 4);
  const float x[4] = {uv.x, uv.y, uv.z, uv.w}, kk[4] = {k.x, k.y, k.z, k.w};
  float r[4];
  if (mode == 0) {
    for (int j = 0; j < 4; ++j) r[j] = act_fwd(x[j], act) * kk[j];
  } else {
    const float4 dv = *reinterpret_cast<const float4*>(io + i4 * 4);
    const float d[4] = {dv.x, dv.y, dv.z, dv.w};
    for (int j = 0; j < 4; ++j) r[j] = d[j] * kk[j] * act_grad(x[j], act);
  }
  *reinterpret_cast<float4*>(io + i4 * 4) = make_float4(r[0], r[1], r[2], r[3]);
}

// ---------------------------------------------------------------------------------------------
// attention backward: one CTA per (sequence, head), Q (pre-scaled), K, V, dO of the head in shared memory.
//   pass 1, thread = query row i:  D_i = dO_i . O_i,  dQ_i = scale * sum_j dS_ij K_j
//   pass 2, thread = key row j:    dV_j = sum_i P~_ij dO_i,  dK_j = sum_i dS_ij (scale q_i)
// with P_ij = exp(s_ij - lse_i), P~ = P * M/(1-p), dS = P * (dO_i.V_j * M/(1-p) - D_i).
// ---------------------------------------------------------------------------------------------
constexpr int kAttnThreads = 288;
constexpr size_t kAttnBwdSmem = (4 * kS * kDh + 2 * kS) * sizeof(float);

__global__ void __launch_bounds__(kAttnThreads)
attn_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ o, const float* __restrict__ lse,
                const float* __restrict__ dout, float* __restrict__ dqkv, DropCfg drop, uint32_t layer_site) {
  extern __shared__ __align__(16) float sm[];
  float* Qs = sm;
  float* Ks = Qs + kS * kDh;
  float* Vs = Ks + kS * kDh;
  float* dOs = Vs + kS * kDh;
  float* Ds = dOs + kS * kDh;
  float* Ls = Ds + kS;
  const int tid = threadIdx.x;
  const int64_t seq = blockIdx.x >> 2;
  const int head = blockIdx.x & 3;
  const float scale = 0.17677669529663688110f;
  const float* base = qkv + seq * (int64_t)kS * 3 * kD;
  const float* dob = dout + seq * (int64_t)kS * kD;
  for (int i = tid; i < kS * (kDh / 4); i += kAttnThreads) {
    const int j = i >> 3, c4 = (i & 7) * 4;
    float4 q = *reinterpret_cast<const float4*>(base + (int64_t)j * 3 * kD + head * kDh + c4);
    q.x *= scale; q.y *= scale; q.z *= scale; q.w *= scale;
    *reinterpret_cast<float4*>(Qs + j * kDh + c4) = q;
    *reinterpret_cast<float4*>(Ks + j * kDh + c4) = *reinterpret_cast<const float4*>(base + (int64_t)j * 3 * kD + kD + head * kDh + c4);
    *reinterpret_cast<float4*>(Vs + j * kDh + c4) = *reinterpret_cast<const float4*>(base + (int64_t)j * 3 * kD + 2 * kD + head * kDh + c4);
    *reinterpret_cast<float4*>(dOs + j * kDh + c4) = *reinterpret_cast<const float4*>(dob + (int64_t)j * kD + head * kDh + c4);
  }
  for (int i = tid; i < kS; i += kAttnThreads) Ls[i] = lse[(seq * kH + head) * kS + i];
  __syncthreads();
  const bool dropping = drop.thresh != 0u;
  const unsigned live = __ballot_sync(0xffffffffu, tid < kS);   // whole quads: kS is a multiple of 4

  if (tid < kS) {   // pass 1
    const int i = tid;
    float q[kDh], d[kDh], dq[kDh];
    float Di = 0.f;
    const float* orow = o + (seq * kS + i) * kD + head * kDh;
#pragma unroll
    for (int c = 0; c < kDh; ++c) {
      q[c] = Qs[i * kDh + c];
      d[c] = dOs[i * kDh + c];
      Di = fmaf(d[c], orow[c], Di);
      dq[c] = 0.f;
    }
    const float li = Ls[i];
    const uint32_t e0 = (uint32_t)(head * kS + i) * kS;
    float4 mk = make_float4(1.f, 1.f, 1.f, 1.f);
    for (int j = 0; j < kS; ++j) {
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int c = 0; c < kDh; ++c) {
        s = fmaf(q[c], Ks[j * kDh + c], s);
        dp = fmaf(d[c], Vs[j * kDh + c], dp);
      }
      if (dropping) {
        const uint32_t e = e0 + j;
        if ((e & 3) == 0) mk = drop.mult4(e >> 2, (uint32_t)seq, layer_site);
        const uint32_t w = e & 3;
        dp *= w == 0 ? mk.x : w == 1 ? mk.y : w == 2 ? mk.z : mk.w;
      }
      const float ds = expf(s - li) * (dp - Di);
#pragma unroll
      for (int c = 0; c < kDh; ++c) dq[c] = fmaf(ds, Ks[j * kDh + c], dq[c]);
    }
    Ds[i] = Di;
    float* out = dqkv + (seq * kS + i) * 3 * kD + head * kDh;
#pragma unroll
    for (int c4 = 0; c4 < kDh; c4 += 4)
      *reinterpret_cast<float4*>(out + c4) = make_float4(dq[c4] * scale, dq[c4 + 1] * scale, dq[c4 + 2] * scale, dq[c4 + 3] * scale);
  }
  __syncthreads();
  if (tid < kS) {   // pass 2
    const int j = tid;
    float k[kDh], v[kDh], dk[kDh], dv[kDh];
#pragma unroll
    for (int c = 0; c < kDh; ++c) {
      k[c] = Ks[j * kDh + c];
      v[c] = Vs[j * kDh + c];
      dk[c] = 0.f;
      dv[c] = 0.f;
    }
    // Dropout multipliers of rows i..i+3 at this key: the four keys of a quad (j & ~3 .. +3) share one Philox call per
    // row, so lane q of the quad computes row i + q and a 4x4 transpose over the quad hands every lane its own column.
    const int q4 = tid & 3;
    float mrow[4] = {1.f, 1.f, 1.f, 1.f};
    for (int i = 0; i < kS; ++i) {
      if (dropping && (i & 3) == 0) {
        const uint4 w = drop.words((uint32_t)((head * kS + i + q4) * kS + (j & ~3)) >> 2, (uint32_t)seq, layer_site);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int c = (q4 + t) & 3, src = (q4 - t) & 3;
          const uint32_t send = c == 0 ? w.x : c == 1 ? w.y : c == 2 ? w.z : w.w;
          const uint32_t got = __shfl_sync(live, send, src, 4);   // word of row i + src, column j
          const float m = got >= drop.thresh ? drop.scale : 0.f;
#pragma unroll
          for (int r = 0; r < 4; ++r) mrow[r] = src == r ? m : mrow[r];
        }
      }
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int c = 0; c < kDh; ++c) {
        s = fmaf(Qs[i * kDh + c], k[c], s);
        dp = fmaf(dOs[i * kDh + c], v[c], dp);
      }
      const float p = expf(s - Ls[i]);
      float pt = p;
      if (dropping) {
        const int r = i & 3;
        const float mult = r == 0 ? mrow[0] : r == 1 ? mrow[1] : r == 2 ? mrow[2] : mrow[3];
        pt = p * mult;
        dp *= mult;
      }
      const float ds = p * (dp - Ds[i]);
#pragma unroll
      for (int c = 0; c < kDh; ++c) {
        dv[c] = fmaf(pt, dOs[i * kDh + c], dv[c]);
        dk[c] = fmaf(ds, Qs[i * kDh + c], dk[c]);
      }
    }
    float* out = dqkv + (seq * kS + j) * 3 * kD + head * kDh;
#pragma unroll
    for (int c4 = 0; c4 < kDh; c4 += 4) {
      *reinterpret_cast<float4*>(out + kD + c4) = make_float4(dk[c4], dk[c4 + 1], dk[c4 + 2], dk[c4 + 3]);
      *reinterpret_cast<float4*>(out + 2 * kD + c4) = make_float4(dv[c4], dv[c4 + 1], dv[c4 + 2], dv[c4 + 3]);
    }
  }
}

// ---- front
// img = pilot_upsampler(x) for every sequence (xs: the real-valued pilots the forward saved)
__global__ void k_upsample(const float* __restrict__ xs, const float* __restrict__ up_wt, const float* __restrict__ up_b,
                           float* __restrict__ img, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nseq * kPix) return;
  const int64_t seq = i / kPix;
  const int p = (int)(i - seq * kPix);
  float acc = up_b[p];
  for (int k = 0; k < kPilots; ++k) acc = fmaf(up_wt[k * kPix + p], xs[seq * kPilots + k], acc);
  img[i] = acc;
}

constexpr int kMlpStride = 2 * kS + 4 * kMaxAdaHidden + 1;   // z|dz [560], h1 [64], h2 [64], dpre2 [64], dpre1 [64], c
constexpr int kMlpH1 = 2 * kS, kMlpH2 = kMlpH1 + 64, kMlpD2 = kMlpH2 + 64, kMlpD1 = kMlpD2 + 64, kMlpC = kMlpD1 + 64;

// one block per (sequence, adapter): recomputes h1, h2, z of the adapter MLP
__global__ void k_mlp_fwd(FrontPack p, const float* __restrict__ cond, float* __restrict__ buf) {
  const int64_t seq = blockIdx.x / 3;
  const int mi = blockIdx.x % 3;
  const MlpPack& mp = p.mlp[mi];
  float* b = buf + (int64_t)blockIdx.x * kMlpStride;
  const float c = cond[(seq >> 1) * 3 + mi];
  const int tid = threadIdx.x;
  if (tid < p.h1) b[kMlpH1 + tid] = fmaxf(fmaf(mp.w0[tid], c, mp.b0[tid]), 0.f);
  if (tid == 0) b[kMlpC] = c;
  __syncthreads();
  if (tid < p.h2) {
    float acc = mp.b1[tid];
    for (int k = 0; k < p.h1; ++k) acc = fmaf(mp.w1[tid * p.h1 + k], b[kMlpH1 + k], acc);
    b[kMlpH2 + tid] = fmaxf(acc, 0.f);
  }
  __syncthreads();
  for (int j = tid; j < 2 * kS; j += blockDim.x) {
    float acc = mp.b2[j];
    for (int k = 0; k < p.h2; ++k) acc = fmaf(mp.w2t[k * 2 * kS + j], b[kMlpH2 + k], acc);
    b[j] = acc;
  }
}

// tok[m][0..5] = Unfold(enh),  tok[m][6 + 2a + e] = z_a[2t + e]
__global__ void k_tokens(const float* __restrict__ enh, const float* __restrict__ mlp, float* __restrict__ tok, int in_dim, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nseq * kS * in_dim) return;
  const int f = (int)(i % in_dim);
  const int64_t m = i / in_dim;
  const int t = (int)(m % kS);
  const int64_t seq = m / kS;
  if (f < kPatchLen) {
    tok[i] = enh[seq * kPix + pix_of(t, f)];
  } else {
    const int a = (f - kPatchLen) >> 1, e = (f - kPatchLen) & 1;
    tok[i] = mlp[(seq * 3 + a) * kMlpStride + 2 * t + e];
  }
}

// dtok[m][k] = sum_c dh[m][c] l1_w[c][k]   (l1_wt is the packed [in_dim][128] transpose)
__global__ void k_dtok(const float* __restrict__ dh, const float* __restrict__ l1_wt, float* __restrict__ dtok, int in_dim, int64_t M) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * in_dim) return;
  const int64_t m = i / in_dim;
  const int k = (int)(i - m * in_dim);
  float acc = 0.f;
  for (int c = 0; c < kD; ++c) acc = fmaf(dh[m * kD + c], l1_wt[k * kD + c], acc);
  dtok[i] = acc;
}

// denh[seq][pix] += dtok[m][f] (Fold of the patch features)
__global__ void k_fold_add(const float* __restrict__ dtok, float* __restrict__ denh, int in_dim, int64_t nseq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nseq * kS * kPatchLen) return;
  const int f = (int)(i % kPatchLen);
  const int64_t m = i / kPatchLen;
  const int t = (int)(m % kS);
  denh[(m / kS) * kPix + pix_of(t, f)] += dtok[m * in_dim + f];
}

// one block per (sequence, adapter): dz from the token gradient, then back through the MLP (dpre2, dpre1 kept)
__global__ void k_mlp_bwd(FrontPack p, const float* __restrict__ dtok, int in_dim, float* __restrict__ buf) {
  const int64_t seq = blockIdx.x / 3;
  const int mi = blockIdx.x % 3;
  const MlpPack& mp = p.mlp[mi];
  float* b = buf + (int64_t)blockIdx.x * kMlpStride;
  const int tid = threadIdx.x;
  for (int j = tid; j < 2 * kS; j += blockDim.x)
    b[j] = dtok[(seq * kS + (j >> 1)) * in_dim + kPatchLen + 2 * mi + (j & 1)];
  __syncthreads();
  if (tid < p.h2) {
    float acc = 0.f;
    for (int j = 0; j < 2 * kS; ++j) acc = fmaf(mp.w2t[tid * 2 * kS + j], b[j], acc);
    b[kMlpD2 + tid] = b[kMlpH2 + tid] > 0.f ? acc : 0.f;
  }
  __syncthreads();
  if (tid < p.h1) {
    float acc = 0.f;
    for (int k = 0; k < p.h2; ++k) acc = fmaf(mp.w1[k * p.h1 + tid], b[kMlpD2 + k], acc);
    b[kMlpD1 + tid] = b[kMlpH1 + tid] > 0.f ? acc : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------
// host orchestration
// ---------------------------------------------------------------------------------------------
struct Ctx {
  const TrainWs& ws;
  float* grads;
  cudaStream_t st;
  bool ok = true;
  bool launched(const char* what, int n = 1) {
    count_launch(n);
    if (!check_launch(what)) ok = false;
    return ok;
  }
  // grads[dst .. dst + N*K) = sum over M rows (see k_wgrad_rows)
  bool wgrad_rows(const float* A, int64_t lda, const float* B, int64_t ldb, int N, int K, int64_t M, size_t dst) {
    if (!ok) return false;
    int64_t rows = (M + kMaxChunks - 1) / kMaxChunks;
    if (rows < 1) rows = 1;
    const int nz = (int)((M + rows - 1) / rows);
    k_wgrad_rows<<<dim3(blocks((int64_t)N * K), nz), 256, 0, st>>>(A, lda, B, ldb, N, K, M, rows, ws.part);
    k_reduce<<<blocks((int64_t)N * K), 256, 0, st>>>(ws.part, nz, (int64_t)N * K, (int64_t)N * K, grads + dst);
    return launched("k_wgrad_rows", 2);
  }
  // grads[dw] = dY^T X over M rows (N x K, both multiples of 128)
  bool wgrad_gemm(const float* dY, const float* X, int N, int K, int64_t M, size_t dst) {
    if (!ok) return false;
    int64_t rows = (M + kMaxChunks - 1) / kMaxChunks;
    rows = (rows + BK - 1) / BK * BK;
    if (rows < 512) rows = 512;
    const int nz = (int)((M + rows - 1) / rows);
    bwd_gemm_kernel<1><<<dim3(N / BM, K / BN, nz), 256, 0, st>>>(dY, X, ws.part, M, 0, N, K, rows, 0);
    k_reduce<<<blocks((int64_t)N * K), 256, 0, st>>>(ws.part, nz, (int64_t)N * K, (int64_t)N * K, grads + dst);
    return launched("bwd_gemm_kernel<1>", 2);
  }
  // C[M][Nc] (+)= A[M][R] . B[R][Nc]
  bool dgrad_gemm(const float* A, const float* B, float* C, int64_t M, int R, int Nc, bool accumulate) {
    if (!ok) return false;
    bwd_gemm_kernel<0><<<dim3(blocks(M, BM), Nc / BN), 256, 0, st>>>(A, B, C, M, R, 0, Nc, 0, accumulate ? 1 : 0);
    return launched("bwd_gemm_kernel<0>");
  }
  // backward of one ConvEnhancer: dy = gradient of its output, x = its input; writes the weight / bias gradients at
  // off[0..7] and the input gradient to dx.  Recomputes the activations from x.
  bool conv_stack(const ConvPack& P, const size_t* off, const float* dy, const float* x, float* dx, int64_t nseq) {
    if (!ok) return false;
    const int64_t n1 = nseq * kPix;
    k_conv_fwd<<<blocks(8 * n1), 256, 0, st>>>(x, P.w0, P.b0, ws.conv_a1, 1, 8, 1, nseq);
    k_conv_fwd<<<blocks(32 * n1), 256, 0, st>>>(ws.conv_a1, P.w1, P.b1, ws.conv_a2, 8, 32, 1, nseq);
    k_conv_fwd<<<blocks(8 * n1), 256, 0, st>>>(ws.conv_a2, P.w2, P.b2, ws.conv_a3, 32, 8, 1, nseq);
    if (!launched("k_conv_fwd", 3)) return false;
    struct Step { const float* dY; const float* X; const float* W; const float* mask; float* dX; int cin, cout; };
    const Step steps[4] = {{dy, ws.conv_a3, P.w3, ws.conv_a3, ws.g8b, 8, 1},
                           {ws.g8b, ws.conv_a2, P.w2, ws.conv_a2, ws.g32, 32, 8},
                           {ws.g32, ws.conv_a1, P.w1, ws.conv_a1, ws.g8a, 8, 32},
                           {ws.g8a, x, P.w0, nullptr, dx, 1, 8}};
    int64_t spc = (nseq + kMaxChunks - 1) / kMaxChunks;
    const int nz = (int)((nseq + spc - 1) / spc);
    for (int i = 0; i < 4; ++i) {
      const Step& s = steps[i];
      const int layer = 3 - i, nw = s.cout * s.cin * 9, n = nw + s.cout;
      k_conv_wgrad<<<dim3(blocks(n), nz), 256, 0, st>>>(s.dY, s.X, s.cin, s.cout, nseq, spc, ws.part);
      k_reduce<<<blocks(nw), 256, 0, st>>>(ws.part, nz, n, nw, grads + off[2 * layer]);
      k_reduce<<<1, 256, 0, st>>>(ws.part + nw, nz, n, s.cout, grads + off[2 * layer + 1]);
      k_conv_dgrad<<<blocks(s.cin * n1), 256, 0, st>>>(s.dY, s.W, s.mask, s.dX, s.cin, s.cout, nseq);
      if (!launched("conv backward", 4)) return false;
    }
    return true;
  }
};

}  // namespace

bool train_backward(const TrainModel& m, const float2* grad_out, int64_t batch, const DropCfg& drop, const TrainWs& ws, float* grads,
                    cudaStream_t st) {
  if (cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAttnBwdSmem) != cudaSuccess) {
    set_error("attn_bwd: cannot opt in to %zu bytes of shared memory", kAttnBwdSmem);
    return false;
  }
  const GradLayout g = grad_layout(m);
  const int64_t nseq = 2 * batch, M = nseq * kS;
  const FrontPack& F = *m.front;
  const HeadPack& Hd = *m.head;
  Ctx cx{ws, grads, st};

  // ---- head: final_refiner, Fold, linear_2
  k_split_grad<<<blocks(nseq * kPix), 256, 0, st>>>(grad_out, ws.g1, nseq);
  k_head_input<<<blocks(M * kPatchLen), 256, 0, st>>>(ws.xout, ws.enh, Hd.l2_w, Hd.l2_b, ws.conv_in, nseq);
  if (!cx.launched("head input", 2)) return false;
  if (!cx.conv_stack(Hd.refine, g.conv[1], ws.g1, ws.conv_in, ws.denh, nseq)) return false;   // denh = d(enh + rec)
  k_unfold<<<blocks(M * kPatchLen), 256, 0, st>>>(ws.denh, ws.dl2, nseq);
  if (!cx.launched("k_unfold")) return false;
  if (!cx.wgrad_rows(ws.dl2, kPatchLen, ws.xout, kD, kPatchLen, kD, M, g.l2_w)) return false;
  if (!cx.wgrad_rows(ws.dl2, kPatchLen, nullptr, 0, kPatchLen, 1, M, g.l2_b)) return false;
  k_dh_from_l2<<<blocks(M * kD), 256, 0, st>>>(ws.dl2, Hd.l2_w, ws.dh, M);
  if (!cx.launched("k_dh_from_l2")) return false;

  // ---- encoder layers, reversed.  ws.dh holds dL/d(layer output) on entry and dL/d(layer input) on exit.
  for (int l = m.num_layers - 1; l >= 0; --l) {
    const LayerPackF32& P = m.layers[l];
    const TrainLayerBufs& B = ws.L[l];
    const size_t* o = &g.layer[12 * l];   // in_w in_b out_w out_b l1_w l1_b l2_w l2_b n1_w n1_b n2_w n2_b
    const uint32_t ls = (uint32_t)l << 8;
    // LN2: s2 = y1 + drop3(f2)
    k_ln_bwd<<<blocks(M * 32), 256, 0, st>>>(ws.dh, B.s2, P.n2_w, ws.dres, ws.dproj, ws.tmp, M, drop, ls | 3u);
    if (!cx.launched("k_ln_bwd")) return false;
    if (!cx.wgrad_rows(ws.tmp, kD, nullptr, 0, kD, 1, M, o[10])) return false;
    if (!cx.wgrad_rows(ws.dh, kD, nullptr, 0, kD, 1, M, o[11])) return false;
    // linear2: f2 = a . W2^T + b2, a = drop2(act(u))
    k_act<<<blocks(M * kFF / 4), 256, 0, st>>>(B.u, ws.abuf, M, m.activation, 0, drop, ls | 2u);
    if (!cx.launched("k_act")) return false;
    if (!cx.wgrad_gemm(ws.dproj, ws.abuf, kD, kFF, M, o[6])) return false;
    if (!cx.wgrad_rows(ws.dproj, kD, nullptr, 0, kD, 1, M, o[7])) return false;
    if (!cx.dgrad_gemm(ws.dproj, P.l2_w, ws.dbig, M, kD, kFF, false)) return false;
    k_act<<<blocks(M * kFF / 4), 256, 0, st>>>(B.u, ws.dbig, M, m.activation, 1, drop, ls | 2u);
    if (!cx.launched("k_act")) return false;
    // linear1: u = y1 . W1^T + b1;  dy1 = ds2 + du . W1
    if (!cx.wgrad_gemm(ws.dbig, B.y1, kFF, kD, M, o[4])) return false;
    if (!cx.wgrad_rows(ws.dbig, kFF, nullptr, 0, kFF, 1, M, o[5])) return false;
    if (!cx.dgrad_gemm(ws.dbig, P.l1_w, ws.dres, M, kFF, kD, true)) return false;
    // LN1: s1 = x + drop1(o . Wo^T + bo)
    k_ln_bwd<<<blocks(M * 32), 256, 0, st>>>(ws.dres, B.s1, P.n1_w, ws.dh, ws.dproj, ws.tmp, M, drop, ls | 1u);
    if (!cx.launched("k_ln_bwd")) return false;
    if (!cx.wgrad_rows(ws.tmp, kD, nullptr, 0, kD, 1, M, o[8])) return false;
    if (!cx.wgrad_rows(ws.dres, kD, nullptr, 0, kD, 1, M, o[9])) return false;
    // out_proj
    if (!cx.wgrad_gemm(ws.dproj, B.o, kD, kD, M, o[2])) return false;
    if (!cx.wgrad_rows(ws.dproj, kD, nullptr, 0, kD, 1, M, o[3])) return false;
    if (!cx.dgrad_gemm(ws.dproj, P.out_w, ws.tmp, M, kD, kD, false)) return false;   // tmp = dO
    // attention
    attn_bwd_kernel<<<(unsigned)(nseq * kH), kAttnThreads, kAttnBwdSmem, st>>>(B.qkv, B.o, B.lse, ws.tmp, ws.dqkv, drop, ls | 0u);
    if (!cx.launched("attn_bwd_kernel")) return false;
    // in_proj: qkv = x . Win^T + bin;  dx = ds1 + dqkv . Win
    if (!cx.wgrad_gemm(ws.dqkv, B.x, 3 * kD, kD, M, o[0])) return false;
    if (!cx.wgrad_rows(ws.dqkv, 3 * kD, nullptr, 0, 3 * kD, 1, M, o[1])) return false;
    if (!cx.dgrad_gemm(ws.dqkv, P.in_w, ws.dh, M, 3 * kD, kD, true)) return false;
  }

  // ---- front.  ws.dh = dL/d(linear_1(tok) + b + pos)
  const int in_dim = F.in_dim;
  if (m.adaptive) {
    k_mlp_fwd<<<(unsigned)(nseq * 3), 64, 0, st>>>(F, ws.cond, ws.mlp);
    if (!cx.launched("k_mlp_fwd")) return false;
  }
  k_tokens<<<blocks(M * in_dim), 256, 0, st>>>(ws.enh, ws.mlp, ws.tok, in_dim, nseq);
  if (!cx.launched("k_tokens")) return false;
  if (!cx.wgrad_rows(ws.dh, kD, ws.tok, in_dim, kD, in_dim, M, g.l1_w)) return false;
  if (!cx.wgrad_rows(ws.dh, kD, nullptr, 0, kD, 1, M, g.l1_b)) return false;
  if (!cx.wgrad_rows(ws.dh, (int64_t)kS * kD, nullptr, 0, kS * kD, 1, nseq, g.pos)) return false;
  if (cudaMemsetAsync(grads + g.pos + (size_t)kS * kD, 0, (size_t)(m.max_seq_len - kS) * kD * sizeof(float), st) != cudaSuccess) {
    set_error("aft_backward: cudaMemsetAsync failed");
    return false;
  }
  k_dtok<<<blocks(M * in_dim), 256, 0, st>>>(ws.dh, F.l1_wt, ws.dtok, in_dim, M);
  k_fold_add<<<blocks(M * kPatchLen), 256, 0, st>>>(ws.dtok, ws.denh, in_dim, nseq);
  if (!cx.launched("k_dtok / k_fold_add", 2)) return false;
  if (m.adaptive) {
    k_mlp_bwd<<<(unsigned)(nseq * 3), 64, 0, st>>>(F, ws.dtok, in_dim, ws.mlp);
    if (!cx.launched("k_mlp_bwd")) return false;
    const int64_t ld = 3 * kMlpStride;
    for (int a = 0; a < 3; ++a) {
      const float* b = ws.mlp + a * kMlpStride;
      if (!cx.wgrad_rows(b + kMlpD1, ld, b + kMlpC, ld, m.h1, 1, nseq, g.mlp[a][0])) return false;
      if (!cx.wgrad_rows(b + kMlpD1, ld, nullptr, 0, m.h1, 1, nseq, g.mlp[a][1])) return false;
      if (!cx.wgrad_rows(b + kMlpD2, ld, b + kMlpH1, ld, m.h2, m.h1, nseq, g.mlp[a][2])) return false;
      if (!cx.wgrad_rows(b + kMlpD2, ld, nullptr, 0, m.h2, 1, nseq, g.mlp[a][3])) return false;
      if (!cx.wgrad_rows(b, ld, b + kMlpH2, ld, 2 * kS, m.h2, nseq, g.mlp[a][4])) return false;
      if (!cx.wgrad_rows(b, ld, nullptr, 0, 2 * kS, 1, nseq, g.mlp[a][5])) return false;
    }
  }
  // initial_enhancer and the up-sampler
  k_upsample<<<blocks(nseq * kPix), 256, 0, st>>>(ws.xs, F.up_wt, F.up_b, ws.conv_in, nseq);
  if (!cx.launched("k_upsample")) return false;
  if (!cx.conv_stack(F.enh, g.conv[0], ws.denh, ws.conv_in, ws.gin, nseq)) return false;
  if (!cx.wgrad_rows(ws.gin, kPix, ws.xs, kPilots, kPix, kPilots, nseq, g.up_w)) return false;
  if (!cx.wgrad_rows(ws.gin, kPix, nullptr, 0, kPix, 1, nseq, g.up_b)) return false;
  return true;
}

}  // namespace aft
