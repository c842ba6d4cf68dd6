// Training forward of the AFT_FP32 path (reference default geometry): the arithmetic of forward_chunk_f32 (aft_api.cu)
// with the dropout of nn.TransformerEncoderLayer at its four sites, and every activation the backward needs saved in
// the caller's workspace (train.cuh).  With p = 0 the output is bit-identical to aft_forward at AFT_FP32.
#include "train.cuh"

namespace aft {

namespace {

size_t align64(size_t v) { return (v + 63) / 64 * 64; }

constexpr int kAttnThreads = 288;   // 9 warps >= 280 query rows

// attn_f32_kernel (attn_f32.cu) plus site-0 dropout on the probabilities and the log-sum-exp of every (row, head)
__global__ void __launch_bounds__(kAttnThreads)
attn_train_kernel(const float* __restrict__ qkv, float* __restrict__ out, float* __restrict__ lse, DropCfg drop,
                  uint32_t layer_site) {
  extern __shared__ __align__(16) float sm[];
  float* Ks = sm;
  float* Vs = sm + kS * kDh;
  const int tid = threadIdx.x;
  const int64_t seq = blockIdx.x >> 2;
  const int head = blockIdx.x & 3;
  const float* base = qkv + seq * (int64_t)kS * 3 * kD;

  for (int i = tid; i < kS * (kDh / 4); i += kAttnThreads) {
    const int j = i >> 3, c4 = (i & 7) * 4;
    *reinterpret_cast<float4*>(Ks + j * kDh + c4) =
        *reinterpret_cast<const float4*>(base + (int64_t)j * 3 * kD + kD + head * kDh + c4);
    *reinterpret_cast<float4*>(Vs + j * kDh + c4) =
        *reinterpret_cast<const float4*>(base + (int64_t)j * 3 * kD + 2 * kD + head * kDh + c4);
  }
  __syncthreads();
  if (tid >= kS) return;

  float q[kDh], o[kDh];
  const float scale = 0.17677669529663688110f;
#pragma unroll
  for (int c4 = 0; c4 < kDh; c4 += 4) {
    const float4 v = *reinterpret_cast<const float4*>(base + (int64_t)tid * 3 * kD + head * kDh + c4);
    q[c4] = v.x * scale; q[c4 + 1] = v.y * scale; q[c4 + 2] = v.z * scale; q[c4 + 3] = v.w * scale;
  }
#pragma unroll
  for (int c = 0; c < kDh; ++c) o[c] = 0.f;
  float m = -INFINITY, l = 0.f;
  const uint32_t row_base = (uint32_t)(head * kS + tid) * kS;   // element index (head*S + q)*S + k
  float4 mk = make_float4(1.f, 1.f, 1.f, 1.f);
  for (int j = 0; j < kS; ++j) {
    float s = 0.f;
#pragma unroll
    for (int c4 = 0; c4 < kDh; c4 += 4) {
      const float4 k = *reinterpret_cast<const float4*>(Ks + j * kDh + c4);
      s = fmaf(q[c4], k.x, s); s = fmaf(q[c4 + 1], k.y, s); s = fmaf(q[c4 + 2], k.z, s); s = fmaf(q[c4 + 3], k.w, s);
    }
    const float mn = fmaxf(m, s);
    const float corr = expf(m - mn);
    float p = expf(s - mn);
    l = fmaf(l, corr, p);
    if (drop.thresh != 0u) {
      const uint32_t e = row_base + j;
      if (j == 0 || (e & 3) == 0) mk = drop.mult4(e >> 2, (uint32_t)seq, layer_site);
      const uint32_t w = e & 3;
      p *= w == 0 ? mk.x : w == 1 ? mk.y : w == 2 ? mk.z : mk.w;
    }
#pragma unroll
    for (int c4 = 0; c4 < kDh; c4 += 4) {
      const float4 v = *reinterpret_cast<const float4*>(Vs + j * kDh + c4);
      o[c4] = fmaf(o[c4], corr, p * v.x); o[c4 + 1] = fmaf(o[c4 + 1], corr, p * v.y);
      o[c4 + 2] = fmaf(o[c4 + 2], corr, p * v.z); o[c4 + 3] = fmaf(o[c4 + 3], corr, p * v.w);
    }
    m = mn;
  }
  const float inv = 1.0f / l;
  float* op = out + (seq * kS + tid) * kD + head * kDh;
#pragma unroll
  for (int c4 = 0; c4 < kDh; c4 += 4)
    *reinterpret_cast<float4*>(op + c4) = make_float4(o[c4] * inv, o[c4 + 1] * inv, o[c4 + 2] * inv, o[c4 + 3] * inv);
  lse[(seq * kH + head) * kS + tid] = m + logf(l);
}

// the header record (passed by value, so the call stays asynchronous) and the inputs the backward needs again:
// real-valued pilots per sequence and the adapter conditions per sample
__global__ void k_save_inputs(TrainHeader hdr, TrainHeader* __restrict__ hdr_out, const float2* __restrict__ pilots,
                              const float* __restrict__ snr, const float* __restrict__ ds, const float* __restrict__ dop,
                              float* __restrict__ xs, float* __restrict__ cond, int64_t batch) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *hdr_out = hdr;
  if (i < batch * kPilots) {
    const float2 v = pilots[i];
    const int64_t b = i / kPilots;
    const int k = (int)(i - b * kPilots);
    xs[(2 * b) * kPilots + k] = v.x;
    xs[(2 * b + 1) * kPilots + k] = v.y;
  }
  if (snr && i < batch) {
    cond[3 * i] = snr[i];
    cond[3 * i + 1] = ds[i];
    cond[3 * i + 2] = dop[i];
  }
}

}  // namespace

TrainWs train_layout(void* base, int64_t batch, int layers) {
  const size_t nseq = 2 * (size_t)batch, M = nseq * kS;
  TrainWs w{};
  char* b = static_cast<char*>(base);
  size_t off = 256;   // header record
  auto take = [&](size_t floats) {
    float* p = b ? reinterpret_cast<float*>(b + off) : nullptr;
    off += align64(floats) * sizeof(float);
    return p;
  };
  w.hdr = reinterpret_cast<TrainHeader*>(b);
  w.xs = take(nseq * kPilots);
  w.cond = take((size_t)batch * 3);
  w.enh = take(nseq * kPix);
  w.L.resize(layers);
  for (auto& l : w.L) {
    l.x = take(M * kD); l.qkv = take(M * 3 * kD); l.o = take(M * kD); l.lse = take(M * kH);
    l.s1 = take(M * kD); l.y1 = take(M * kD); l.u = take(M * kFF); l.s2 = take(M * kD);
  }
  w.xout = take(M * kD);
  w.abuf = take(M * kFF);
  w.dh = take(M * kD); w.dres = take(M * kD); w.dproj = take(M * kD); w.tmp = take(M * kD);
  w.dbig = take(M * kFF); w.dqkv = take(M * 3 * kD);
  w.conv_in = take(nseq * kPix); w.conv_a1 = take(nseq * 8 * kPix); w.conv_a2 = take(nseq * 32 * kPix);
  w.conv_a3 = take(nseq * 8 * kPix);
  w.g1 = take(nseq * kPix); w.g8a = take(nseq * 8 * kPix); w.g32 = take(nseq * 32 * kPix); w.g8b = take(nseq * 8 * kPix);
  w.gin = take(nseq * kPix);
  w.denh = take(nseq * kPix); w.tok = take(M * 12); w.dtok = take(M * 12); w.dl2 = take(M * kPatchLen);
  w.mlp = take(nseq * 3 * (2 * kS + 4 * kMaxAdaHidden + 1));
  w.part = take((size_t)kMaxChunks * 3 * kD * kD);
  w.bytes = off;
  return w;
}

GradLayout grad_layout(const TrainModel& m) {
  GradLayout g{};
  size_t o = 0;
  auto at = [&](size_t n) { const size_t r = o; o += n; return r; };
  g.up_w = at((size_t)kPix * kPilots); g.up_b = at(kPix);
  static const int cw[4] = {72, 2304, 2304, 72}, cb[4] = {8, 32, 8, 1};
  for (int s = 0; s < 2; ++s)
    for (int i = 0; i < 4; ++i) { g.conv[s][2 * i] = at(cw[i]); g.conv[s][2 * i + 1] = at(cb[i]); }
  if (m.adaptive)
    for (int k = 0; k < 3; ++k) {
      g.mlp[k][0] = at(m.h1); g.mlp[k][1] = at(m.h1);
      g.mlp[k][2] = at((size_t)m.h2 * m.h1); g.mlp[k][3] = at(m.h2);
      g.mlp[k][4] = at((size_t)2 * kS * m.h2); g.mlp[k][5] = at(2 * kS);
    }
  const int in_dim = kPatchLen + (m.adaptive ? kAda : 0);
  g.l1_w = at((size_t)kD * in_dim); g.l1_b = at(kD);
  g.pos = at((size_t)m.max_seq_len * kD);
  g.l2_w = at((size_t)kPatchLen * kD); g.l2_b = at(kPatchLen);
  static const size_t lsz[12] = {3 * kD * kD, 3 * kD, kD * kD, kD, kFF * kD, kFF, kD * kFF, kD, kD, kD, kD, kD};
  for (int l = 0; l < m.num_layers; ++l)
    for (int i = 0; i < 12; ++i) g.layer.push_back(at(lsz[i]));
  g.total = o;
  return g;
}

bool train_forward(const TrainModel& m, const TrainHeader& hdr, const float2* pilots, const float* snr, const float* ds, const float* dop,
                   float2* out, int64_t batch, const DropCfg& drop, const TrainWs& ws, cudaStream_t st) {
  const int64_t nseq = 2 * batch, M = nseq * kS;
  const size_t smem = 2 * kS * kDh * sizeof(float);
  if (cudaFuncSetAttribute(attn_train_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("attn_train: cannot opt in to %zu bytes of shared memory", smem);
    return false;
  }
  k_save_inputs<<<(unsigned)((batch * kPilots + 255) / 256), 256, 0, st>>>(hdr, ws.hdr, pilots, m.adaptive ? snr : nullptr,
                                                                          ds, dop, ws.xs, ws.cond, batch);
  count_launch();
  if (!check_launch("k_save_inputs")) return false;
  if (!launch_frontend(*m.front, pilots, snr, ds, dop, ws.enh, ws.L[0].x, nullptr, batch, st)) return false;
  for (int l = 0; l < m.num_layers; ++l) {
    const LayerPackF32& P = m.layers[l];
    const TrainLayerBufs& B = ws.L[l];
    float* xnext = l + 1 < m.num_layers ? ws.L[l + 1].x : ws.xout;
    const uint32_t ls = (uint32_t)l << 8;
    if (!launch_gemm_f32(kEpiBias, B.x, P.in_w, P.in_b, B.qkv, M, 3 * kD, kD, 0, nullptr, nullptr, nullptr, st)) return false;
    attn_train_kernel<<<(unsigned)(nseq * kH), kAttnThreads, smem, st>>>(B.qkv, B.o, B.lse, drop, ls | 0u);
    count_launch();
    if (!check_launch("attn_train_kernel")) return false;
    if (!launch_gemm_f32_train(kEpiTrainResLn, B.o, P.out_w, P.out_b, B.y1, M, kD, kD, 0, B.x, P.n1_w, P.n1_b,
                               TrainEpi{B.s1, drop, ls | 1u}, st)) return false;
    if (!launch_gemm_f32_train(kEpiTrainAct, B.y1, P.l1_w, P.l1_b, ws.abuf, M, kFF, kD, m.activation, nullptr, nullptr,
                               nullptr, TrainEpi{B.u, drop, ls | 2u}, st)) return false;
    if (!launch_gemm_f32_train(kEpiTrainResLn, ws.abuf, P.l2_w, P.l2_b, xnext, M, kD, kFF, 0, B.y1, P.n2_w, P.n2_b,
                               TrainEpi{B.s2, drop, ls | 3u}, st)) return false;
  }
  return launch_head(*m.head, ws.xout, ws.enh, out, batch, st);
}

}  // namespace aft
