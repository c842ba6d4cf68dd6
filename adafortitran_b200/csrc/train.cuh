// Training path (AFT_FP32, reference default geometry): dropout rule, workspace layout and the entry points of
// train_fwd.cu / train_bwd.cu.  Nothing here is part of the ABI (that is include/aft.h).
#pragma once

#include <vector>

#include "aft_internal.cuh"

namespace aft {

// ---------------------------------------------------------------------------------------------
// Dropout rule (include/aft.h, "Dropout"): Philox4x32-10, key (seed_lo, seed_hi), counter
// (i >> 2, seq0 + seq, (layer << 8) | site, 0) with seq the call-local sequence and seq0 = 2 * sample0 the first global
// sequence of the call; element i uses output word i & 3 and is kept iff that word >= thresh, thresh = floor(p * 2^32).
// Kept values are scaled by 1 / (1 - p).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

struct DropCfg {
  uint32_t thresh;      // floor(p * 2^32); 0 = no dropout
  float scale;          // 1 / (1 - p)
  uint32_t seed_lo, seed_hi;
  uint32_t seq0;        // 2 * sample0: global sequence index of the call's first sequence
  __device__ __forceinline__ uint4 words(uint32_t i4, uint32_t seq, uint32_t layer_site) const {
    return philox4x32_10(make_uint4(i4, seq0 + seq, layer_site, 0u), seed_lo, seed_hi);
  }
  // multipliers (0 or scale) of the four elements 4*i4 .. 4*i4+3
  __device__ __forceinline__ float4 mult4(uint32_t i4, uint32_t seq, uint32_t layer_site) const {
    const uint4 w = words(i4, seq, layer_site);
    return make_float4(w.x >= thresh ? scale : 0.f, w.y >= thresh ? scale : 0.f, w.z >= thresh ? scale : 0.f,
                       w.w >= thresh ? scale : 0.f);
  }
  __device__ __forceinline__ float mult(uint32_t i, uint32_t seq, uint32_t layer_site) const {
    const uint4 w = words(i >> 2, seq, layer_site);
    const uint32_t v = (i & 3) == 0 ? w.x : (i & 3) == 1 ? w.y : (i & 3) == 2 ? w.z : w.w;
    return v >= thresh ? scale : 0.f;
  }
};

// Extra state of the training epilogues of gemm_f32.cu
struct TrainEpi {
  float* aux;           // kEpiTrainResLn: pre-LayerNorm sum; kEpiTrainAct: pre-activation
  DropCfg drop;
  uint32_t layer_site;  // (layer << 8) | site
};

// C = LN(drop(A W^T + b) + residual), aux = the pre-LN sum      (sites 1 and 3)
// C = drop(act(A W^T + b)),            aux = the pre-activation  (site 2)
enum TrainEpiKind { kEpiTrainResLn = 3, kEpiTrainAct = 4 };
bool launch_gemm_f32_train(int epi, const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K,
                           int act, const float* residual, const float* gamma, const float* beta, const TrainEpi& te,
                           cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// Workspace: a 256-byte header record, the saved activations, then the backward scratch.
// ---------------------------------------------------------------------------------------------
struct TrainHeader {
  uint64_t magic;
  int64_t batch;
  int32_t layers, adaptive;
  float dropout;
  uint32_t thresh;
  uint64_t seed;
  int64_t sample0;      // global index of the forward's first sample (aft_forward_train_offset)
};
constexpr uint64_t kTrainMagic = 0x31574b5254544641ull;   // "AFTTRKW1"
constexpr int kMaxChunks = 128;                          // partial tiles of the deterministic weight-gradient sums

struct TrainLayerBufs {
  float *x, *qkv, *o, *lse, *s1, *y1, *u, *s2;   // x = layer input; lse [nseq][4][280]
};

struct TrainWs {
  TrainHeader* hdr;
  // saved by the forward
  float* xs;                         // [nseq][24] real-valued pilots
  float* cond;                       // [batch][3] snr, delay spread, doppler (adaptive only)
  float* enh;                        // [nseq][1680]
  std::vector<TrainLayerBufs> L;     // per layer
  float* xout;                       // [M][128] output of the last layer
  // scratch
  float *abuf, *dh, *dres, *dproj, *tmp, *dbig, *dqkv;
  float *conv_in, *conv_a1, *conv_a2, *conv_a3;          // recomputed ConvEnhancer activations [nseq][c][1680]
  float *g1, *g8a, *g32, *g8b, *gin;                     // their gradients
  float *denh, *tok, *dtok, *dl2, *mlp;                  // front / head scratch
  float* part;                                           // [kMaxChunks][49152] partial sums
  size_t bytes;
};

// lays the workspace out from `base` (nullptr: only measures)
TrainWs train_layout(void* base, int64_t batch, int layers);

struct TrainModel {   // what the training kernels read from the handle
  const FrontPack* front;
  const HeadPack* head;
  const LayerPackF32* layers;
  int num_layers, activation, adaptive, h1, h2, max_seq_len;
};

// gradient offsets (floats) in the flat buffer, in the order of include/aft.h
struct GradLayout {
  size_t up_w, up_b, conv[2][8], mlp[3][6], l1_w, l1_b, pos, l2_w, l2_b;
  std::vector<size_t> layer;   // 12 entries per layer
  size_t total;
};
GradLayout grad_layout(const TrainModel& m);

// writes `hdr` to the workspace's header record, then runs the forward
bool train_forward(const TrainModel& m, const TrainHeader& hdr, const float2* pilots, const float* snr, const float* ds, const float* dop,
                   float2* out, int64_t batch, const DropCfg& drop, const TrainWs& ws, cudaStream_t st);
bool train_backward(const TrainModel& m, const float2* grad_out, int64_t batch, const DropCfg& drop, const TrainWs& ws, float* grads,
                    cudaStream_t st);

}  // namespace aft
