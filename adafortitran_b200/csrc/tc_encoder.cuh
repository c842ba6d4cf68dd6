// bf16 tcgen05 encoder path (AFT_BF16): declarations used by aft_api.cu.
#pragma once

#include <vector>

#include "aft_internal.cuh"

namespace aft {

// bf16 operand images of the encoder weights + fp32 epilogue vectors, one entry per layer
struct TcLayer {
  const __nv_bfloat16* w_in;    // in_proj  image: N=384 rows, K=128  (2 chunks x 384 rows x 128 B), q rows pre-scaled
  const __nv_bfloat16* w_out;   // out_proj image: N=128, K=128
  const __nv_bfloat16* w_l1;    // linear1  image: N=256, K=128
  const __nv_bfloat16* w_l2;    // linear2  image: N=128, K=256 (4 chunks)
  const float* b_in;            // [384], q part pre-scaled
  const float *b_out, *b_l1, *b_l2, *n1_w, *n1_b, *n2_w, *n2_b;
};

struct TcWeights {
  void* arena = nullptr;
  size_t arena_bytes = 0;
  int num_layers = 0;
  TcLayer* layers_dev = nullptr;        // device copy of the table
  std::vector<TcLayer> layers;          // host copy
  void* conv_front = nullptr;           // tensor-core packs of the two ConvEnhancers (conv_tc.cuh), inside the arena
  void* conv_head = nullptr;
};

bool tc_weights_alloc(TcWeights& w, int num_layers);
void tc_weights_free(TcWeights& w);
bool tc_weights_pack(TcWeights& w, const std::vector<LayerPackF32>& src, const ConvPack& enh, const ConvPack& refine, cudaStream_t st);
size_t tc_workspace_bytes(int64_t chunk_samples);
struct TcProfileHook {
  void (*mark)(void* ctx, cudaStream_t st);   // nullptr when profiling is off
  void* ctx;
};
bool tc_forward_chunk(const TcWeights& w, const FrontPack& front, const HeadPack& head, int activation, int sm_count,
                      const float2* pilots, const float* snr, const float* ds, const float* dop, const OutDst& out,
                      int64_t nsamples, void* workspace, cudaStream_t st, TcProfileHook hook);
bool tc_selftest(int which, double* max_err, cudaStream_t st);

// tc_long.cu : the encoder for any sequence length (activations in global memory as per-row-tile operand images,
// streaming attention).  h_in / h_out: fp32 [nseq * S][128] rows (may alias); workspace of tc_long_workspace_bytes().
size_t tc_long_workspace_bytes(int64_t nseq, int S);
bool tc_long_encoder(const TcWeights& w, int activation, int sm_count, const float* h_in, float* h_out, int64_t nseq, int S,
                     void* workspace, cudaStream_t st);

}  // namespace aft
