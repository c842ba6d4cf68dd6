// Internal declarations shared by the translation units of libaft_b200.so.
// Nothing here is part of the ABI (that is include/aft.h).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/aft.h"

namespace aft {

// ---------------------------------------------------------------------------------------------
// Compile-time shape of the hot path (reference default config; SURVEY.md §8).  aft_create()
// rejects every other shape with AFT_ERR_UNSUPPORTED -- there is no generic / fallback path.
// ---------------------------------------------------------------------------------------------
constexpr int kGridH = 120;                 // subcarriers
constexpr int kGridW = 14;                  // OFDM symbols
constexpr int kPix = kGridH * kGridW;       // 1680
constexpr int kPilots = 24;                 // 12 x 2
constexpr int kPatchH = 3, kPatchW = 2, kPatchLen = 6;
constexpr int kTokW = kGridW / kPatchW;     // 7 patches per row of patches
constexpr int kS = (kGridH / kPatchH) * kTokW;  // 280 tokens
constexpr int kD = 128;                     // model dim
constexpr int kH = 4;                       // heads
constexpr int kDh = 32;                     // head dim
constexpr int kFF = 256;                    // feed-forward dim
constexpr int kAda = 6;                     // adaptive features per token
constexpr int kMaxAdaHidden = 64;           // bound on adapt_h1 / adapt_h2
constexpr int kMaxLayers = 32;

// padded conv planes: (120+2) x (14+2), zero border
constexpr int kPW = kGridW + 2;             // 16
constexpr int kPH = kGridH + 2;             // 122
constexpr int kPlane = kPW * kPH;           // 1952

// ---------------------------------------------------------------------------------------------
// Packed parameters (device).  fp32 re-layouts used by the SIMT kernels; bf16 operand images used
// by the tcgen05 kernels are declared in tc_common.cuh.
// ---------------------------------------------------------------------------------------------
struct ConvPack {          // one ConvEnhancer; weights tap-major, cout fastest
  const float* w0;         // [9][8]          (cin = 1)
  const float* w1;         // [9][8][32]
  const float* w2;         // [9][32][8]
  const float* w3;         // [9][8]          (cout = 1)
  const float* b0;         // [8]
  const float* b1;         // [32]
  const float* b2;         // [8]
  const float* b3;         // [1]
};

struct MlpPack {           // one adapter encoder
  const float* w0;         // [h1]
  const float* b0;         // [h1]
  const float* w1;         // [h2][h1]
  const float* b1;         // [h2]
  const float* w2t;        // [h2][560]  (transposed: coalesced over outputs)
  const float* b2;         // [560]
};

struct LayerPackF32 {      // torch layouts, owned copies
  const float *in_w, *in_b, *out_w, *out_b, *l1_w, *l1_b, *l2_w, *l2_b, *n1_w, *n1_b, *n2_w, *n2_b;
};

struct FrontPack {
  const float* up_wt;      // [24][1680]
  const float* up_b;       // [1680]
  ConvPack enh;
  MlpPack mlp[3];          // snr, ds, dop
  int h1, h2;
  const float* l1_wt;      // [in_dim][128]  (in_dim = 6 or 12)
  const float* posb;       // [280][128] = pos[t] + linear_1.bias
  int in_dim;
  int adaptive;
};

struct HeadPack {
  const float* l2_w;       // [6][128]
  const float* l2_b;       // [6]
  ConvPack refine;
};

// Where the head stores the estimates of a chunk: up to 9 destinations (the caller's `out` and, for the fused
// all-gather of the multi-GPU evaluation path, this rank's row range inside every peer's gather buffer -- peer device
// memory mapped into this process, written with plain 16-byte stores over NVLink).  ptr[d] addresses sample 0 of the chunk.
struct OutDst {
  float2* ptr[9];
  int n;
};

// ---------------------------------------------------------------------------------------------
// launch bookkeeping / error plumbing (aft_api.cu)
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
bool check_launch(const char* what);   // cudaGetLastError() -> set_error; true when OK

// ---------------------------------------------------------------------------------------------
// kernels launchers (each returns false after set_error on failure)
// ---------------------------------------------------------------------------------------------
// frontend.cu : pilots -> upsample -> ConvEnhancer -> patchify (+adapter) -> linear_1 + pos
//   enh  : [nseq][1680] fp32 (kept for the residual in the head)
//   h    : [nseq][280][128] fp32 residual stream
//   hb   : optional bf16 operand image of h (tc_common.cuh layout), may be nullptr
bool launch_frontend(const FrontPack& p, const float2* pilots, const float* snr, const float* ds, const float* dop,
                     float* enh, float* h, __nv_bfloat16* hb, int64_t nsamples, cudaStream_t st);

// head.cu : linear_2 -> fold -> + enh -> ConvEnhancer -> interleaved complex store
bool launch_head(const HeadPack& p, const float* h, const float* enh, float2* out, int64_t nsamples, cudaStream_t st);

// conv_tc.cu : the same two stages for the AFT_BF16 path, ConvEnhancer on the tensor cores (persistent CTAs)
size_t conv_tc_pack_bytes();
void conv_tc_dump_timeline();
bool conv_tc_pack(const ConvPack& src, void* dst, cudaStream_t st);
//   zbuf : [nsamples][3][2 S] fp32 scratch for the adaptive features (written by adapter_kernel; unused for FortiTran)
bool launch_frontend_tc(const FrontPack& p, const void* pack, const float2* pilots, const float* snr, const float* ds,
                        const float* dop, float* zbuf, float* enh, __nv_bfloat16* hb, int64_t nsamples, int sm_count, cudaStream_t st);
bool launch_head_tc(const HeadPack& p, const void* pack, const void* himg, const float* enh, const OutDst& out, int64_t nsamples,
                    int sm_count, cudaStream_t st);

// gemm_f32.cu : C[M,N] = A[M,K] * W[N,K]^T + bias, fp32 FMA
enum GemmEpi { kEpiBias = 0, kEpiBiasAct = 1, kEpiBiasResLn = 2 };
bool launch_gemm_f32(int epi, const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K,
                     int act, const float* residual, const float* gamma, const float* beta, cudaStream_t st);

// the same product for arbitrary N, K (bias epilogue, guarded edges)
bool launch_gemm_f32_any(const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K, cudaStream_t st);

// attn_f32.cu : per (sequence, head) softmax(q k^T / sqrt(dh)) v, fp32
bool launch_attn_f32(const float* qkv, float* out, int64_t nseq, cudaStream_t st);

// aux.cu : "next" rows N2 / N3 -- pilot extraction from the sparse LS grid, LinearEstimator
bool launch_extract_pilots(const float2* grid, float2* pilots, int32_t* counts, int64_t batch, int cells, int expected, cudaStream_t st);
bool launch_linear(const float* w, const float* bias, const float* x, float* y, int64_t batch, int in_dim, int out_dim, cudaStream_t st);
size_t linear_backward_workspace_bytes(int64_t batch, int in_dim, int out_dim);   // >= 256
bool launch_linear_backward(const float* w, const float* x, const float* gy, float* grad_w, float* grad_b, float* grad_x,
                            int64_t batch, int in_dim, int out_dim, void* workspace, cudaStream_t st);

// synth.cu : synthetic channels and noisy pilots (include/aft.h, "Synthetic channels"); arguments checked by the caller
bool launch_synthetic_channels(const AftConfig& cfg, uint64_t seed, int64_t sample0, int64_t batch, float* snr, float* ds,
                               float* dop, bool draw_conditions, float2* pilots, float2* truth, cudaStream_t st);

// generic_f32.cu : AFT_FP32 path for non-default grids (activations in global memory, runtime extents)
size_t generic_front_scratch_floats(int64_t nsamples, int P, int pix, int S);
size_t generic_head_scratch_floats(int64_t nsamples, int pix);
bool launch_generic_frontend(const FrontPack& p, const float2* pilots, const float* snr, const float* ds, const float* dop, float* enh,
                             float* h, float* scratch, int64_t nsamples, int H, int W, int P, int ph, int pw, cudaStream_t st);
bool launch_generic_attention(const float* qkv, float* out, int64_t nseq, int S, cudaStream_t st);
bool launch_generic_head(const HeadPack& p, const float* h, const float* enh, float2* out, float* scratch, int64_t nsamples, int H, int W,
                         int ph, int pw, cudaStream_t st);

// reduce.cu
bool launch_error_sums(const float2* est, const float2* truth, int64_t count, double* sums, cudaStream_t st);
// copies src[count] (complex64) to every destination of `dst` (peer scatter of the non-fused paths), rows at any offset
bool launch_scatter_rows(const float2* src, int64_t count, const OutDst& dst, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

}  // namespace aft
