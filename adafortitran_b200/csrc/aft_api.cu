// C-ABI of libaft_b200.so (include/aft.h): handle lifetime, weight packing, forward orchestration.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "aft_internal.cuh"
#include "tc_encoder.cuh"
#include "train.cuh"

namespace aft {

// ---------------------------------------------------------------------------------------------
// error / launch bookkeeping
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_error;
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

bool check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return false;
  }
  return true;
}

#define AFT_CUDA(call)                                                                    \
  do {                                                                                    \
    const cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess) {                                                             \
      set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return AFT_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

// ---------------------------------------------------------------------------------------------
// packing kernels (run once per aft_load_weights)
// ---------------------------------------------------------------------------------------------
__global__ void k_copy(const float* src, float* dst, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}
// src [R][C] -> dst [C][R]
__global__ void k_transpose(const float* src, float* dst, int R, int C) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < R * C) {
    const int r = i / C, c = i - r * C;
    dst[c * R + r] = src[i];
  }
}
// conv weight [cout][cin][3][3] -> [tap][cin][cout]
__global__ void k_conv_repack(const float* src, float* dst, int cout, int cin) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cout * cin * 9) {
    const int co = i / (cin * 9), rem = i - co * cin * 9;
    const int ci = rem / 9, t = rem - ci * 9;
    dst[(t * cin + ci) * cout + co] = src[i];
  }
}
// posb[t][c] = pos[t][c] + bias[c]
__global__ void k_posb(const float* pos, const float* bias, float* dst, int n, int d) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = pos[i] + bias[i % d];
}

static inline unsigned blocks_for(int n) { return (unsigned)((n + 255) / 256); }

}  // namespace aft

using namespace aft;

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct AftHandle {
  AftConfig cfg;
  // Shape mode.  false: the reference default grid, served by the specialised kernels (both precisions).  true: any
  // other grid / pilot / patch geometry, served by the shape-generic AFT_FP32 kernels (generic_f32.cu); AFT_BF16 is
  // rejected for such a handle.
  bool generic = false;
  int H = kGridH, W = kGridW, P = kPilots, ph = kPatchH, pw = kPatchW, S = kS, pix = kPix, patch_len = kPatchLen;
  int device = -1;
  int sm_count = 0;
  bool loaded = false;
  float* arena = nullptr;       // packed fp32 parameters
  size_t arena_floats = 0;
  FrontPack front{};
  HeadPack head{};
  std::vector<LayerPackF32> layers;
  TcWeights tc{};               // bf16 operand images (tc_encoder.cuh)
  // stage profile (aft_profile_enable / aft_profile_read)
  bool profile = false;
  std::vector<cudaEvent_t> prof_events;   // groups of 4: start, after frontend, after encoder, after head
  size_t prof_used = 0;
  int64_t prof_launches[3] = {0, 0, 0};
  // aft_forward_host resources (lazy)
  struct HostLane {
    cudaStream_t stream = nullptr;
    void* d_in = nullptr;       // pilots | snr | ds | dop
    void* d_out = nullptr;
    void* ws = nullptr;
    size_t ws_bytes = 0;
    int64_t cap = 0;
  } lanes[2];
};

namespace {

constexpr int64_t kChunkF32 = 1024;    // samples per internal chunk, fp32 path (~1.5 GB of scratch)
constexpr int64_t kChunkBf16 = 8192;   // bf16 path
constexpr int64_t kHostChunk = 2048;   // samples per pipelined host chunk

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

size_t ws_bytes_f32(int64_t bc) {
  const size_t nseq = 2 * (size_t)bc;
  size_t f = 0;
  f += align_up(nseq * kPix, 64);            // enh
  f += align_up(nseq * kS * kD, 64);         // h
  f += align_up(nseq * kS * 3 * kD, 64);     // qkv (ffn hidden aliases it)
  f += align_up(nseq * kS * kD, 64);         // attention output
  return f * sizeof(float);
}

int validate(const AftConfig& c, bool* generic) {
  auto bad = [](const char* what) {
    set_error("unsupported configuration: %s (supported: model_dim 128, 4 heads, ff 256, adapter [h1<=64, h2<=64, 2*tokens], "
              "patch sizes dividing the grid; the tensor-core AFT_BF16 path additionally needs the reference default grid "
              "120x14, pilots 12x2, patch 3x2)", what);
    return AFT_ERR_UNSUPPORTED;
  };
  if (c.model_dim != kD || c.num_head != kH || c.ff_dim != kFF) return bad("model_dim / num_head / ff_dim");
  if (c.num_layers < 1 || c.num_layers > kMaxLayers) return bad("num_layers");
  if (c.activation != AFT_ACT_RELU && c.activation != AFT_ACT_GELU) return bad("activation");
  if (c.num_scs < 1 || c.num_symbols < 1 || c.pilot_scs < 1 || c.pilot_symbols < 1) return bad("grid extents");
  if (c.patch_scs < 1 || c.patch_symbols < 1 || c.num_scs % c.patch_scs != 0 || c.num_symbols % c.patch_symbols != 0)
    return bad("patch_size must divide the ofdm grid");
  if (c.patch_scs * c.patch_symbols > 64) return bad("patch_size (more than 64 elements)");
  if ((int64_t)c.pilot_scs * c.pilot_symbols > 4096) return bad("more than 4096 pilots");
  if ((int64_t)c.num_scs * c.num_symbols > (1 << 22)) return bad("ofdm grid (more than 4M points)");
  const int S = (c.num_scs / c.patch_scs) * (c.num_symbols / c.patch_symbols);
  if (c.max_seq_len < S) return bad("max_seq_len < sequence length");
  if (c.adaptive) {
    if (c.adapt_h1 < 1 || c.adapt_h1 > kMaxAdaHidden || c.adapt_h2 < 1 || c.adapt_h2 > kMaxAdaHidden) return bad("adapter hidden sizes");
    if (c.adapt_h3 != 2 * S) return bad("channel_adaptivity_hidden_sizes[2] must be 2*num_patches");
    if (c.adaptive_token_length != kAda) return bad("adaptive_token_length");
  }
  *generic = !(c.num_scs == kGridH && c.num_symbols == kGridW && c.pilot_scs == 12 && c.pilot_symbols == 2 &&
               c.patch_scs == kPatchH && c.patch_symbols == kPatchW);
  return AFT_OK;
}

struct ArenaCursor {
  float* base;
  size_t off = 0;
  float* take(size_t n) {
    float* p = base ? base + off : nullptr;
    off += align_up(n, 64);
    return p;
  }
};

// lays the packed parameters out in the arena; with base == nullptr only measures
size_t layout_arena(AftHandle* h, float* base) {
  const AftConfig& c = h->cfg;
  ArenaCursor a{base};
  auto conv = [&](ConvPack& p) {
    p.w0 = a.take(72); p.w1 = a.take(2304); p.w2 = a.take(2304); p.w3 = a.take(72);
    p.b0 = a.take(8); p.b1 = a.take(32); p.b2 = a.take(8); p.b3 = a.take(8);
  };
  const int in_dim = h->patch_len + (c.adaptive ? kAda : 0);
  h->front.up_wt = a.take((size_t)h->P * h->pix);
  h->front.up_b = a.take(h->pix);
  conv(h->front.enh);
  for (int m = 0; m < 3; ++m) {
    MlpPack& mp = h->front.mlp[m];
    if (c.adaptive) {
      mp.w0 = a.take(c.adapt_h1); mp.b0 = a.take(c.adapt_h1);
      mp.w1 = a.take((size_t)c.adapt_h2 * c.adapt_h1); mp.b1 = a.take(c.adapt_h2);
      mp.w2t = a.take((size_t)c.adapt_h2 * 2 * h->S); mp.b2 = a.take(2 * h->S);
    } else {
      mp = MlpPack{};
    }
  }
  h->front.h1 = c.adapt_h1; h->front.h2 = c.adapt_h2;
  h->front.l1_wt = a.take((size_t)in_dim * kD);
  h->front.posb = a.take((size_t)h->S * kD);
  h->front.in_dim = in_dim;
  h->front.adaptive = c.adaptive;
  h->head.l2_w = a.take((size_t)h->patch_len * kD);
  h->head.l2_b = a.take(64);
  conv(h->head.refine);
  h->layers.resize(c.num_layers);
  for (auto& L : h->layers) {
    L.in_w = a.take(3 * kD * kD); L.in_b = a.take(3 * kD);
    L.out_w = a.take(kD * kD); L.out_b = a.take(kD);
    L.l1_w = a.take(kFF * kD); L.l1_b = a.take(kFF);
    L.l2_w = a.take(kD * kFF); L.l2_b = a.take(kD);
    L.n1_w = a.take(kD); L.n1_b = a.take(kD); L.n2_w = a.take(kD); L.n2_b = a.take(kD);
  }
  return a.off;
}

bool pack_conv(const AftConvStack& src, const ConvPack& dst, cudaStream_t st) {
  for (int i = 0; i < 4; ++i)
    if (!src.w[i] || !src.b[i]) { set_error("conv stack: NULL parameter pointer"); return false; }
  k_conv_repack<<<1, 256, 0, st>>>(src.w[0], const_cast<float*>(dst.w0), 8, 1);
  k_conv_repack<<<blocks_for(2304), 256, 0, st>>>(src.w[1], const_cast<float*>(dst.w1), 32, 8);
  k_conv_repack<<<blocks_for(2304), 256, 0, st>>>(src.w[2], const_cast<float*>(dst.w2), 8, 32);
  k_conv_repack<<<1, 256, 0, st>>>(src.w[3], const_cast<float*>(dst.w3), 1, 8);
  k_copy<<<1, 256, 0, st>>>(src.b[0], const_cast<float*>(dst.b0), 8);
  k_copy<<<1, 256, 0, st>>>(src.b[1], const_cast<float*>(dst.b1), 32);
  k_copy<<<1, 256, 0, st>>>(src.b[2], const_cast<float*>(dst.b2), 8);
  k_copy<<<1, 256, 0, st>>>(src.b[3], const_cast<float*>(dst.b3), 1);
  count_launch(8);
  return check_launch("pack_conv");
}

bool copy_to(const float* src, const float* dst, int n, cudaStream_t st, const char* name) {
  if (!src) { set_error("NULL parameter pointer: %s", name); return false; }
  k_copy<<<blocks_for(n), 256, 0, st>>>(src, const_cast<float*>(dst), n);
  count_launch();
  return check_launch(name);
}

// records the next profile event on `st` (no-op unless profiling is enabled)
void prof_mark(AftHandle* h, cudaStream_t st) {
  if (!h->profile) return;
  if (h->prof_used == h->prof_events.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    h->prof_events.push_back(e);
  }
  cudaEventRecord(h->prof_events[h->prof_used++], st);
}

void prof_mark_cb(void* ctx, cudaStream_t st) { prof_mark(static_cast<AftHandle*>(ctx), st); }

int forward_chunk_f32(AftHandle* h, const float2* pilots, const float* snr, const float* ds, const float* dop,
                      float2* out, int64_t bc, float* ws, cudaStream_t st) {
  const int64_t nseq = 2 * bc, M = nseq * kS;
  float* enh = ws;
  float* hbuf = enh + align_up((size_t)nseq * kPix, 64);
  float* qkv = hbuf + align_up((size_t)nseq * kS * kD, 64);
  float* att = qkv + align_up((size_t)nseq * kS * 3 * kD, 64);
  float* ffn = qkv;
  prof_mark(h, st);
  if (!launch_frontend(h->front, pilots, snr, ds, dop, enh, hbuf, nullptr, bc, st)) return AFT_ERR_CUDA;
  prof_mark(h, st);
  for (const LayerPackF32& L : h->layers) {
    if (!launch_gemm_f32(kEpiBias, hbuf, L.in_w, L.in_b, qkv, M, 3 * kD, kD, 0, nullptr, nullptr, nullptr, st)) return AFT_ERR_CUDA;
    if (!launch_attn_f32(qkv, att, nseq, st)) return AFT_ERR_CUDA;
    if (!launch_gemm_f32(kEpiBiasResLn, att, L.out_w, L.out_b, hbuf, M, kD, kD, 0, hbuf, L.n1_w, L.n1_b, st)) return AFT_ERR_CUDA;
    if (!launch_gemm_f32(kEpiBiasAct, hbuf, L.l1_w, L.l1_b, ffn, M, kFF, kD, h->cfg.activation, nullptr, nullptr, nullptr, st)) return AFT_ERR_CUDA;
    if (!launch_gemm_f32(kEpiBiasResLn, ffn, L.l2_w, L.l2_b, hbuf, M, kD, kFF, 0, hbuf, L.n2_w, L.n2_b, st)) return AFT_ERR_CUDA;
  }
  prof_mark(h, st);
  if (!launch_head(h->head, hbuf, enh, out, bc, st)) return AFT_ERR_CUDA;
  prof_mark(h, st);
  if (h->profile) { h->prof_launches[0] += 1; h->prof_launches[1] += 5 * (int64_t)h->layers.size(); h->prof_launches[2] += 1; }
  return AFT_OK;
}

// ---- shape-generic AFT_FP32 path (generic_f32.cu)
size_t generic_floats_per_chunk(const AftHandle* h, int64_t bc, int precision = AFT_FP32) {
  const size_t nseq = 2 * (size_t)bc, M = nseq * h->S;
  size_t f = 0;
  f += align_up(nseq * h->pix, 64);          // enh
  f += align_up(M * kD, 64);                 // h
  if (precision == AFT_BF16) {
    f += align_up(tc_long_workspace_bytes((int64_t)nseq, h->S) / sizeof(float) + 256, 64);   // operand images of tc_long.cu
  } else {
    f += align_up(M * 3 * kD, 64);           // qkv (ffn hidden aliases it)
    f += align_up(M * kD, 64);               // attention output
  }
  const size_t a = generic_front_scratch_floats(bc, h->P, h->pix, h->S), b = generic_head_scratch_floats(bc, h->pix);
  f += align_up(a > b ? a : b, 64);          // frontend / head scratch (conv planes)
  return f;
}
// samples per internal chunk: about 1 GB of scratch, at least one sample
int64_t generic_chunk(const AftHandle* h, int precision = AFT_FP32) {
  // about 1 GB of scratch (3 GB on the tensor-core path, whose kernels want more row tiles per launch), at least one sample
  const size_t per = generic_floats_per_chunk(h, 1, precision) * sizeof(float);
  int64_t bc = (int64_t)((size_t(precision == AFT_BF16 ? 3 : 1) << 30) / (per ? per : 1));
  if (bc < 1) bc = 1;
  if (bc > kChunkF32) bc = kChunkF32;
  if (2 * bc > 65535) bc = 32767;            // sequences are a grid dimension of the attention kernel
  return bc;
}

int forward_chunk_generic(AftHandle* h, const float2* pilots, const float* snr, const float* ds, const float* dop, float2* out,
                          int64_t bc, float* ws, cudaStream_t st, int precision) {
  const int64_t nseq = 2 * bc, M = nseq * h->S;
  float* enh = ws;
  float* hbuf = enh + align_up((size_t)nseq * h->pix, 64);
  if (precision == AFT_BF16) {
    // tensor-core encoder over row-tile operand images (tc_long.cu); frontend and head stay on the shape-generic fp32 kernels
    float* img = hbuf + align_up((size_t)M * kD, 64);
    float* scratch = img + align_up(tc_long_workspace_bytes(nseq, h->S) / sizeof(float) + 256, 64);
    void* img_aligned = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(img) + 1023) & ~uintptr_t(1023));
    prof_mark(h, st);
    if (!launch_generic_frontend(h->front, pilots, snr, ds, dop, enh, hbuf, scratch, bc, h->H, h->W, h->P, h->ph, h->pw, st)) return AFT_ERR_CUDA;
    prof_mark(h, st);
    if (!tc_long_encoder(h->tc, h->cfg.activation, h->sm_count, hbuf, hbuf, nseq, h->S, img_aligned, st)) return AFT_ERR_CUDA;
    prof_mark(h, st);
    if (!launch_generic_head(h->head, hbuf, enh, out, scratch, bc, h->H, h->W, h->ph, h->pw, st)) return AFT_ERR_CUDA;
    prof_mark(h, st);
    if (h->profile) { h->prof_launches[0] += 1; h->prof_launches[1] += 2 * (int64_t)h->layers.size() + 2; h->prof_launches[2] += 1; }
    return AFT_OK;
  }
  float* qkv = hbuf + align_up((size_t)M * kD, 64);
  float* att = qkv + align_up((size_t)M * 3 * kD, 64);
  float* scratch = att + align_up((size_t)M * kD, 64);
  float* ffn = qkv;
  prof_mark(h, st);
  if (!launch_generic_frontend(h->front, pilots, snr, ds, dop, enh, hbuf, scratch, bc, h->H, h->W, h->P, h->ph, h->pw, st)) return AFT_ERR_CUDA;
  prof_mark(h, st);
  for (const LayerPackF32& L : h->layers) {
    if (!launch_gemm_f32(kEpiBias, hbuf, L.in_w, L.in_b, qkv, M, 3 * kD, kD, 0, nullptr, nullptr, nullptr, st)) return AFT_ERR_CUDA;
    if (!launch_generic_attention(qkv, att, nseq, h->S, st)) return AFT_ERR_CUDA;
    if (!launch_gemm_f32(kEpiBiasResLn, att, L.out_w, L.out_b, hbuf, M, kD, kD, 0, hbuf, L.n1_w, L.n1_b, st)) return AFT_ERR_CUDA;
    if (!launch_gemm_f32(kEpiBiasAct, hbuf, L.l1_w, L.l1_b, ffn, M, kFF, kD, h->cfg.activation, nullptr, nullptr, nullptr, st)) return AFT_ERR_CUDA;
    if (!launch_gemm_f32(kEpiBiasResLn, ffn, L.l2_w, L.l2_b, hbuf, M, kD, kFF, 0, hbuf, L.n2_w, L.n2_b, st)) return AFT_ERR_CUDA;
  }
  prof_mark(h, st);
  if (!launch_generic_head(h->head, hbuf, enh, out, scratch, bc, h->H, h->W, h->ph, h->pw, st)) return AFT_ERR_CUDA;
  prof_mark(h, st);
  if (h->profile) { h->prof_launches[0] += 1; h->prof_launches[1] += 5 * (int64_t)h->layers.size(); h->prof_launches[2] += 1; }
  return AFT_OK;
}

int64_t chunk_for(const AftHandle* h, int precision) {
  if (h->generic) return generic_chunk(h, precision);
  return precision == AFT_BF16 ? kChunkBf16 : kChunkF32;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// exported entry points
// ---------------------------------------------------------------------------------------------
extern "C" {

int aft_abi_version(void) { return AFT_ABI_VERSION; }

const char* aft_last_error(void) { return g_error.c_str(); }

int64_t aft_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int aft_create(const AftConfig* cfg, AftHandle** out) {
  if (!cfg || !out) { set_error("aft_create: NULL argument"); return AFT_ERR_INVALID; }
  *out = nullptr;
  bool generic = false;
  const int v = validate(*cfg, &generic);
  if (v != AFT_OK) return v;
  int dev = -1;
  AFT_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  AFT_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_error("aft_create: device %d is sm_%d%d; this library contains sm_100a code only (no fallback path)", dev,
              prop.major, prop.minor);
    return AFT_ERR_CUDA;
  }
  AftHandle* h = new (std::nothrow) AftHandle();
  if (!h) { set_error("aft_create: out of host memory"); return AFT_ERR_INVALID; }
  h->cfg = *cfg;
  h->generic = generic;
  h->H = cfg->num_scs; h->W = cfg->num_symbols; h->P = cfg->pilot_scs * cfg->pilot_symbols;
  h->ph = cfg->patch_scs; h->pw = cfg->patch_symbols; h->patch_len = h->ph * h->pw;
  h->S = (h->H / h->ph) * (h->W / h->pw); h->pix = h->H * h->W;
  h->device = dev;
  h->sm_count = prop.multiProcessorCount;
  h->arena_floats = layout_arena(h, nullptr);
  cudaError_t e = cudaMalloc(&h->arena, h->arena_floats * sizeof(float));
  if (e != cudaSuccess) {
    set_error("aft_create: cudaMalloc(%zu) failed: %s", h->arena_floats * sizeof(float), cudaGetErrorString(e));
    delete h;
    return AFT_ERR_CUDA;
  }
  layout_arena(h, h->arena);
  if (!tc_weights_alloc(h->tc, cfg->num_layers)) {
    cudaFree(h->arena);
    delete h;
    return AFT_ERR_CUDA;
  }
  *out = h;
  return AFT_OK;
}

void aft_destroy(AftHandle* h) {
  if (!h) return;
  for (auto& ln : h->lanes) {
    if (ln.d_in) cudaFree(ln.d_in);
    if (ln.d_out) cudaFree(ln.d_out);
    if (ln.ws) cudaFree(ln.ws);
    if (ln.stream) cudaStreamDestroy(ln.stream);
  }
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  tc_weights_free(h->tc);
  if (h->arena) cudaFree(h->arena);
  delete h;
}

int aft_load_weights(AftHandle* h, const AftWeights* w, void* stream) {
  if (!h || !w) { set_error("aft_load_weights: NULL argument"); return AFT_ERR_INVALID; }
  if (w->num_layers != h->cfg.num_layers || !w->layers) {
    set_error("aft_load_weights: expected %d encoder layers, got %d", h->cfg.num_layers, w->num_layers);
    return AFT_ERR_INVALID;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const AftConfig& c = h->cfg;
  if (!w->upsampler_w || !w->upsampler_b || !w->linear_1_w || !w->linear_1_b || !w->pos_table || !w->linear_2_w || !w->linear_2_b) {
    set_error("aft_load_weights: NULL parameter pointer");
    return AFT_ERR_INVALID;
  }
  auto mut = [](const float* p) { return const_cast<float*>(p); };
  if (h->generic) {   // the generic linear kernel reads W [out][in] as it is
    if (cudaMemcpyAsync(mut(h->front.up_wt), w->upsampler_w, (size_t)h->pix * h->P * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
      set_error("aft_load_weights: copy of pilot_upsampler.weight failed");
      return AFT_ERR_CUDA;
    }
  } else {
    k_transpose<<<blocks_for(kPix * kPilots), 256, 0, st>>>(w->upsampler_w, mut(h->front.up_wt), kPix, kPilots);
    count_launch();
  }
  if (!copy_to(w->upsampler_b, h->front.up_b, h->pix, st, "pilot_upsampler.bias")) return AFT_ERR_CUDA;
  if (!pack_conv(w->initial_enhancer, h->front.enh, st)) return AFT_ERR_CUDA;
  if (!pack_conv(w->final_refiner, h->head.refine, st)) return AFT_ERR_CUDA;
  if (c.adaptive) {
    const AftMlp* src[3] = {&w->snr_encoder, &w->ds_encoder, &w->dop_encoder};
    for (int m = 0; m < 3; ++m) {
      const MlpPack& mp = h->front.mlp[m];
      for (int i = 0; i < 3; ++i)
        if (!src[m]->w[i] || !src[m]->b[i]) { set_error("aft_load_weights: NULL channel_adapter parameter"); return AFT_ERR_INVALID; }
      if (!copy_to(src[m]->w[0], mp.w0, c.adapt_h1, st, "adapter.0.weight")) return AFT_ERR_CUDA;
      if (!copy_to(src[m]->b[0], mp.b0, c.adapt_h1, st, "adapter.0.bias")) return AFT_ERR_CUDA;
      if (!copy_to(src[m]->w[1], mp.w1, c.adapt_h2 * c.adapt_h1, st, "adapter.2.weight")) return AFT_ERR_CUDA;
      if (!copy_to(src[m]->b[1], mp.b1, c.adapt_h2, st, "adapter.2.bias")) return AFT_ERR_CUDA;
      k_transpose<<<blocks_for(2 * h->S * c.adapt_h2), 256, 0, st>>>(src[m]->w[2], mut(mp.w2t), 2 * h->S, c.adapt_h2);
      count_launch();
      if (!copy_to(src[m]->b[2], mp.b2, 2 * h->S, st, "adapter.4.bias")) return AFT_ERR_CUDA;
    }
  }
  k_transpose<<<blocks_for(kD * h->front.in_dim), 256, 0, st>>>(w->linear_1_w, mut(h->front.l1_wt), kD, h->front.in_dim);
  k_posb<<<blocks_for(h->S * kD), 256, 0, st>>>(w->pos_table, w->linear_1_b, mut(h->front.posb), h->S * kD, kD);
  count_launch(2);
  if (!copy_to(w->linear_2_w, h->head.l2_w, h->patch_len * kD, st, "linear_2.weight")) return AFT_ERR_CUDA;
  if (!copy_to(w->linear_2_b, h->head.l2_b, h->patch_len, st, "linear_2.bias")) return AFT_ERR_CUDA;
  for (int l = 0; l < c.num_layers; ++l) {
    const AftEncoderLayer& s = w->layers[l];
    const LayerPackF32& d = h->layers[l];
    const struct { const float* s; const float* d; int n; const char* name; } items[] = {
        {s.in_proj_w, d.in_w, 3 * kD * kD, "in_proj_weight"}, {s.in_proj_b, d.in_b, 3 * kD, "in_proj_bias"},
        {s.out_proj_w, d.out_w, kD * kD, "out_proj.weight"}, {s.out_proj_b, d.out_b, kD, "out_proj.bias"},
        {s.lin1_w, d.l1_w, kFF * kD, "linear1.weight"}, {s.lin1_b, d.l1_b, kFF, "linear1.bias"},
        {s.lin2_w, d.l2_w, kD * kFF, "linear2.weight"}, {s.lin2_b, d.l2_b, kD, "linear2.bias"},
        {s.norm1_w, d.n1_w, kD, "norm1.weight"}, {s.norm1_b, d.n1_b, kD, "norm1.bias"},
        {s.norm2_w, d.n2_w, kD, "norm2.weight"}, {s.norm2_b, d.n2_b, kD, "norm2.bias"}};
    for (const auto& it : items)
      if (!copy_to(it.s, it.d, it.n, st, it.name)) return AFT_ERR_CUDA;
  }
  if (!tc_weights_pack(h->tc, h->layers, h->front.enh, h->head.refine, st)) return AFT_ERR_CUDA;
  if (!check_launch("aft_load_weights")) return AFT_ERR_CUDA;
  h->loaded = true;
  return AFT_OK;
}

size_t aft_workspace_bytes(const AftHandle* h, int64_t batch, int precision) {
  if (!h || batch < 0) { set_error("aft_workspace_bytes: bad argument"); return 0; }
  if (precision != AFT_FP32 && precision != AFT_BF16) { set_error("aft_workspace_bytes: bad precision"); return 0; }
  int64_t bc = batch < chunk_for(h, precision) ? batch : chunk_for(h, precision);
  if (bc < 1) bc = 1;
  if (h->generic) return generic_floats_per_chunk(h, bc, precision) * sizeof(float);
  return precision == AFT_BF16 ? tc_workspace_bytes(bc) : ws_bytes_f32(bc);
}

}  // extern "C"

namespace {

bool misaligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; }

// Destinations of a forward of `batch` > 0 samples, checked before anything is allocated, copied or launched, so that a
// refused call leaves no work behind.  `has_out`: the chunks are computed into a device buffer `out` (the caller's, or
// the staging lane of the host entry when `out` is NULL).  The fused tensor-core head stores whole rows by bulk copies;
// a reference-grid row is 13,440 bytes, so a 16-byte aligned base keeps every row aligned.  The scatter kernel of the
// other paths copies rows at any 8-byte offset, so gather buffers need an aligned base only.
int check_dst(const AftHandle* h, bool has_out, const void* out, const AftGather* g, int64_t batch, int precision,
              const char* fn) {
  const bool fused = !h->generic && precision == AFT_BF16;
  if (!has_out && !g) { set_error("%s: no destination (NULL out and no gather plan)", fn); return AFT_ERR_INVALID; }
  if (!has_out && !fused) {
    set_error("%s: this path needs a local `out` buffer (the scatter to the gather buffers reads it)", fn);
    return AFT_ERR_INVALID;
  }
  if (fused && out && misaligned16(out)) { set_error("%s: out is not 16-byte aligned", fn); return AFT_ERR_INVALID; }
  if (!g) return AFT_OK;
  if (g->world < 1 || g->world > 8 || g->rank < 0 || g->rank >= g->world || g->rows_per_rank < 0 || g->row0 < 0) {
    set_error("%s: bad gather plan (world %d, rank %d, rows_per_rank %lld, row0 %lld)", fn, g->world, g->rank,
              (long long)g->rows_per_rank, (long long)g->row0);
    return AFT_ERR_INVALID;
  }
  if (batch > g->rows_per_rank - g->row0) {
    set_error("%s: rows [%lld, %lld) exceed rows_per_rank %lld", fn, (long long)g->row0, (long long)(g->row0 + batch),
              (long long)g->rows_per_rank);
    return AFT_ERR_INVALID;
  }
  for (int p = 0; p < g->world; ++p) {
    if (!g->peer_out[p]) { set_error("%s: NULL gather buffer for rank %d", fn, p); return AFT_ERR_INVALID; }
    if (misaligned16(g->peer_out[p])) { set_error("%s: gather buffer of rank %d is not 16-byte aligned", fn, p); return AFT_ERR_INVALID; }
  }
  return AFT_OK;
}

// destinations of the chunk that starts at local sample c0: the caller's buffer (if any) and, with a gather plan, this
// rank's row range in every gather buffer (checked by check_dst)
void make_dst(const AftHandle* h, float2* out, const AftGather* g, int64_t c0, OutDst* dst) {
  dst->n = 0;
  if (out) dst->ptr[dst->n++] = out + c0 * h->pix;
  if (g)
    for (int p = 0; p < g->world; ++p)
      dst->ptr[dst->n++] = static_cast<float2*>(g->peer_out[p]) + (g->rank * g->rows_per_rank + g->row0 + c0) * h->pix;
}

int forward_impl(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread, const float* doppler,
                 void* out, int64_t batch, int precision, void* workspace, size_t workspace_bytes, void* stream, const AftGather* gather);

}  // namespace

extern "C" {

int aft_forward(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread, const float* doppler,
                void* out, int64_t batch, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (h && batch > 0 && !out) { set_error("aft_forward: NULL pilots / out"); return AFT_ERR_INVALID; }
  return forward_impl(h, pilots, snr, delay_spread, doppler, out, batch, precision, workspace, workspace_bytes, stream, nullptr);
}

int aft_forward_gather(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread, const float* doppler,
                       void* out, int64_t batch, int precision, void* workspace, size_t workspace_bytes, void* stream,
                       const AftGather* gather) {
  if (!gather) { set_error("aft_forward_gather: NULL gather plan"); return AFT_ERR_INVALID; }
  return forward_impl(h, pilots, snr, delay_spread, doppler, out, batch, precision, workspace, workspace_bytes, stream, gather);
}

}  // extern "C"

namespace {

int forward_impl(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread, const float* doppler,
                 void* out, int64_t batch, int precision, void* workspace, size_t workspace_bytes, void* stream, const AftGather* gather) {
  if (!h) { set_error("aft_forward: NULL handle"); return AFT_ERR_INVALID; }
  if (batch < 0) { set_error("aft_forward: negative batch"); return AFT_ERR_INVALID; }
  if (precision != AFT_FP32 && precision != AFT_BF16) { set_error("aft_forward: bad precision %d", precision); return AFT_ERR_INVALID; }
  if (!h->loaded) { set_error("aft_forward: weights not loaded (call aft_load_weights first)"); return AFT_ERR_STATE; }
  if (batch == 0) return AFT_OK;
  if (!pilots) { set_error("aft_forward: NULL pilots / out"); return AFT_ERR_INVALID; }
  if (h->cfg.adaptive) {
    if (!snr || !delay_spread || !doppler) {
      set_error("aft_forward: meta_data is required when channel adaptation is enabled");
      return AFT_ERR_INVALID;
    }
  }
  const bool fused = !h->generic && precision == AFT_BF16;   // the tensor-core head stores to all destinations itself
  int rc = check_dst(h, out != nullptr, out, gather, batch, precision, gather ? "aft_forward_gather" : "aft_forward");
  if (rc != AFT_OK) return rc;
  const size_t need = aft_workspace_bytes(h, batch, precision);
  if (!workspace || workspace_bytes < need) {
    set_error("aft_forward: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return AFT_ERR_WORKSPACE;
  }
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
    set_error("aft_forward: workspace must be 256-byte aligned");
    return AFT_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t chunk = chunk_for(h, precision);
  const float2* pin = static_cast<const float2*>(pilots);
  float2* pout = static_cast<float2*>(out);
  for (int64_t c0 = 0; c0 < batch; c0 += chunk) {
    const int64_t bc = batch - c0 < chunk ? batch - c0 : chunk;
    const float* s0 = h->cfg.adaptive ? snr + c0 : nullptr;
    const float* s1 = h->cfg.adaptive ? delay_spread + c0 : nullptr;
    const float* s2 = h->cfg.adaptive ? doppler + c0 : nullptr;
    OutDst dst;
    make_dst(h, fused ? pout : nullptr, gather, c0, &dst);
    if (h->generic) {
      rc = forward_chunk_generic(h, pin + c0 * h->P, s0, s1, s2, pout + c0 * h->pix, bc, static_cast<float*>(workspace), st, precision);
    } else if (precision == AFT_FP32) {
      rc = forward_chunk_f32(h, pin + c0 * kPilots, s0, s1, s2, pout + c0 * kPix, bc, static_cast<float*>(workspace), st);
    } else {
      TcProfileHook hook{h->profile ? &prof_mark_cb : nullptr, h};
      rc = tc_forward_chunk(h->tc, h->front, h->head, h->cfg.activation, h->sm_count, pin + c0 * kPilots, s0, s1, s2,
                            dst, bc, workspace, st, hook) ? AFT_OK : AFT_ERR_CUDA;
      if (h->profile) { h->prof_launches[0] += 1; h->prof_launches[1] += 1; h->prof_launches[2] += 1; }
    }
    if (rc != AFT_OK) return rc;
    if (!fused && gather && !launch_scatter_rows(pout + c0 * h->pix, bc * h->pix, dst, st)) return AFT_ERR_CUDA;
  }
  return AFT_OK;
}

}  // namespace

extern "C" {

int aft_forward_host(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                     const float* doppler, void* out, int64_t batch, int precision) {
  if (h && batch > 0 && !out) { set_error("aft_forward_host: NULL pilots / out"); return AFT_ERR_INVALID; }
  return aft_forward_host_gather(h, pilots, snr, delay_spread, doppler, out, batch, precision, nullptr);
}

int aft_forward_host_gather(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                            const float* doppler, void* out, int64_t batch, int precision, const AftGather* gather) {
  if (!h) { set_error("aft_forward_host: NULL handle"); return AFT_ERR_INVALID; }
  if (batch < 0) { set_error("aft_forward_host: negative batch"); return AFT_ERR_INVALID; }
  if (batch == 0) return AFT_OK;
  if (!pilots || (!out && !gather)) { set_error("aft_forward_host: NULL pilots / out"); return AFT_ERR_INVALID; }
  if (precision != AFT_FP32 && precision != AFT_BF16) { set_error("aft_forward_host: bad precision %d", precision); return AFT_ERR_INVALID; }
  if (!h->loaded) { set_error("aft_forward_host: weights not loaded (call aft_load_weights first)"); return AFT_ERR_STATE; }
  const bool ada = h->cfg.adaptive != 0;
  if (ada && (!snr || !delay_spread || !doppler)) {
    set_error("aft_forward_host: meta_data is required when channel adaptation is enabled");
    return AFT_ERR_INVALID;
  }
  // every chunk is computed into a staging lane, so the plan is all there is left to refuse
  int rc = check_dst(h, true, nullptr, gather, batch, precision, gather ? "aft_forward_host_gather" : "aft_forward_host");
  if (rc != AFT_OK) return rc;
  int64_t hc = batch < kHostChunk ? batch : kHostChunk;
  if (h->generic && hc > chunk_for(h, precision)) hc = chunk_for(h, precision);
  const size_t in_bytes = (size_t)hc * (h->P * sizeof(float2) + 3 * sizeof(float));
  const size_t out_bytes = (size_t)hc * h->pix * sizeof(float2);
  const size_t ws_need = aft_workspace_bytes(h, hc, precision);
  if (ws_need == 0) return AFT_ERR_INVALID;
  for (auto& ln : h->lanes) {
    if (!ln.stream) AFT_CUDA(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking));
    if (ln.cap < hc) {
      if (ln.d_in) cudaFree(ln.d_in);
      if (ln.d_out) cudaFree(ln.d_out);
      ln.d_in = ln.d_out = nullptr;
      AFT_CUDA(cudaMalloc(&ln.d_in, in_bytes));
      AFT_CUDA(cudaMalloc(&ln.d_out, out_bytes));
      ln.cap = hc;
    }
    if (ln.ws_bytes < ws_need) {
      if (ln.ws) cudaFree(ln.ws);
      ln.ws = nullptr;
      AFT_CUDA(cudaMalloc(&ln.ws, ws_need));
      ln.ws_bytes = ws_need;
    }
  }
  const char* hp = static_cast<const char*>(pilots);
  char* ho = static_cast<char*>(out);
  int lane = 0;
  // Chunk sizes taper towards the end (.., hc, hc/2, hc/4, hc/4): the device-to-host copy of the last chunk is the only
  // one that no compute hides, so the last chunk is small; partial waves of the small chunks are filled by the other lane.
  int64_t bc = 0;
  for (int64_t c0 = 0; c0 < batch; c0 += bc, lane ^= 1) {
    AftHandle::HostLane& ln = h->lanes[lane];
    const int64_t rem = batch - c0;
    bc = rem < hc ? rem : hc;
    if (!h->generic && batch > hc && rem <= hc + hc / 2 && rem > hc / 4) {
      bc = (rem / 2 + 63) / 64 * 64;
      if (bc < hc / 4) bc = hc / 4;
      if (bc > rem) bc = rem;
    }
    char* din = static_cast<char*>(ln.d_in);
    float* dmeta = reinterpret_cast<float*>(din + (size_t)ln.cap * h->P * sizeof(float2));
    // from the first copy on, a failure breaks out of the loop: the lanes are synchronised below before the call
    // returns, so no copy reads the caller's host buffers after it
    auto copy = [&](void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
      const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, ln.stream);
      if (e != cudaSuccess) { set_error("aft_forward_host: cudaMemcpyAsync failed: %s", cudaGetErrorString(e)); rc = AFT_ERR_CUDA; }
      return rc == AFT_OK;
    };
    if (!copy(din, hp + (size_t)c0 * h->P * sizeof(float2), (size_t)bc * h->P * sizeof(float2), cudaMemcpyHostToDevice)) break;
    if (ada && !(copy(dmeta, snr + c0, bc * sizeof(float), cudaMemcpyHostToDevice) &&
                 copy(dmeta + ln.cap, delay_spread + c0, bc * sizeof(float), cudaMemcpyHostToDevice) &&
                 copy(dmeta + 2 * ln.cap, doppler + c0, bc * sizeof(float), cudaMemcpyHostToDevice)))
      break;
    AftGather gsub;
    if (gather) { gsub = *gather; gsub.row0 = gather->row0 + c0; }
    rc = forward_impl(h, din, ada ? dmeta : nullptr, ada ? dmeta + ln.cap : nullptr, ada ? dmeta + 2 * ln.cap : nullptr,
                      ln.d_out, bc, precision, ln.ws, ln.ws_bytes, ln.stream, gather ? &gsub : nullptr);
    if (rc != AFT_OK) break;
    if (out && !copy(ho + (size_t)c0 * h->pix * sizeof(float2), ln.d_out, (size_t)bc * h->pix * sizeof(float2), cudaMemcpyDeviceToHost))
      break;
  }
  for (auto& ln : h->lanes) {
    const cudaError_t e = cudaStreamSynchronize(ln.stream);
    if (e != cudaSuccess && rc == AFT_OK) {
      set_error("aft_forward_host: cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
      rc = AFT_ERR_CUDA;
    }
  }
  return rc;
}

int aft_peer_alloc(size_t bytes, void** dev_ptr, void* handle64) {
  if (!dev_ptr || !handle64 || bytes == 0) { set_error("aft_peer_alloc: bad argument"); return AFT_ERR_INVALID; }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI documents a 64-byte handle");
  *dev_ptr = nullptr;
  AFT_CUDA(cudaMalloc(dev_ptr, bytes));
  cudaIpcMemHandle_t hd;
  const cudaError_t e = cudaIpcGetMemHandle(&hd, *dev_ptr);
  if (e != cudaSuccess) {
    set_error("aft_peer_alloc: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    cudaFree(*dev_ptr);
    *dev_ptr = nullptr;
    return AFT_ERR_CUDA;
  }
  memcpy(handle64, &hd, sizeof(hd));
  return AFT_OK;
}

int aft_peer_open(const void* handle64, void** dev_ptr) {
  if (!dev_ptr || !handle64) { set_error("aft_peer_open: bad argument"); return AFT_ERR_INVALID; }
  cudaIpcMemHandle_t hd;
  memcpy(&hd, handle64, sizeof(hd));
  *dev_ptr = nullptr;
  AFT_CUDA(cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return AFT_OK;
}

int aft_peer_close(void* dev_ptr) {
  if (!dev_ptr) return AFT_OK;
  AFT_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return AFT_OK;
}

int aft_peer_free(void* dev_ptr) {
  if (!dev_ptr) return AFT_OK;
  AFT_CUDA(cudaFree(dev_ptr));
  return AFT_OK;
}

int aft_error_sums(const void* est, const void* truth, int64_t count, double* sums, void* stream) {
  if (count < 0 || !sums || (count > 0 && (!est || !truth))) { set_error("aft_error_sums: bad argument"); return AFT_ERR_INVALID; }
  if (count == 0) return AFT_OK;
  return launch_error_sums(static_cast<const float2*>(est), static_cast<const float2*>(truth), count, sums,
                           static_cast<cudaStream_t>(stream)) ? AFT_OK : AFT_ERR_CUDA;
}

int aft_extract_pilots(const void* ls_grid, void* pilots, int32_t* counts, int64_t batch, int32_t cells, int32_t expected, void* stream) {
  if (batch < 0 || cells <= 0 || expected <= 0 || expected > cells || (batch > 0 && (!ls_grid || !pilots || !counts))) {
    set_error("aft_extract_pilots: bad argument");
    return AFT_ERR_INVALID;
  }
  return launch_extract_pilots(static_cast<const float2*>(ls_grid), static_cast<float2*>(pilots), counts, batch, cells, expected,
                               static_cast<cudaStream_t>(stream)) ? AFT_OK : AFT_ERR_CUDA;
}

int aft_linear_forward(const float* weight, const float* bias, const float* x, float* y, int64_t batch, int32_t in_dim, int32_t out_dim,
                       void* stream) {
  if (batch < 0 || in_dim <= 0 || out_dim <= 0 || !weight || !bias || (batch > 0 && (!x || !y))) {
    set_error("aft_linear_forward: bad argument");
    return AFT_ERR_INVALID;
  }
  if (in_dim > 4096) { set_error("aft_linear_forward: in_dim %d not supported (<= 4096)", in_dim); return AFT_ERR_UNSUPPORTED; }
  return launch_linear(weight, bias, x, y, batch, in_dim, out_dim, static_cast<cudaStream_t>(stream)) ? AFT_OK : AFT_ERR_CUDA;
}

size_t aft_linear_backward_workspace_bytes(int64_t batch, int32_t in_dim, int32_t out_dim) {
  if (batch < 0 || in_dim <= 0 || out_dim <= 0 || in_dim > 4096) {
    set_error("aft_linear_backward_workspace_bytes: bad shape (batch >= 0, 0 < in_dim <= 4096, out_dim > 0)");
    return 0;
  }
  return linear_backward_workspace_bytes(batch, in_dim, out_dim);
}

int aft_linear_backward(const float* weight, const float* x, const float* grad_y, float* grad_w, float* grad_b, float* grad_x,
                        int64_t batch, int32_t in_dim, int32_t out_dim, void* workspace, size_t workspace_bytes, void* stream) {
  if (batch < 0 || in_dim <= 0 || out_dim <= 0 || !weight || !grad_w || !grad_b || (batch > 0 && (!x || !grad_y))) {
    set_error("aft_linear_backward: bad argument");
    return AFT_ERR_INVALID;
  }
  if (in_dim > 4096) { set_error("aft_linear_backward: in_dim %d not supported (<= 4096)", in_dim); return AFT_ERR_INVALID; }
  const size_t need = linear_backward_workspace_bytes(batch, in_dim, out_dim);
  if (!workspace || workspace_bytes < need) {
    set_error("aft_linear_backward: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return AFT_ERR_WORKSPACE;
  }
  return launch_linear_backward(weight, x, grad_y, grad_w, grad_b, grad_x, batch, in_dim, out_dim, workspace,
                                static_cast<cudaStream_t>(stream)) ? AFT_OK : AFT_ERR_CUDA;
}

int aft_synthetic_channels(const AftConfig* cfg, uint64_t seed, int64_t sample0, int64_t batch, float* snr, float* delay_spread,
                           float* doppler, int32_t draw_conditions, void* pilots, void* truth, void* stream) {
  if (!cfg) { set_error("aft_synthetic_channels: NULL config"); return AFT_ERR_INVALID; }
  if (batch < 0 || sample0 < 0 || batch > INT64_MAX - sample0) {
    set_error("aft_synthetic_channels: samples [%lld, %lld + %lld) outside [0, 2^63)", (long long)sample0, (long long)sample0,
              (long long)batch);
    return AFT_ERR_INVALID;
  }
  const AftConfig& c = *cfg;
  if (c.num_scs <= 0 || c.num_symbols <= 0 || c.pilot_scs <= 0 || c.pilot_symbols <= 0 || c.pilot_scs > c.num_scs ||
      c.pilot_symbols > 2 || c.num_symbols <= (c.pilot_symbols == 2 ? 11 : 2)) {
    set_error("aft_synthetic_channels: bad grid %dx%d / pilots %dx%d (extents > 0, pilot_scs <= num_scs, pilot_symbols <= 2 at "
              "symbols [2, 11] < num_symbols)", c.num_scs, c.num_symbols, c.pilot_scs, c.pilot_symbols);
    return AFT_ERR_INVALID;
  }
  if (c.num_symbols > 256) {
    set_error("aft_synthetic_channels: num_symbols %d not supported (<= 256)", c.num_symbols);
    return AFT_ERR_UNSUPPORTED;
  }
  if (batch > 0 && (!snr || !delay_spread || !doppler || !pilots || !truth)) {
    set_error("aft_synthetic_channels: NULL condition / pilots / truth buffer");
    return AFT_ERR_INVALID;
  }
  if (batch > 0 && ((reinterpret_cast<uintptr_t>(pilots) | reinterpret_cast<uintptr_t>(truth)) & 7)) {
    set_error("aft_synthetic_channels: pilots / truth not 8-byte aligned (complex64)");
    return AFT_ERR_INVALID;
  }
  if (batch == 0) return AFT_OK;
  return launch_synthetic_channels(c, seed, sample0, batch, snr, delay_spread, doppler, draw_conditions != 0,
                                   static_cast<float2*>(pilots), static_cast<float2*>(truth), static_cast<cudaStream_t>(stream))
             ? AFT_OK : AFT_ERR_CUDA;
}

int aft_profile_enable(AftHandle* h, int enable) {
  if (!h) { set_error("aft_profile_enable: NULL handle"); return AFT_ERR_INVALID; }
  h->profile = enable != 0;
  h->prof_used = 0;
  h->prof_launches[0] = h->prof_launches[1] = h->prof_launches[2] = 0;
  return AFT_OK;
}

int aft_profile_read(AftHandle* h, double* ms, int64_t* launches) {
  if (!h || !ms || !launches) { set_error("aft_profile_read: NULL argument"); return AFT_ERR_INVALID; }
  ms[0] = ms[1] = ms[2] = 0.0;
  for (size_t i = 0; i + 3 < h->prof_used; i += 4) {
    AFT_CUDA(cudaEventSynchronize(h->prof_events[i + 3]));
    for (int s = 0; s < 3; ++s) {
      float t = 0.f;
      AFT_CUDA(cudaEventElapsedTime(&t, h->prof_events[i + s], h->prof_events[i + s + 1]));
      ms[s] += t;
    }
  }
  for (int s = 0; s < 3; ++s) { launches[s] = h->prof_launches[s]; h->prof_launches[s] = 0; }
  h->prof_used = 0;
  return AFT_OK;
}

int aft_selftest(int which, double* max_err, void* stream) {
  if (!max_err) { set_error("aft_selftest: NULL max_err"); return AFT_ERR_INVALID; }
  return tc_selftest(which, max_err, static_cast<cudaStream_t>(stream)) ? AFT_OK : AFT_ERR_CUDA;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// training path (train_fwd.cu / train_bwd.cu)
// ---------------------------------------------------------------------------------------------
namespace {

TrainModel train_model(const AftHandle* h) {
  return TrainModel{&h->front, &h->head, h->layers.data(), h->cfg.num_layers, h->cfg.activation, h->cfg.adaptive,
                    h->cfg.adapt_h1, h->cfg.adapt_h2, h->cfg.max_seq_len};
}

int train_unsupported(const char* fn) {
  set_error("%s: training covers only the reference default geometry (grid 120x14, pilots 12x2, patch 3x2)", fn);
  return AFT_ERR_UNSUPPORTED;
}

// common checks of aft_forward_train / aft_backward; fills *ws when the workspace is usable
int train_check_ws(const AftHandle* h, const char* fn, int64_t batch, void* workspace, size_t workspace_bytes, TrainWs* ws) {
  const size_t need = train_layout(nullptr, batch, h->cfg.num_layers).bytes;
  if (!workspace || workspace_bytes < need) {
    set_error("%s: workspace too small (%zu < %zu bytes)", fn, workspace_bytes, need);
    return AFT_ERR_WORKSPACE;
  }
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
    set_error("%s: workspace must be 256-byte aligned", fn);
    return AFT_ERR_WORKSPACE;
  }
  *ws = train_layout(workspace, batch, h->cfg.num_layers);
  return AFT_OK;
}

DropCfg drop_cfg(float p, uint64_t seed, int64_t sample0) {
  DropCfg d;
  d.thresh = (uint32_t)std::floor((double)p * 4294967296.0);
  d.scale = 1.0f / (1.0f - p);
  d.seed_lo = (uint32_t)(seed & 0xffffffffu);
  d.seed_hi = (uint32_t)(seed >> 32);
  d.seq0 = (uint32_t)(2 * sample0);   // < 2^32: checked by aft_forward_train_offset
  return d;
}

}  // namespace

extern "C" {

int64_t aft_param_count(const AftHandle* h) {
  if (!h) { set_error("aft_param_count: NULL handle"); return 0; }
  if (h->generic) { train_unsupported("aft_param_count"); return 0; }
  return (int64_t)grad_layout(train_model(h)).total;
}

size_t aft_train_workspace_bytes(const AftHandle* h, int64_t batch) {
  if (!h || batch < 0) { set_error("aft_train_workspace_bytes: bad argument"); return 0; }
  if (h->generic) { train_unsupported("aft_train_workspace_bytes"); return 0; }
  return train_layout(nullptr, batch, h->cfg.num_layers).bytes;
}

int aft_forward_train_offset(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                             const float* doppler, void* out, int64_t batch, int64_t sample0, float dropout, uint64_t seed,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) { set_error("aft_forward_train: NULL handle"); return AFT_ERR_INVALID; }
  if (h->generic) return train_unsupported("aft_forward_train");
  if (!(dropout >= 0.f && dropout < 1.f)) { set_error("aft_forward_train: dropout %g outside [0, 1)", (double)dropout); return AFT_ERR_INVALID; }
  if (batch < 0) { set_error("aft_forward_train: negative batch"); return AFT_ERR_INVALID; }
  // the global sequence index 2 * (sample0 + b) + part is the 32-bit second word of the Philox counter
  if (sample0 < 0 || sample0 > (int64_t{1} << 31) - batch) {
    set_error("aft_forward_train: samples [%lld, %lld) outside [0, 2^31)", (long long)sample0,
              (long long)sample0 + (long long)batch);
    return AFT_ERR_INVALID;
  }
  if (!h->loaded) { set_error("aft_forward_train: weights not loaded (call aft_load_weights first)"); return AFT_ERR_STATE; }
  if (batch == 0) return AFT_OK;
  if (!pilots || !out) { set_error("aft_forward_train: NULL pilots / out"); return AFT_ERR_INVALID; }
  if (h->cfg.adaptive && (!snr || !delay_spread || !doppler)) {
    set_error("aft_forward_train: meta_data is required when channel adaptation is enabled");
    return AFT_ERR_INVALID;
  }
  TrainWs ws;
  const int rc = train_check_ws(h, "aft_forward_train", batch, workspace, workspace_bytes, &ws);
  if (rc != AFT_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const DropCfg drop = drop_cfg(dropout, seed, sample0);
  // the header record tells aft_backward which forward filled the workspace (written on the device by the first kernel)
  const TrainHeader hdr{kTrainMagic, batch, h->cfg.num_layers, h->cfg.adaptive, dropout, drop.thresh, seed, sample0};
  if (!train_forward(train_model(h), hdr, static_cast<const float2*>(pilots), snr, delay_spread, doppler, static_cast<float2*>(out),
                     batch, drop, ws, st))
    return AFT_ERR_CUDA;
  return AFT_OK;
}

int aft_forward_train(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread, const float* doppler,
                      void* out, int64_t batch, float dropout, uint64_t seed, void* workspace, size_t workspace_bytes,
                      void* stream) {
  return aft_forward_train_offset(h, pilots, snr, delay_spread, doppler, out, batch, 0, dropout, seed, workspace,
                                  workspace_bytes, stream);
}

int aft_backward(AftHandle* h, const void* grad_out, int64_t batch, void* workspace, size_t workspace_bytes, float* grads,
                 void* stream) {
  if (!h) { set_error("aft_backward: NULL handle"); return AFT_ERR_INVALID; }
  if (h->generic) return train_unsupported("aft_backward");
  if (batch < 0) { set_error("aft_backward: negative batch"); return AFT_ERR_INVALID; }
  if (!h->loaded) { set_error("aft_backward: weights not loaded (call aft_load_weights first)"); return AFT_ERR_STATE; }
  if (batch == 0) return AFT_OK;
  if (!grad_out || !grads) { set_error("aft_backward: NULL grad_out / grads"); return AFT_ERR_INVALID; }
  if (!workspace || workspace_bytes < sizeof(TrainHeader) || (reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
    set_error("aft_backward: workspace NULL, too small or not 256-byte aligned");
    return AFT_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the header record of the forward: a 48-byte read-back, so this call synchronises with `stream`
  TrainHeader hdr{};
  AFT_CUDA(cudaMemcpyAsync(&hdr, workspace, sizeof(hdr), cudaMemcpyDeviceToHost, st));
  AFT_CUDA(cudaStreamSynchronize(st));
  if (hdr.magic != kTrainMagic || hdr.layers != h->cfg.num_layers || hdr.adaptive != h->cfg.adaptive) {
    set_error("aft_backward: the workspace was not filled by aft_forward_train of this estimator");
    return AFT_ERR_INVALID;
  }
  if (hdr.batch != batch) {
    set_error("aft_backward: batch %lld differs from the forward's %lld", (long long)batch, (long long)hdr.batch);
    return AFT_ERR_INVALID;
  }
  TrainWs ws;
  const int rc = train_check_ws(h, "aft_backward", batch, workspace, workspace_bytes, &ws);
  if (rc != AFT_OK) return rc;
  const DropCfg drop = drop_cfg(hdr.dropout, hdr.seed, hdr.sample0);
  if (!train_backward(train_model(h), static_cast<const float2*>(grad_out), batch, drop, ws, grads, st))
    return AFT_ERR_CUDA;
  return AFT_OK;
}

}  // extern "C"

