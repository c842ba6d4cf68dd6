/*
 * aft.h -- C-ABI of the B200-native AdaFortiTran / FortiTran inference forward pass.
 *
 * This is the drop-in boundary below the reference's Python operator API.  The reference has no FFI
 * of its own (pure PyTorch): its "operator interface" for the hot path is the nn.Module surface of
 * src/models (reference file:line in each entry below).  A maintainer binds these entry points with
 * ctypes (see INTEGRATION.md); adafortitran_b200/_capi.py is that binding.
 *
 * Conventions: plain C, plain pointers and sizes, no torch / CUDA types in signatures (a stream is
 * passed as void* == cudaStream_t).  Every function returns AFT_OK (0) or a negative AftStatus and
 * never throws; aft_last_error() gives the message for the calling thread.  All "device" pointers
 * must belong to the CUDA device that was current when aft_create() ran.  There is no CPU fallback:
 * without a sm_100-class device aft_create() fails with AFT_ERR_CUDA.
 */
#ifndef AFT_H_
#define AFT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AFT_ABI_VERSION 3

#if defined(__GNUC__)
#define AFT_API __attribute__((visibility("default")))
#else
#define AFT_API
#endif

typedef enum AftStatus {
  AFT_OK = 0,
  AFT_ERR_INVALID = -1,      /* bad argument (NULL pointer, negative size, ...)                      */
  AFT_ERR_UNSUPPORTED = -2,  /* configuration outside what the sm_100a kernels are specialised for   */
  AFT_ERR_CUDA = -3,         /* a CUDA runtime call or kernel launch failed; see aft_last_error()    */
  AFT_ERR_WORKSPACE = -4,    /* workspace pointer NULL / too small for this batch                    */
  AFT_ERR_STATE = -5         /* forward before aft_load_weights()                                    */
} AftStatus;

typedef enum AftPrecision {
  AFT_FP32 = 0,  /* CUDA-core fp32 FMA path; parity gate: max|y-ref|/max|ref| <= 1e-4               */
  AFT_BF16 = 1   /* tcgen05 path: bf16 MMA operands, fp32 accumulate / softmax / LayerNorm / residual */
} AftPrecision;

typedef enum AftActivation { AFT_ACT_RELU = 0, AFT_ACT_GELU = 1 } AftActivation;

/* Shape of one estimator.  Mirrors SystemConfig + ModelConfig (reference src/config/schemas.py:20-45,
 * 113-175; config/system_config.yaml, config/adafortitran.yaml, config/fortitran.yaml). */
typedef struct AftConfig {
  int32_t num_scs, num_symbols;        /* ofdm.num_scs, ofdm.num_symbols            (120, 14) */
  int32_t pilot_scs, pilot_symbols;    /* pilot.num_scs, pilot.num_symbols          (12, 2)   */
  int32_t patch_scs, patch_symbols;    /* patch_size                                (3, 2)    */
  int32_t num_layers;                  /* num_layers                                (6)       */
  int32_t model_dim, num_head;         /* model_dim, num_head                       (128, 4)  */
  int32_t ff_dim;                      /* 2*model_dim, reference encoders.py:47     (256)     */
  int32_t activation;                  /* AftActivation                             (gelu)    */
  int32_t adaptive;                    /* 1 = AdaFortiTranEstimator, 0 = FortiTranEstimator   */
  int32_t adapt_h1, adapt_h2, adapt_h3;/* channel_adaptivity_hidden_sizes           (7,42,560)*/
  int32_t adaptive_token_length;       /* adaptive_token_length                     (6)       */
  int32_t max_seq_len;                 /* rows of the positional table              (512)     */
} AftConfig;

/* Device pointers to the fp32 parameters, torch layouts ([out, in] row-major for Linear,
 * [cout, cin, 3, 3] for Conv2d).  Names follow the reference state_dict (SURVEY.md Appendix A). */
typedef struct AftConvStack {          /* ConvEnhancer, reference enhancers.py:12-20 */
  const float* w[4];                   /* conv_block.{0,2,4,6}.weight */
  const float* b[4];                   /* conv_block.{0,2,4,6}.bias   */
} AftConvStack;

typedef struct AftMlp {                /* one ChannelAdapter encoder, channel_adaptivity.py:34-40 */
  const float* w[3];                   /* {0,2,4}.weight: [h1,1], [h2,h1], [h3,h2] */
  const float* b[3];
} AftMlp;

typedef struct AftEncoderLayer {       /* nn.TransformerEncoderLayer, reference encoders.py:44-51 */
  const float *in_proj_w, *in_proj_b;  /* self_attn.in_proj_{weight,bias}: [3d,d], [3d]; rows q|k|v */
  const float *out_proj_w, *out_proj_b;/* self_attn.out_proj: [d,d], [d]                            */
  const float *lin1_w, *lin1_b;        /* linear1: [ff,d], [ff]                                     */
  const float *lin2_w, *lin2_b;        /* linear2: [d,ff], [d]                                      */
  const float *norm1_w, *norm1_b, *norm2_w, *norm2_b;
} AftEncoderLayer;

typedef struct AftWeights {
  const float *upsampler_w, *upsampler_b;   /* pilot_upsampler: [num_scs*num_symbols, pilot_scs*pilot_symbols] */
  AftConvStack initial_enhancer, final_refiner;
  AftMlp snr_encoder, ds_encoder, dop_encoder; /* ignored unless adaptive */
  const float *linear_1_w, *linear_1_b;     /* transformer_encoder.linear_1: [d, patch_len(+adaptive_token_length)] */
  const float *pos_table;                   /* position_embeddings or pe: [max_seq_len, d] */
  const float *linear_2_w, *linear_2_b;     /* transformer_encoder.linear_2: [patch_len, d] */
  const AftEncoderLayer* layers;            /* host array of num_layers entries */
  int32_t num_layers;
} AftWeights;

typedef struct AftHandle AftHandle;

/* ABI version of the loaded library (== AFT_ABI_VERSION of the header it was built from). */
AFT_API int aft_abi_version(void);

/* Message of the last failure on the calling thread ("" if none). */
AFT_API const char* aft_last_error(void);

/* Replaces the constructor BaseFortiTranEstimator.__init__ / _setup_dimensions / _build_architecture
 * (reference src/models/fortitran.py:23-126).  Validates the shape against what the kernels support and
 * allocates the packed-weight arena on the current device.  Supported: model_dim 128, 4 heads, ff 256, patch sizes
 * dividing the grid.  The reference default geometry (grid 120x14, pilots 12x2, patch 3x2) runs on kernels specialised
 * for it in both precisions; any other geometry (e.g. 3276x14: 7644 tokens) runs on the shape-generic kernels: AFT_FP32
 * on CUDA cores, AFT_BF16 on the long-sequence tensor-core path (sequence in global memory, streaming attention). */
AFT_API int aft_create(const AftConfig* cfg, AftHandle** out);
AFT_API void aft_destroy(AftHandle* h);

/* Replaces nn.Module.load_state_dict / parameter ownership (reference src/main/trainer.py:683-703).
 * Reads the fp32 parameters (device pointers) and builds the private packed copies (fp32 re-layouts and
 * bf16 MMA operand images).  Call again whenever a parameter changes.  Asynchronous on `stream`. */
AFT_API int aft_load_weights(AftHandle* h, const AftWeights* w, void* stream);

/* Bytes of device scratch aft_forward needs for a batch of `batch` samples at `precision`
 * (0 on error).  Large batches are processed in internal chunks, so this saturates. */
AFT_API size_t aft_workspace_bytes(const AftHandle* h, int64_t batch, int precision);

/* Replaces BaseFortiTranEstimator.forward (reference src/models/fortitran.py:145-182) on device buffers.
 *   pilots : complex64 [batch, pilot_scs, pilot_symbols], interleaved re/im        (device)
 *   snr, delay_spread, doppler : float32 [batch]; all NULL iff the handle is not adaptive (device)
 *   out    : complex64 [batch, num_scs, num_symbols], interleaved re/im            (device, 16-byte aligned)
 * Asynchronous on `stream`; no allocation, no host synchronisation. */
AFT_API int aft_forward(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                const float* doppler, void* out, int64_t batch, int precision,
                void* workspace, size_t workspace_bytes, void* stream);

/* Same contract with HOST buffers (pinned or pageable): the call stages host->device copies of the
 * inputs and the device->host copy of the estimates itself, chunked and overlapped with compute on
 * internal streams, and returns after the last byte of `out` has landed.  This is the end-to-end
 * entry point bench.py times as `e2e`. */
AFT_API int aft_forward_host(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                     const float* doppler, void* out, int64_t batch, int precision);

/* Multi-GPU evaluation path (SURVEY.md §8e; caller contract: reference src/main/trainer.py:328-347, one process per
 * GPU, batch-sharded replicas).  The all-gather of the estimates is FUSED into the forward: the kernel that produces
 * the complex64 estimates stores every 16-byte vector to all `world` gather buffers -- its own and the peers', which are
 * peer device memory mapped into this process (aft_peer_open) and are written with plain stores over NVLink while the
 * next samples are being computed.  Local sample i lands at row  rank * rows_per_rank + row0 + i  of every
 * peer_out[p] (complex64 [world * rows_per_rank, num_scs, num_symbols]).  The stores are complete (and visible to the
 * peers) when the work enqueued on `stream` has completed on every rank: follow the call with a cross-rank
 * synchronisation on the same stream (the evaluator's NCCL all-reduce of the error sums does it) before reading. */
typedef struct AftGather {
  void* peer_out[8];      /* gather buffer of every rank as seen from THIS process, peer_out[rank] = the local one */
  int32_t world, rank;    /* 1 <= world <= 8                                                                     */
  int64_t rows_per_rank;  /* samples per rank in the gathered array                                              */
  int64_t row0;           /* offset of this call's first sample inside the rank's shard (chunked callers)        */
} AftGather;

/* aft_forward with the fused all-gather.  `out` may be NULL (the estimates then only go to the gather buffers). */
AFT_API int aft_forward_gather(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                const float* doppler, void* out, int64_t batch, int precision,
                void* workspace, size_t workspace_bytes, void* stream, const AftGather* gather);

/* aft_forward_host with the fused all-gather: host inputs in, estimates of the local shard out to `out` (host, may be
 * NULL) and to every gather buffer.  Returns after the local work has completed (peers: see above). */
AFT_API int aft_forward_host_gather(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                     const float* doppler, void* out, int64_t batch, int precision, const AftGather* gather);

/* Peer-visible device memory for the gather buffers: cudaMalloc + cudaIpcGetMemHandle on the owner, cudaIpcOpenMemHandle
 * (peer access enabled lazily) on the other ranks of the node.  `handle` is a 64-byte opaque blob the caller moves
 * between the processes (torch.distributed.all_gather_object in adafortitran_b200/distributed.py). */
AFT_API int aft_peer_alloc(size_t bytes, void** dev_ptr, void* handle64);
AFT_API int aft_peer_open(const void* handle64, void** dev_ptr);
AFT_API int aft_peer_close(void* dev_ptr);
AFT_API int aft_peer_free(void* dev_ptr);

/* "Next" row N1 (SURVEY.md §8f): the reduction ModelEvaluator._evaluate_dataloader performs right after the
 * forward (reference src/main/trainer.py:338-345 with src/utils.py:164-180): accumulates
 * sums[0] += sum|est-truth|^2, sums[1] += sum|truth|^2 over complex64 [count] arrays (device, fp64 sums). */
AFT_API int aft_error_sums(const void* est, const void* truth, int64_t count, double* sums, void* stream);

/* "Next" row N2: batched form of MatDataset._process_channel_data (reference src/data/dataset.py:95-144): the pilots
 * of a sample are the non-zero entries of its sparse LS grid (complex64 [batch, cells], cells = subcarriers * symbols,
 * row-major), in row-major order.  Writes the first `expected` of them to pilots[batch, expected] and the number of
 * non-zero entries found to counts[batch] (int32, device); a count != expected is the reference's ValueError and is
 * raised by the host binding.  All pointers are device pointers. */
AFT_API int aft_extract_pilots(const void* ls_grid, void* pilots, int32_t* counts, int64_t batch, int32_t cells,
                               int32_t expected, void* stream);

/* "Next" row N3: LinearEstimator.forward (reference src/models/linear.py:60-95): y[batch, out_dim] =
 * x[batch, in_dim] . W[out_dim, in_dim]^T + bias, fp32, device pointers. */
AFT_API int aft_linear_forward(const float* weight, const float* bias, const float* x, float* y, int64_t batch,
                               int32_t in_dim, int32_t out_dim, void* stream);

/* Number of kernel launches issued by this library on the calling process since load (for bench.py). */
AFT_API int64_t aft_launch_count(void);

/* Stage timing for bench.py's roofline: when enabled, aft_forward brackets the frontend, encoder and head
 * launches of every chunk with CUDA events on the launch stream.  aft_profile_read synchronises on the recorded
 * events, returns the accumulated milliseconds per stage (ms[0..2] = frontend, encoder, head) and the number of
 * launches per stage, and resets the accumulators.  fp32 path: "encoder" covers its GEMM + attention kernels. */
AFT_API int aft_profile_enable(AftHandle* h, int enable);
AFT_API int aft_profile_read(AftHandle* h, double* ms, int64_t* launches);

/* ---- Training (AFT_FP32 on CUDA cores, reference default geometry only) ----------------------------------------
 * A handle on any other geometry returns AFT_ERR_UNSUPPORTED from the five calls below.
 *
 * Flat gradient layout: every parameter in torch layout without padding, in this order:
 *   pilot_upsampler w, b;  initial_enhancer w0 b0 w1 b1 w2 b2 w3 b3;  final_refiner w0 b0 .. w3 b3;
 *   (adaptive only) snr_encoder w0 b0 w1 b1 w2 b2, ds_encoder ..., dop_encoder ...;
 *   linear_1 w, b;  positional table [max_seq_len, model_dim] (rows >= 280 are 0);  linear_2 w, b;
 *   per encoder layer: in_proj w b, out_proj w b, linear1 w b, linear2 w b, norm1 w b, norm2 w b.
 *
 * Dropout: nn.TransformerEncoderLayer's four sites (post-norm): 0 the attention probabilities, element index
 * (head*S + q)*S + k; 1 the out_proj output before the residual add, row*128 + col; 2 the FFN activation,
 * row*256 + col; 3 the linear2 output before the residual add, row*128 + col (row = token of the sequence).
 * Element i of sequence seq = 2 * (sample0 + sample) + part (part 0 re, 1 im; sample = the index within the call,
 * sample0 = the global index of the call's first sample, 0 for aft_forward_train) in layer l at site s takes output
 * word i & 3 of Philox4x32-10 with key (seed & 0xffffffff, seed >> 32) and counter (i >> 2, seq, (l << 8) | s, 0),
 * and is kept iff that word >= floor(p * 2^32) (p as float, widened to double); kept values are scaled by 1 / (1 - p).
 * So a batch split into calls over consecutive sample ranges, each with its sample0 and the same seed, draws exactly
 * the masks of one call over the whole batch. */

/* Floats in the flat gradient buffer of aft_backward (0 on error). */
AFT_API int64_t aft_param_count(const AftHandle* h);
/* Bytes of the training workspace for `batch` samples: saved activations + backward scratch (0 on error). */
AFT_API size_t aft_train_workspace_bytes(const AftHandle* h, int64_t batch);
/* Training forward, AFT_FP32 only: as aft_forward, plus dropout with probability `dropout` (0 <= p < 1) at the four
 * sites of nn.TransformerEncoderLayer, masks drawn from `seed` (see "Dropout" above); saves what aft_backward needs in
 * `workspace` (256-byte aligned).  Asynchronous on `stream`, no allocation, no host synchronisation.  With p = 0 the
 * output is bit-identical to aft_forward at AFT_FP32. */
AFT_API int aft_forward_train(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                              const float* doppler, void* out, int64_t batch, float dropout, uint64_t seed,
                              void* workspace, size_t workspace_bytes, void* stream);
/* aft_forward_train for samples sample0 .. sample0 + batch - 1 of a larger (e.g. data-parallel) batch: the dropout masks
 * use the global sequence index (see "Dropout" above); aft_forward_train is the case sample0 = 0.  The sequence index is
 * the 32-bit second counter word, so AFT_ERR_INVALID, with nothing launched, unless 0 <= sample0 and
 * sample0 + batch <= 2^31.  aft_backward reads sample0 from the workspace with the seed and p. */
AFT_API int aft_forward_train_offset(AftHandle* h, const void* pilots, const float* snr, const float* delay_spread,
                                     const float* doppler, void* out, int64_t batch, int64_t sample0, float dropout,
                                     uint64_t seed, void* workspace, size_t workspace_bytes, void* stream);
/* Gradients of all parameters for grad_out = dL/d(out) (complex64 [batch, num_scs, num_symbols]: re = dL/dRe, im = dL/dIm).
 * Overwrites grads[aft_param_count(h)] (fp32, device).  Consumes the workspace of the aft_forward_train call it follows;
 * reads that call's header record back first (so it synchronises with `stream`) and returns AFT_ERR_INVALID when
 * `batch` differs from it.  Deterministic: the same inputs and seed give bit-identical gradients. */
AFT_API int aft_backward(AftHandle* h, const void* grad_out, int64_t batch, void* workspace, size_t workspace_bytes,
                         float* grads, void* stream);

/* Device-side self tests of the tcgen05 building blocks against SIMT code (returns max abs error in
 * *max_err; used by tests/ to localise failures).  which: 0 = UMMA GEMM tile, 1 = attention tile. */
AFT_API int aft_selftest(int which, double* max_err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AFT_H_ */
