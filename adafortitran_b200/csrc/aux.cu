// "Next" rows N2 and N3 (SURVEY.md 8f), the callers / models either side of the hot path:
//   * pilot extraction -- what MatDataset._process_channel_data does per file (reference src/data/dataset.py:95-144):
//     the LS estimate arrives as a [subcarriers, symbols] grid that is zero off the pilot positions; the pilots are its
//     non-zero entries in row-major order.  Batched, on the device: one warp per sample, ballot + prefix compaction.
//     Index / byte work, HBM bound: reads 8 * scs * symbols bytes per sample.
//   * LinearEstimator -- y = W x + b with W [out, in] (reference src/models/linear.py:60-95).  HBM bound on the result
//     (4 * out bytes per sample against 4 * in read); W^T is staged in shared memory once per CTA.
#include "aft_internal.cuh"
#include "tc_ptx.cuh"

namespace aft {

namespace {

// grid[b][i] != 0+0j exactly as the reference's boolean mask (NaN counts as non-zero, -0.0 as zero)
__device__ __forceinline__ bool nonzero(float2 v) { return v.x != 0.0f || v.y != 0.0f; }

__global__ void __launch_bounds__(256)
extract_pilots_kernel(const float2* __restrict__ grid, float2* __restrict__ pilots, int32_t* __restrict__ counts, int64_t batch,
                      int cells, int expected) {
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp; b < batch; b += nwarps) {
    const float2* g = grid + b * cells;
    float2* out = pilots + b * expected;
    int found = 0;
    int base = 0;
    if ((cells & 1) == 0) {
      // two entries (16 bytes) per lane and four such loads in flight: 2 KB of the row per warp iteration
      const float4* g4 = reinterpret_cast<const float4*>(g);
      const int pairs = cells >> 1;
      for (; base + 4 * 32 <= pairs; base += 4 * 32) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = g4[base + u * 32 + lane];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float2 a = make_float2(v[u].x, v[u].y), c = make_float2(v[u].z, v[u].w);
          const bool na = nonzero(a), nc = nonzero(c);
          const unsigned ma = __ballot_sync(0xffffffffu, na), mc = __ballot_sync(0xffffffffu, nc);
          const int pa = found + __popc(ma & lt) + __popc(mc & lt);   // row-major: entries 2 lane, 2 lane + 1
          if (na && pa < expected) out[pa] = a;
          if (nc && pa + (na ? 1 : 0) < expected) out[pa + (na ? 1 : 0)] = c;
          found += __popc(ma) + __popc(mc);
        }
      }
      base *= 2;   // continue entry-wise
    }
    for (; base < cells; base += 32) {
      const int i = base + lane;
      float2 v = make_float2(0.f, 0.f);
      if (i < cells) v = g[i];
      const bool nz = i < cells && nonzero(v);
      const unsigned m = __ballot_sync(0xffffffffu, nz);
      const int pos = found + __popc(m & lt);
      if (nz && pos < expected) out[pos] = v;
      found += __popc(m);
    }
    if (lane == 0) counts[b] = found;
    // samples with fewer non-zeros than expected leave the remaining slots untouched; the host checks counts
  }
}

// LinearEstimator, weights in registers: thread <-> FOUR CONSECUTIVE output features (rows of W), each row held as
// kIn / 2 packed fp32 pairs (w_k, w_k+1).  Samples are streamed through shared memory in groups of kGroup; a 16-byte
// broadcast load delivers (x_k .. x_k+3), i.e. the packed operands of two FFMA2 per output: the accumulator pair of an
// output holds its even-k and odd-k partial sums, added at the end.  The result leaves as ONE 16-byte store per thread and
// sample: every variant with 4-byte stores (scalar FMA, FFMA2, 2 / 4 / 5 outputs per thread, 11 .. 27 warps) ran at the
// same ~800 clk per sample and SM, i.e. one warp-wide store instruction per ~15 clk -- the store path is paid per
// instruction, not per byte (a 16-byte-per-thread fill reaches 7.5 TB/s on this GPU, tools/write_bw.py).
template <int kIn, int kOut, int kThreadsL>
__global__ void __launch_bounds__(kThreadsL)
linear_regw_kernel(const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ x, float* __restrict__ y,
                   int64_t batch, int out_dim) {
  static_assert(kIn % 4 == 0, "four k steps per shared load");
  static_assert(kOut % 4 == 0, "16-byte stores");
  constexpr int kGroup = 64;
  __shared__ __align__(16) float xs[2][kGroup * kIn + 4];   // + 4: the pipelined load runs one step past the last sample
  const int nthr = out_dim / kOut;                          // out_dim % kOut == 0 (checked by the launcher)
  const bool owner = (int)threadIdx.x < nthr;
  unsigned long long wr[kOut][kIn / 2];
  float br[kOut];
#pragma unroll
  for (int j = 0; j < kOut; ++j) {
    const size_t o = (size_t)threadIdx.x * kOut + j;
    br[j] = owner ? bias[o] : 0.f;
#pragma unroll
    for (int k2 = 0; k2 < kIn / 2; ++k2) {
      const float a = owner ? w[o * kIn + 2 * k2] : 0.f, b = owner ? w[o * kIn + 2 * k2 + 1] : 0.f;
      asm("mov.b64 %0, {%1, %2};" : "=l"(wr[j][k2]) : "f"(a), "f"(b));
    }
  }
  // x groups arrive by 1-D bulk copies (one elected thread, completion on an mbarrier per buffer): the copy of group
  // g + 1 is issued before group g is computed, so no warp ever waits for a global load
  __shared__ __align__(8) unsigned long long bars[2];
  const uint32_t bar0 = ptx::smem_u32(&bars[0]);
  const int64_t stride = (int64_t)gridDim.x * kGroup;
  auto fetch = [&](int64_t g0, int b) {
    const uint32_t bytes = (uint32_t)((batch - g0 < kGroup ? batch - g0 : kGroup) * kIn * sizeof(float));
    ptx::mbar_arrive_expect_tx(bar0 + 8 * b, bytes);
    ptx::bulk_g2s(ptx::smem_u32(&xs[b][0]), x + g0 * kIn, bytes, bar0 + 8 * b);
  };
  if (threadIdx.x == 0) {
    ptx::mbar_init(bar0, 1);
    ptx::mbar_init(bar0 + 8, 1);
    ptx::fence_mbar_init();
    if ((int64_t)blockIdx.x * kGroup < batch) fetch((int64_t)blockIdx.x * kGroup, 0);
  }
  __syncthreads();
  int buf = 0;
  uint32_t it = 0;
  for (int64_t b0 = (int64_t)blockIdx.x * kGroup; b0 < batch; b0 += stride, buf ^= 1, ++it) {
    const int nb = (int)(batch - b0 < kGroup ? batch - b0 : kGroup);
    __syncthreads();   // every warp has finished the previous group: its buffer may be refilled
    if (threadIdx.x == 0 && b0 + stride < batch) {
      ptx::fence_proxy_async_smem();
      fetch(b0 + stride, buf ^ 1);
    }
    ptx::mbar_wait(bar0 + 8 * buf, (it >> 1) & 1);
    if (owner) {
      float4* yp = reinterpret_cast<float4*>(y + b0 * out_dim) + threadIdx.x * (kOut / 4);
      const ulonglong2* xp = reinterpret_cast<const ulonglong2*>(&xs[buf][0]);
      ulonglong2 xa = xp[0];                               // software pipeline: the next 16 bytes of x are in flight
      for (int s = 0; s < nb; ++s, yp += out_dim / 4, xp += kIn / 4) {
        unsigned long long acc[kOut];
#pragma unroll
        for (int j = 0; j < kOut; ++j) asm("mov.b64 %0, {%1, %2};" : "=l"(acc[j]) : "f"(br[j]), "f"(0.f));
#pragma unroll
        for (int k4 = 0; k4 < kIn / 4; ++k4) {
          const ulonglong2 xb = xp[k4 + 1];                // (x_k+4 .. x_k+7), or the next sample's first four (pad at the end)
#pragma unroll
          for (int j = 0; j < kOut; ++j) {
            asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc[j]) : "l"(wr[j][2 * k4]), "l"(xa.x));
            asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc[j]) : "l"(wr[j][2 * k4 + 1]), "l"(xa.y));
          }
          xa = xb;
        }
        float r[kOut];
#pragma unroll
        for (int j = 0; j < kOut; ++j) {
          float a0, a1;
          asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(acc[j]));
          r[j] = a0 + a1;
        }
#pragma unroll
        for (int j = 0; j < kOut; j += 4) yp[j / 4] = make_float4(r[j], r[j + 1], r[j + 2], r[j + 3]);
      }
    }
  }
}

// One CTA: W^T [in][out] in shared memory (when it fits), thread <-> output index, loop over the CTA's samples.
template <bool kSmemW>
__global__ void __launch_bounds__(256)
linear_kernel(const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ x, float* __restrict__ y,
              int64_t batch, int in_dim, int out_dim) {
  extern __shared__ float sm[];
  float* wt = sm;                                   // [in][out] (kSmemW)
  float* xs = sm + (kSmemW ? (size_t)in_dim * out_dim : 0);   // [8][in]: a group of samples
  if (kSmemW) {
    for (int i = threadIdx.x; i < in_dim * out_dim; i += blockDim.x) {
      const int o = i / in_dim, k = i - o * in_dim;   // coalesced read of W [out][in]
      wt[k * out_dim + o] = w[i];
    }
  }
  __syncthreads();
  constexpr int kGroup = 8;
  for (int64_t b0 = (int64_t)blockIdx.x * kGroup; b0 < batch; b0 += (int64_t)gridDim.x * kGroup) {
    const int nb = (int)(batch - b0 < kGroup ? batch - b0 : kGroup);
    for (int i = threadIdx.x; i < nb * in_dim; i += blockDim.x) xs[i] = x[b0 * in_dim + i];
    __syncthreads();
    for (int o = threadIdx.x; o < out_dim; o += blockDim.x) {
      float acc[kGroup];
      const float bo = bias[o];
#pragma unroll
      for (int j = 0; j < kGroup; ++j) acc[j] = bo;
      for (int k = 0; k < in_dim; ++k) {
        const float wk = kSmemW ? wt[k * out_dim + o] : w[(size_t)o * in_dim + k];
#pragma unroll
        for (int j = 0; j < kGroup; ++j) acc[j] = fmaf(wk, xs[j * in_dim + k], acc[j]);   // xs: broadcast reads
      }
#pragma unroll
      for (int j = 0; j < kGroup; ++j)
        if (j < nb) y[(b0 + j) * out_dim + o] = acc[j];
    }
    __syncthreads();
  }
}

// LinearEstimator backward: the three products of y = W x + b, all C[m][n] = sum_r A[r][m] B[r][n] in one kernel family.
//   kXgrad false: C[o][c] = sum_b gy[b][o] [x | 1][b][c]  -> grad_w[o][k] (c < in_dim) and grad_b[o] (c == in_dim)
//   kXgrad true : C[b][k] = sum_o gy[b][o] W[o][k]        -> grad_x
// A CTA owns a slab of kBwdTileM rows of C and TX * 4 of its columns; a thread owns 4 x 4 elements.  The reduction index r
// runs in groups of kBwdGroup staged in shared memory (the next group is loaded into registers while the current one is
// computed).  Each group's 32 products are summed in fp32 and the group sums are added in fp64, so the error does not
// grow with the length of the sum (10^6 samples, or out_dim = 45864 for grad_x).  The weight gradient splits the batch
// over blockIdx.z into contiguous ranges of whole groups (linear_bwd_plan); with more than one range every CTA writes an
// fp32 partial of its tile and linear_bwd_reduce_kernel adds the partials in range order in fp64.  No atomics anywhere:
// the same inputs give bit-identical gradients.  kVec: 16-byte global loads (the reference shape, 16-byte aligned gy,
// x and W, out_dim % 4 == 0); otherwise element loads with any alignment and any extents.
constexpr int kBwdTileM = 128, kBwdGroup = 32;

template <bool kXgrad, int TX, bool kVec>
__global__ void __launch_bounds__(32 * TX)
linear_bwd_kernel(const float* __restrict__ gy, const float* __restrict__ bop, float* __restrict__ c0, float* __restrict__ c1,
                  int64_t batch, int in_dim, int out_dim, int64_t range) {
  constexpr int kThreads = 32 * TX, kTileN = 4 * TX, G = kBwdGroup;
  constexpr int kA4 = (G * kBwdTileM / 4 + kThreads - 1) / kThreads;   // 16-byte A loads per thread and group
  constexpr int kA1 = (G * kBwdTileM + kThreads - 1) / kThreads;       // element A loads
  __shared__ __align__(16) float As[G][kBwdTileM + 4];
  __shared__ __align__(16) float Bs[G][kTileN];
  const int tid = threadIdx.x, tx = tid % TX, ty = tid / TX;
  const int64_t M = kXgrad ? batch : out_dim, R = kXgrad ? (int64_t)out_dim : batch;
  const int N = kXgrad ? in_dim : in_dim + 1;
  const int64_t m0 = (int64_t)blockIdx.x * kBwdTileM;
  const int n0 = blockIdx.y * kTileN;
  const int64_t r_begin = kXgrad ? 0 : (int64_t)blockIdx.z * range;
  const int64_t r_end = kXgrad ? R : (r_begin + range < R ? r_begin + range : R);

  // A[r][m]: gy[r][m] (weight gradient) or gy[m][r] (input gradient).  B[r][n]: [x | 1][r][n] or W[r][n].  Out of range: 0.
  auto a_at = [&](int64_t r, int64_t m) -> float {
    if (r >= r_end || m >= M) return 0.f;
    return kXgrad ? gy[m * out_dim + r] : gy[r * out_dim + m];
  };
  auto b_at = [&](int64_t r, int n) -> float {
    if (r >= r_end || n >= N) return 0.f;
    if (!kXgrad && n == in_dim) return 1.f;
    return bop[r * in_dim + n];
  };
  float4 pa4[kVec ? kA4 : 1], pb4;
  float pa1[kVec ? 1 : kA1], pb1[kVec ? 1 : 4];
  auto load = [&](int64_t r0) {
    if (kVec) {
#pragma unroll
      for (int i = 0; i < kA4; ++i) {
        const int idx = tid + i * kThreads;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (idx < G * kBwdTileM / 4) {
          // weight gradient: 4 consecutive outputs of one sample; input gradient: 4 consecutive outputs of one sample
          // (transposed into As on the store).  out_dim % 4 == 0, so a vector is either all in range or all out.
          const int64_t r = kXgrad ? r0 + 4 * (idx % (G / 4)) : r0 + idx / (kBwdTileM / 4);
          const int64_t m = kXgrad ? m0 + idx / (G / 4) : m0 + 4 * (idx % (kBwdTileM / 4));
          if (r < r_end && m < M) v = *reinterpret_cast<const float4*>(kXgrad ? gy + m * out_dim + r : gy + r * out_dim + m);
        }
        pa4[i] = v;
      }
      const int64_t r = r0 + ty;
      const int n = n0 + 4 * tx;   // in_dim % 4 == 0: a vector of B is all columns < in_dim or all >= in_dim
      pb4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < r_end && n < in_dim) pb4 = *reinterpret_cast<const float4*>(bop + r * in_dim + n);
      else if (r < r_end && !kXgrad && n == in_dim) pb4.x = 1.f;
    } else {
#pragma unroll
      for (int i = 0; i < kA1; ++i) {
        const int idx = tid + i * kThreads;
        // consecutive threads read consecutive addresses: m fastest (weight gradient), r fastest (input gradient)
        pa1[i] = idx >= G * kBwdTileM ? 0.f
                 : kXgrad ? a_at(r0 + idx % G, m0 + idx / G) : a_at(r0 + idx / kBwdTileM, m0 + idx % kBwdTileM);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int idx = tid + i * kThreads;
        pb1[i] = b_at(r0 + idx / kTileN, n0 + idx % kTileN);
      }
    }
  };
  auto store = [&]() {
    if (kVec) {
#pragma unroll
      for (int i = 0; i < kA4; ++i) {
        const int idx = tid + i * kThreads;
        if (idx >= G * kBwdTileM / 4) continue;
        if (kXgrad) {
          const int r = 4 * (idx % (G / 4)), m = idx / (G / 4);
          As[r][m] = pa4[i].x; As[r + 1][m] = pa4[i].y; As[r + 2][m] = pa4[i].z; As[r + 3][m] = pa4[i].w;
        } else {
          *reinterpret_cast<float4*>(&As[idx / (kBwdTileM / 4)][4 * (idx % (kBwdTileM / 4))]) = pa4[i];
        }
      }
      *reinterpret_cast<float4*>(&Bs[ty][4 * tx]) = pb4;
    } else {
#pragma unroll
      for (int i = 0; i < kA1; ++i) {
        const int idx = tid + i * kThreads;
        if (idx >= G * kBwdTileM) continue;
        if (kXgrad) As[idx % G][idx / G] = pa1[i];
        else As[idx / kBwdTileM][idx % kBwdTileM] = pa1[i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int idx = tid + i * kThreads;
        Bs[idx / kTileN][idx % kTileN] = pb1[i];
      }
    }
  };

  double dacc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) dacc[i][j] = 0.0;
  if (r_begin < r_end) load(r_begin);
  for (int64_t r0 = r_begin; r0 < r_end; r0 += G) {
    store();
    __syncthreads();
    if (r0 + G < r_end) load(r0 + G);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 8
    for (int r = 0; r < G; ++r) {
      const float4 a = *reinterpret_cast<const float4*>(&As[r][4 * ty]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[r][4 * tx]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dacc[i][j] += acc[i][j];
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + 4 * ty + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + 4 * tx + j;
      if (n >= N) continue;
      const float v = (float)dacc[i][j];
      if (kXgrad) c0[m * in_dim + n] = v;
      else if (gridDim.z > 1) c0[((int64_t)blockIdx.z * M + m) * N + n] = v;   // partial of batch range z, [z][o][in_dim + 1]
      else if (n < in_dim) c0[m * in_dim + n] = v;
      else c1[m] = v;
    }
  }
}

// grad_w / grad_b from the partials of the nz batch ranges, summed in range order in fp64
__global__ void __launch_bounds__(256)
linear_bwd_reduce_kernel(const float* __restrict__ part, int nz, int64_t count, int in_dim, float* __restrict__ grad_w,
                         float* __restrict__ grad_b) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double s = 0.0;
  for (int z = 0; z < nz; ++z) s += part[z * count + i];
  const int64_t o = i / (in_dim + 1);
  const int c = (int)(i - o * (in_dim + 1));
  if (c < in_dim) grad_w[o * in_dim + c] = (float)s;
  else grad_b[o] = (float)s;
}

// Split of the batch for the weight gradient, a function of the shape only (so the workspace size is too): enough
// batch ranges for ~4 CTAs per SM, at most 64, each a whole number of groups; no split once the tiles alone fill that.
struct LinearBwdPlan {
  int64_t nz, range;
};
LinearBwdPlan linear_bwd_plan(int64_t batch, int in_dim, int out_dim) {
  constexpr int64_t kTarget = 4 * 148, kMaxSplit = 64;
  const int64_t tiles = (out_dim + kBwdTileM - 1) / kBwdTileM * ((in_dim + 1 + 31) / 32);
  const int64_t groups = (batch + kBwdGroup - 1) / kBwdGroup;
  int64_t nz = tiles >= kTarget ? 1 : (kTarget + tiles - 1) / tiles;
  if (nz > kMaxSplit) nz = kMaxSplit;
  if (nz > groups) nz = groups;
  if (nz < 1) nz = 1;
  const int64_t per = groups > 0 ? (groups + nz - 1) / nz : 1;   // groups per range
  return {groups > 0 ? (groups + per - 1) / per : 1, per * kBwdGroup};
}

}  // namespace

size_t linear_backward_workspace_bytes(int64_t batch, int in_dim, int out_dim) {
  const LinearBwdPlan p = linear_bwd_plan(batch, in_dim, out_dim);
  const size_t part = p.nz > 1 ? (size_t)p.nz * out_dim * (in_dim + 1) * sizeof(float) : 0;
  return part > 256 ? part : 256;
}

bool launch_linear_backward(const float* w, const float* x, const float* gy, float* grad_w, float* grad_b, float* grad_x,
                            int64_t batch, int in_dim, int out_dim, void* workspace, cudaStream_t st) {
  if (batch == 0) {   // empty sums: zero gradients
    if (cudaMemsetAsync(grad_w, 0, (size_t)out_dim * in_dim * sizeof(float), st) != cudaSuccess ||
        cudaMemsetAsync(grad_b, 0, (size_t)out_dim * sizeof(float), st) != cudaSuccess) {
      set_error("aft_linear_backward: cudaMemsetAsync failed");
      return false;
    }
    return true;
  }
  auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool ref = in_dim == 24 && out_dim % 4 == 0 && a16(gy);   // the reference shape: 16-byte loads
  const LinearBwdPlan p = linear_bwd_plan(batch, in_dim, out_dim);
  float* part = p.nz > 1 ? static_cast<float*>(workspace) : grad_w;
  // columns of [x | 1]: 28 per CTA on the fast path (24 + bias + 3 zero), 32 otherwise; one column tile for in_dim = 24
  // either way, so the split does not depend on the path
  const dim3 gw((unsigned)((out_dim + kBwdTileM - 1) / kBwdTileM), (unsigned)((in_dim + 1 + 31) / 32), (unsigned)p.nz);
  if (ref && a16(x)) {
    linear_bwd_kernel<false, 7, true><<<gw, 32 * 7, 0, st>>>(gy, x, part, grad_b, batch, in_dim, out_dim, p.range);
  } else {
    linear_bwd_kernel<false, 8, false><<<gw, 32 * 8, 0, st>>>(gy, x, part, grad_b, batch, in_dim, out_dim, p.range);
  }
  count_launch();
  if (!check_launch("linear_bwd_kernel")) return false;
  if (p.nz > 1) {
    const int64_t count = (int64_t)out_dim * (in_dim + 1);
    linear_bwd_reduce_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(part, (int)p.nz, count, in_dim, grad_w, grad_b);
    count_launch();
    if (!check_launch("linear_bwd_reduce_kernel")) return false;
  }
  if (grad_x) {
    const unsigned rows = (unsigned)((batch + kBwdTileM - 1) / kBwdTileM);
    if (ref && a16(w)) {
      linear_bwd_kernel<true, 6, true><<<dim3(rows, 1), 32 * 6, 0, st>>>(gy, w, grad_x, nullptr, batch, in_dim, out_dim, 0);
    } else {
      linear_bwd_kernel<true, 8, false><<<dim3(rows, (unsigned)((in_dim + 31) / 32)), 32 * 8, 0, st>>>(gy, w, grad_x, nullptr, batch,
                                                                                                     in_dim, out_dim, 0);
    }
    count_launch();
    if (!check_launch("linear_bwd_kernel")) return false;
  }
  return true;
}

bool launch_extract_pilots(const float2* grid, float2* pilots, int32_t* counts, int64_t batch, int cells, int expected, cudaStream_t st) {
  if (batch <= 0) return true;
  int64_t blocks = (batch + 7) / 8;           // 8 warps per CTA, one sample per warp per pass
  if (blocks > 148 * 8) blocks = 148 * 8;
  extract_pilots_kernel<<<(unsigned)blocks, 256, 0, st>>>(grid, pilots, counts, batch, cells, expected);
  count_launch();
  return check_launch("extract_pilots_kernel");
}

bool launch_linear(const float* w, const float* bias, const float* x, float* y, int64_t batch, int in_dim, int out_dim, cudaStream_t st) {
  if (batch <= 0) return true;
  if (in_dim == 24 && out_dim % 4 == 0 && out_dim <= 4 * 448 && ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x)) & 15) == 0) {
    // the reference configuration (24 pilots -> 1680 grid points): 420 owner threads x 4 consecutive outputs
    int64_t nb = (batch + 63) / 64;
    if (nb > 148) nb = 148;                   // 14 warps x 128 registers: one CTA per SM, grid-stride over sample groups
    linear_regw_kernel<24, 4, 448><<<(unsigned)nb, 448, 0, st>>>(w, bias, x, y, batch, out_dim);
    count_launch();
    return check_launch("linear_regw_kernel");
  }
  const size_t wbytes = (size_t)in_dim * out_dim * sizeof(float), xbytes = (size_t)8 * in_dim * sizeof(float);
  int64_t blocks = (batch + 7) / 8;
  if (blocks > 148) blocks = 148;              // persistent: W^T is staged once per CTA
  if (wbytes + xbytes <= 200 * 1024) {
    if (cudaFuncSetAttribute(linear_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(wbytes + xbytes)) != cudaSuccess) {
      set_error("linear_kernel: cannot opt in to %zu bytes of shared memory", wbytes + xbytes);
      return false;
    }
    linear_kernel<true><<<(unsigned)blocks, 256, wbytes + xbytes, st>>>(w, bias, x, y, batch, in_dim, out_dim);
  } else {
    if (xbytes > 48 * 1024 &&
        cudaFuncSetAttribute(linear_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xbytes) != cudaSuccess) {
      set_error("linear_kernel: cannot opt in to %zu bytes of shared memory", xbytes);
      return false;
    }
    if (blocks < 148 && out_dim > 4096) blocks = 148;   // few samples, many outputs: idle CTAs cost nothing
    linear_kernel<false><<<(unsigned)blocks, 256, xbytes, st>>>(w, bias, x, y, batch, in_dim, out_dim);
  }
  count_launch();
  return check_launch("linear_kernel");
}

}  // namespace aft
