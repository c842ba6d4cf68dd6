// "Next" row N1 (SURVEY.md 8f): the reduction the reference evaluator performs right after the forward
// (src/main/trainer.py:338-345 via src/utils.py:164-180): sum |est - truth|^2 and sum |truth|^2 over
// complex64 arrays, accumulated in fp64 on the device (no per-batch host sync).
#include "aft_internal.cuh"

namespace aft {

namespace {

__global__ void __launch_bounds__(256)
error_sums_kernel(const float2* __restrict__ est, const float2* __restrict__ truth, int64_t n, double* sums) {
  double e = 0.0, p = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float2 a = est[i], b = truth[i];
    const float dr = a.x - b.x, di = a.y - b.y;
    e += (double)(dr * dr + di * di);
    p += (double)(b.x * b.x + b.y * b.y);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    e += __shfl_xor_sync(0xffffffffu, e, off);
    p += __shfl_xor_sync(0xffffffffu, p, off);
  }
  __shared__ double se[8], sp[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { se[warp] = e; sp[warp] = p; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double te = 0.0, tp = 0.0;
    for (int w = 0; w < 8; ++w) { te += se[w]; tp += sp[w]; }
    atomicAdd(&sums[0], te);
    atomicAdd(&sums[1], tp);
  }
}

// src -> every destination.  vec16 (the source and every destination 16-byte aligned): 16 bytes (two complex64) per
// access, an odd tail element copied by thread 0.  Otherwise 8 bytes per access: a row is pix * 8 bytes, so on a grid
// with odd pix a row at an odd offset is only 8-byte aligned.
__global__ void __launch_bounds__(256)
scatter_rows_kernel(const float2* __restrict__ src, int64_t count, OutDst dst, bool vec16) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (!vec16) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
      const float2 v = src[i];
      for (int d = 0; d < dst.n; ++d) dst.ptr[d][i] = v;
    }
    return;
  }
  const int64_t n4 = count >> 1;
  const float4* s4 = reinterpret_cast<const float4*>(src);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = s4[i];
    for (int d = 0; d < dst.n; ++d) reinterpret_cast<float4*>(dst.ptr[d])[i] = v;
  }
  if ((count & 1) && blockIdx.x == 0 && threadIdx.x == 0)
    for (int d = 0; d < dst.n; ++d) dst.ptr[d][count - 1] = src[count - 1];
}

}  // namespace

bool launch_scatter_rows(const float2* src, int64_t count, const OutDst& dst, cudaStream_t st) {
  if (dst.n <= 0 || count <= 0) return true;
  bool vec16 = (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  for (int d = 0; d < dst.n; ++d) vec16 = vec16 && (reinterpret_cast<uintptr_t>(dst.ptr[d]) & 15) == 0;
  int64_t blocks = (count / 2 + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  if (blocks < 1) blocks = 1;
  scatter_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, count, dst, vec16);
  count_launch();
  return check_launch("scatter_rows_kernel");
}

bool launch_error_sums(const float2* est, const float2* truth, int64_t count, double* sums, cudaStream_t st) {
  int64_t blocks = (count + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  error_sums_kernel<<<(unsigned)blocks, 256, 0, st>>>(est, truth, count, sums);
  count_launch();
  return check_launch("error_sums_kernel");
}

}  // namespace aft
