// Synthetic doubly-selective channels and noisy pilots on the device (include/aft.h, "Synthetic channels").
// Every random number of a sample comes from Philox4x32-10 (train.cuh) with the sample's 64-bit global index in the
// counter, so a sample is the same whichever call, chunk or rank computes it.
#include <cmath>

#include "aft_internal.cuh"
#include "train.cuh"

namespace aft {

namespace {

constexpr int kTaps = 8;
constexpr uint32_t kSynthTag = 0x53594E54u;          // "SYNT": fourth counter word; dropout counters have 0 there
constexpr double kSubcarrierHz = 15e3;
constexpr double kSymbolSec = 1e-3 / 14;
constexpr int kCtasPerSm = 4;

struct SynthArgs {
  int num_scs, num_symbols, pilot_scs, pilot_symbols;
  int pilot_step;           // num_scs / pilot_scs
  uint32_t k0, k1;          // seed lo / hi
  int64_t sample0, batch;
  float *snr, *ds, *dop;
  int draw;
  float2 *pilots, *truth;
  int cols;                 // threads per truth row: num_symbols / V
  int rows;                 // rows of a pass: blockDim.x / cols
  int chunk;                // subcarriers whose frequency factors are held in shared memory at a time
};

__device__ __forceinline__ uint4 draw(const SynthArgs& a, uint64_t s, uint32_t j) {
  return philox4x32_10(make_uint4(j, (uint32_t)s, (uint32_t)(s >> 32), kSynthTag), a.k0, a.k1);
}
// ((w >> 8) | 1) * 2^-24: in (0, 1) and exact in fp32
__device__ __forceinline__ float uniform(uint32_t w) { return (float)((w >> 8) | 1u) * 0x1p-24f; }
__device__ __forceinline__ int grid_index(uint32_t w) { return (int)(((w >> 8) * 7u) >> 24); }

// e^{j 2 pi x} for a turn count x in fp64: the integer turns are removed in fp64, the rest (|r| <= 1/2) goes to sincospif
__device__ __forceinline__ float2 cis_turns(double x) {
  const double r = x - rint(x);
  float s, c;
  sincospif((float)(2.0 * r), &s, &c);
  return make_float2(c, s);
}
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}

// One CTA generates one sample at a time (grid-stride over samples).  Shared memory: the taps (turns per subcarrier
// tau * df, Doppler nu, complex amplitude), the Doppler factors with the amplitudes G[l][t] = a_t e^{j2pi nu_t l Ts}, and
// the frequency factors F[k][t] = e^{-j2pi k df tau_t} of `chunk` subcarriers.  Thread (r, c) of a pass holds G of its V
// symbols in registers and writes V consecutive grid points of rows r, r + rows, ... of the chunk: H = sum_t F[k][t] G[l][t].
// A thread whose point is a pilot position also writes that pilot, so the pilots cost no phase of their own.
template <int V>
__global__ void __launch_bounds__(256, kCtasPerSm)
synth_kernel(const SynthArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  double* fturn = reinterpret_cast<double*>(smem);                     // [8]
  double* nu = fturn + kTaps;                                          // [8]
  float2* amp = reinterpret_cast<float2*>(nu + kTaps);                 // [8]
  float* cond = reinterpret_cast<float*>(amp + kTaps);                 // snr, sigma (+ pad to 16 bytes)
  float2* G = reinterpret_cast<float2*>(cond + 4);                     // [num_symbols][8]
  float2* F = G + (size_t)a.num_symbols * kTaps;                       // [chunk][8]
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int P = a.pilot_scs * a.pilot_symbols;
  const int col = tid % a.cols, row = tid / a.cols;

  for (int64_t i = blockIdx.x; i < a.batch; i += gridDim.x) {
    const uint64_t s = (uint64_t)(a.sample0 + i);
    // ---- draw 0: the condition; draws 1..8: the taps
    if (tid < kTaps) {
      float snr, ds, dop;
      if (a.draw) {
        const uint4 w = draw(a, s, 0);
        snr = 5.f * grid_index(w.x);
        ds = 50.f * (grid_index(w.y) + 1);
        dop = 200.f * (grid_index(w.z) + 1);
        if (tid == 0) { a.snr[i] = snr; a.ds[i] = ds; a.dop[i] = dop; }
      } else {
        snr = a.snr[i]; ds = a.ds[i]; dop = a.dop[i];
      }
      const uint4 w = draw(a, s, 1 + tid);
      const float u_tau = uniform(w.x), u_ph = uniform(w.y), u_dop = uniform(w.z);
      const double tau = -(double)ds * 1e-9 * log((double)u_tau);
      // p_t = exp(-tau_t / ds) / sum = u_t / sum
      float sum = u_tau;
      sum += __shfl_xor_sync(0xffu, sum, 1);
      sum += __shfl_xor_sync(0xffu, sum, 2);
      sum += __shfl_xor_sync(0xffu, sum, 4);
      float sp, cp;
      sincospif(2.f * u_ph, &sp, &cp);
      const float m = sqrtf(u_tau / sum);
      fturn[tid] = kSubcarrierHz * tau;
      nu[tid] = (double)dop * cospi(2.0 * (double)u_dop);
      amp[tid] = make_float2(m * cp, m * sp);
      if (tid == 0) { cond[0] = snr; cond[1] = (float)exp10(-(double)snr / 20.0); }
    }
    __syncthreads();
    // ---- Doppler factors
    for (int e = tid; e < a.num_symbols * kTaps; e += nthr) {
      const int l = e >> 3, t = e & 7;
      G[e] = cmul(amp[t], cis_turns(nu[t] * ((double)l * kSymbolSec)));
    }
    // ---- the grid, `chunk` subcarriers at a time
    float2 g[V][kTaps];
    for (int k0 = 0; k0 < a.num_scs; k0 += a.chunk) {
      const int kc = min(a.chunk, a.num_scs - k0);
      __syncthreads();                      // G written (first chunk); F of the previous chunk consumed
      for (int e = tid; e < kc * kTaps; e += nthr) F[e] = cis_turns(-(double)(k0 + (e >> 3)) * fturn[e & 7]);
      __syncthreads();
      if (k0 == 0) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float4* g4 = reinterpret_cast<const float4*>(G + (size_t)(col * V + v) * kTaps);
#pragma unroll
          for (int t2 = 0; t2 < kTaps / 2; ++t2) {
            const float4 x = g4[t2];
            g[v][2 * t2] = make_float2(x.x, x.y);
            g[v][2 * t2 + 1] = make_float2(x.z, x.w);
          }
        }
      }
      float2* base = a.truth + ((size_t)i * a.num_scs + k0) * a.num_symbols + col * V;
      for (int kk = row; kk < kc; kk += a.rows) {
        const float4* f4 = reinterpret_cast<const float4*>(F + kk * kTaps);
        float2 acc[V];
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] = make_float2(0.f, 0.f);
#pragma unroll
        for (int t2 = 0; t2 < kTaps / 2; ++t2) {
          const float4 x = f4[t2];
          const float2 fa = make_float2(x.x, x.y), fb = make_float2(x.z, x.w);
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const float2 ga = g[v][2 * t2], gb = g[v][2 * t2 + 1];
            acc[v].x = fmaf(fa.x, ga.x, acc[v].x); acc[v].x = fmaf(-fa.y, ga.y, acc[v].x);
            acc[v].y = fmaf(fa.x, ga.y, acc[v].y); acc[v].y = fmaf(fa.y, ga.x, acc[v].y);
            acc[v].x = fmaf(fb.x, gb.x, acc[v].x); acc[v].x = fmaf(-fb.y, gb.y, acc[v].x);
            acc[v].y = fmaf(fb.x, gb.y, acc[v].y); acc[v].y = fmaf(fb.y, gb.x, acc[v].y);
          }
        }
        float2* dst = base + (size_t)kk * a.num_symbols;
        if constexpr (V == 2) {
          *reinterpret_cast<float4*>(dst) = make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y);
        } else {
          *dst = acc[0];
        }
        // pilot (ip, m) = this grid point + CN(0, sigma^2) from draw 9 + p / 2, p = ip * pilot_symbols + m
        const int k = k0 + kk, ip = k / a.pilot_step;
        if (ip * a.pilot_step == k && ip < a.pilot_scs) {
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const int l = col * V + v;
            const int m = l == 2 ? 0 : (l == 11 && a.pilot_symbols == 2) ? 1 : -1;
            if (m < 0) continue;
            const int p = ip * a.pilot_symbols + m;
            const uint4 w = draw(a, s, 9 + (p >> 1));
            const float u1 = uniform(p & 1 ? w.z : w.x), u2 = uniform(p & 1 ? w.w : w.y);
            const float r = sqrtf(-2.f * logf(u1)) * cond[1] * 0.70710678118654752f;
            float sn, cn;
            sincospif(2.f * u2, &sn, &cn);
            a.pilots[i * P + p] = make_float2(acc[v].x + r * cn, acc[v].y + r * sn);
          }
        }
      }
    }
    __syncthreads();                        // the taps of this sample are read until here
  }
}

template <int V>
bool launch_synth_v(SynthArgs a, cudaStream_t st) {
  a.cols = a.num_symbols / V;
  a.rows = 256 / a.cols;                     // num_symbols <= 256 (aft_synthetic_channels): 1 <= rows, threads <= 256
  const int threads = a.cols * a.rows;
  a.chunk = max(4 * a.rows, (threads + kTaps - 1) / kTaps);
  // under the 48 KB default: G is at most 16 KB (num_symbols <= 256), F at most 32 KB (chunk 512 at num_symbols 4)
  const size_t smem = kTaps * (2 * sizeof(double) + sizeof(float2)) + 4 * sizeof(float) +
                      (size_t)(a.num_symbols + a.chunk) * kTaps * sizeof(float2);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t blocks = a.batch < (int64_t)sms * kCtasPerSm ? a.batch : (int64_t)sms * kCtasPerSm;
  synth_kernel<V><<<(unsigned)blocks, threads, smem, st>>>(a);
  count_launch();
  return check_launch("synth_kernel");
}

}  // namespace

bool launch_synthetic_channels(const AftConfig& cfg, uint64_t seed, int64_t sample0, int64_t batch, float* snr, float* ds,
                               float* dop, bool draw_conditions, float2* pilots, float2* truth, cudaStream_t st) {
  SynthArgs a{};
  a.num_scs = cfg.num_scs; a.num_symbols = cfg.num_symbols;
  a.pilot_scs = cfg.pilot_scs; a.pilot_symbols = cfg.pilot_symbols;
  a.pilot_step = cfg.num_scs / cfg.pilot_scs;
  a.k0 = (uint32_t)seed; a.k1 = (uint32_t)(seed >> 32);
  a.sample0 = sample0; a.batch = batch;
  a.snr = snr; a.ds = ds; a.dop = dop; a.draw = draw_conditions ? 1 : 0;
  a.pilots = pilots; a.truth = truth;
  const bool vec16 = cfg.num_symbols % 2 == 0 && (reinterpret_cast<uintptr_t>(truth) & 15) == 0;
  return vec16 ? launch_synth_v<2>(a, st) : launch_synth_v<1>(a, st);
}

}  // namespace aft
