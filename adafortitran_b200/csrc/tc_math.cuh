// Device helpers shared by the tcgen05 kernels (tc_encoder.cu, tc_long.cu): fast exponentials / GELU, packed fp32x2
// arithmetic (FADD2 / FMUL2 / FFMA2 of sm_100), shared-memory vector accesses, batched TMEM loads.
#pragma once

#include "tc_layout.cuh"
#include "tc_ptx.cuh"

namespace aft {
namespace tcm {

using namespace ptx;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exp2 for x <= 0 on the FMA / ALU pipes (no MUFU): Cody-Waite split x = n + f, |f| <= 0.5 by the 1.5 * 2^23 rounding trick,
// cubic minimax for 2^f (max rel. error 1.9e-4, 20x below the bf16 rounding of P), 2^n added straight into the exponent
// field ((bits(t) << 23) == (n << 23) because the low 9 bits of the magic constant are zero).
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -126.0f);
  const float t = x + 12582912.0f;
  const float f = x - (t - 12582912.0f);
  float p = fmaf(f, 0.05322283f, 0.2424649f);
  p = fmaf(p, f, 0.69373846f);
  p = fmaf(p, f, 1.0f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Packed fp32 pairs (FADD2 / FMUL2 / FFMA2 of sm_100): half the issue slots of the scalar forms, same rounding per lane.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
// 2^x for a pair of x <= 0 on the FMA / ALU pipes: x = n + f with |f| <= 0.5 by the 1.5 * 2^23 rounding trick, cubic minimax
// for 2^f (max relative error 1.9e-4, ten times below the bf16 rounding of P), n added into the exponent field.
__device__ __forceinline__ f32x2 ex2_poly2(f32x2 x2) {
  float a, b;
  unpack2(x2, a, b);
  const f32x2 xc = pack2(fmaxf(a, -126.0f), fmaxf(b, -126.0f));
  const f32x2 t2 = add2(xc, pack2(12582912.0f, 12582912.0f));
  const f32x2 nr = fma2(t2, pack2(-1.0f, -1.0f), pack2(12582912.0f, 12582912.0f));   // -(t - magic) = -n
  const f32x2 f2 = add2(xc, nr);
  f32x2 p2 = fma2(f2, pack2(0.05322283f, 0.05322283f), pack2(0.2424649f, 0.2424649f));
  p2 = fma2(p2, f2, pack2(0.69373846f, 0.69373846f));
  p2 = fma2(p2, f2, pack2(1.0f, 1.0f));
  float pa, pb, ta, tb;
  unpack2(p2, pa, pb);
  unpack2(t2, ta, tb);
  return pack2(__int_as_float(__float_as_int(pa) + (__float_as_int(ta) << 23)), __int_as_float(__float_as_int(pb) + (__float_as_int(tb) << 23)));
}
__device__ __forceinline__ f32x2 bf16x2_to_f32x2(uint32_t w) { return pack2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u)); }
__device__ __forceinline__ uint32_t pack_bf16_pair(f32x2 v) {
  float lo, hi;
  unpack2(v, lo, hi);
  return pack_bf16x2(lo, hi);
}
// GELU(x) = x Phi(x) with Phi(x) ~ 0.5 (1 + tanh(x (a + b x^2 + c x^4))), coefficients fitted to the erf form
// (max |error| 2.5e-5 over the real line, plus the 2^-11 relative error of MUFU.TANH: |x| 2.4e-4 at most, i.e. at or
// below the bf16 rounding of the hidden activations it feeds).  One MUFU per element; the arithmetic around it is packed fp32x2 (a pair of elements per call).
__device__ __forceinline__ f32x2 gelu_tanh2(f32x2 x) {
  const f32x2 x2 = mul2(x, x);
  const f32x2 u = mul2(x, fma2(x2, fma2(x2, pack2(-3.51516789e-4f, -3.51516789e-4f), pack2(3.70056460e-2f, 3.70056460e-2f)),
                               pack2(7.97507884e-1f, 7.97507884e-1f)));
  float ua, ub, ta, tb;
  unpack2(u, ua, ub);
  asm("tanh.approx.f32 %0, %1;" : "=f"(ta) : "f"(ua));
  asm("tanh.approx.f32 %0, %1;" : "=f"(tb) : "f"(ub));
  const f32x2 hx = mul2(x, pack2(0.5f, 0.5f));
  return fma2(hx, pack2(ta, tb), hx);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d));
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void st_shared_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v));
}
__device__ __forceinline__ float ld_shared_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// one arrival per compute warp: every lane has fenced its own TMEM / shared-memory accesses before calling
__device__ __forceinline__ void warp_arrive(uint32_t bar, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
}

// n consecutive accumulator columns (n a multiple of 8) -> registers, without waiting
template <int N>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t (&x)[N]) {
  static_assert(N % 8 == 0, "column count must be a multiple of 8");
#pragma unroll
  for (int i = 0; i < N / 16; ++i) tmem_ld16p(taddr + i * 16, x + i * 16);
  if (N % 16) tmem_ld8p(taddr + (N / 16) * 16, x + (N / 16) * 16);
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {   // 16-byte shared load of 4 floats (epilogue vectors)
  const uint4 v = ld_shared_v4(addr);
  return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

}  // namespace tcm
}  // namespace aft
