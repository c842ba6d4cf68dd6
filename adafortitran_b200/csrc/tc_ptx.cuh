// Thin inline-PTX wrappers for the sm_100a features the bf16 path is built on:
// mbarrier, cp.async.bulk (TMA 1-D bulk copies), tcgen05 (TMEM alloc / mma / commit / ld / st / fences).
// Descriptor bit layouts follow the PTX ISA "tcgen05 shared memory descriptor" / "instruction descriptor"
// tables (same encodings as cute/arch/mma_sm100_desc.hpp, consulted for the field positions only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace aft {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes));
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Diagnostics channel: device pointer to mapped host memory (survives a trapped kernel), set by the host.
// Record layout: slot [block % 64][warp % 16] = 1<<63 | block<<40 | thread<<24 | parity<<16 | (barrier smem address & 0xFFFF).
__device__ unsigned long long* g_wait_diag = nullptr;

// Bounded wait: a protocol bug must surface as a trap (reported as a CUDA error), never as a hung GPU.  The first
// threads to time out leave a record and keep waiting a little so that every stuck role gets to report.
__device__ __forceinline__ void mbar_wait_timeout(uint32_t bar, uint32_t parity) {
  if (g_wait_diag != nullptr)
    g_wait_diag[(blockIdx.x & 63) * 16 + ((threadIdx.x >> 5) & 15)] =
        (1ull << 63) | ((unsigned long long)blockIdx.x << 40) | ((unsigned long long)threadIdx.x << 24) |
        ((unsigned long long)parity << 16) | (bar & 0xFFFFu);
  __threadfence_system();
}
// -DAFT_TC_CHAOS: every wait is preceded by a pseudo-random, warp-uniform delay of up to ~8 us for one call in four.
// Shakes the relative timing of the roles (MMA issuer, producer, compute warps); a protocol that relies on timing rather
// than on its barriers then hangs into the bounded wait below and is reported by the wait-timeout diagnostics.
__device__ __forceinline__ void chaos_delay() {
#ifdef AFT_TC_CHAOS
  uint32_t c;
  asm volatile("mov.u32 %0, %%clock;" : "=r"(c));
  c = __shfl_sync(0xFFFFFFFFu, c, 0);
  const uint32_t h = (c ^ ((threadIdx.x >> 5) * 0x9E3779B9u) ^ (blockIdx.x * 0x85EBCA6Bu)) * 2654435761u;
  if (((h >> 28) & 3) == 0) __nanosleep((h >> 8) & 0x1FFF);
#endif
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or the hint (ns) expires.
// The plain form returns after a short, implementation-defined time; in a kernel whose roles wait most of the time the
// resulting poll loops were a quarter of all issued instructions and competed with the working warps of their
// sub-partition for issue slots (ncu: 12 % of the warp samples "not selected").
__device__ __forceinline__ bool mbar_try_wait_for(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#ifndef AFT_TC_WAIT_HINT_NS
#define AFT_TC_WAIT_HINT_NS 100000u     // suspend hint of one try_wait (100 us)
#endif
// Time budget of one wait (wall clock, not poll counts: under compute-sanitizer, a debugger or time slicing a legitimate
// wait can take arbitrarily many polls).  The chaos build injects up to ~8 us per wait on purpose.
constexpr unsigned long long kWaitReportNs = 4000000000ull, kWaitTrapNs = 6000000000ull;
// slow path (rare: the first try_wait already sleeps up to the hint): poll with the hint, watch the wall clock
__device__ __forceinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  const unsigned long long t0 = global_timer_ns();
  bool reported = false;
  while (!mbar_try_wait_for(bar, parity, AFT_TC_WAIT_HINT_NS)) {
    const unsigned long long dt = global_timer_ns() - t0;
    if (!reported && dt > kWaitReportNs) { mbar_wait_timeout(bar, parity); reported = true; }
    if (dt > kWaitTrapNs) __trap();
  }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  chaos_delay();
  if (!mbar_try_wait_for(bar, parity, AFT_TC_WAIT_HINT_NS)) mbar_wait_slow(bar, parity);
}
// same contract; kept as a separate name for the roles whose waits are not latency critical (producer)
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  if (!mbar_try_wait_for(bar, parity, AFT_TC_WAIT_HINT_NS)) mbar_wait_slow(bar, parity);
}

// ---------------------------------------------------------------------------------------------
// proxies / fences
// ---------------------------------------------------------------------------------------------
// generic-proxy shared-memory writes -> visible to the async proxy (tcgen05.mma / bulk copies)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads));
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads));
}

// ---------------------------------------------------------------------------------------------
// 1-D bulk copy global -> shared, completion on an mbarrier (bytes must be a multiple of 16)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src_gmem), "r"(bytes), "r"(bar)
               : "memory");
}

// L2 prefetch of a global range (bytes a multiple of 16): no destination, no completion tracking
__device__ __forceinline__ void bulk_prefetch_l2(const void* src_gmem, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
// 1-D bulk copy shared -> global (bulk async-group completion)
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(src_smem), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // source may be reused
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }         // writes complete

// ---------------------------------------------------------------------------------------------
// TMEM allocation (whole warp executes)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols));
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols));
}

// ---------------------------------------------------------------------------------------------
// descriptors
// ---------------------------------------------------------------------------------------------
enum : uint32_t { kSwizzleNone = 0, kSwizzle128 = 2, kSwizzle64 = 4, kSwizzle32 = 6 };

// shared-memory matrix descriptor: start address, leading / stride byte offsets (all >> 4), version 1 (Blackwell),
// base offset 0 (operand atoms are aligned to their swizzle repeat), layout type in bits [61,64)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout & 7) << 61;
  return d;
}
// K-major operand, rows of 128 bytes (64 bf16), SWIZZLE_128B: 8-row atoms of 1024 bytes
__device__ __forceinline__ uint64_t desc_k_sw128(uint32_t saddr) { return make_smem_desc(saddr, 16, 1024, kSwizzle128); }
// the same descriptor with a zero start address (constant part)
__host__ __device__ constexpr uint64_t desc_k_sw128_const() {
  return ((uint64_t)(16 >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)kSwizzle128 << 61);
}
// K-major operand, rows of 64 bytes (32 bf16), SWIZZLE_64B: 8-row atoms of 512 bytes
__device__ __forceinline__ uint64_t desc_k_sw64(uint32_t saddr) { return make_smem_desc(saddr, 16, 512, kSwizzle64); }
// MN-major operand, 32 contiguous MN elements (64 bytes) per K row, SWIZZLE_64B: 8 K-rows per 512-byte atom
__device__ __forceinline__ uint64_t desc_mn_sw64(uint32_t saddr) { return make_smem_desc(saddr, 512, 512, kSwizzle64); }

// instruction descriptor for kind::f16 with bf16 operands and fp32 accumulation
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                         // D format: F32
         | (1u << 7)                       // A format: BF16
         | (1u << 10)                      // B format: BF16
         | ((a_mn_major ? 1u : 0u) << 15)  // A major
         | ((b_mn_major ? 1u : 0u) << 16)  // B major
         | ((uint32_t)(N >> 3) << 17)      // N / 8
         | ((uint32_t)(M >> 4) << 24);     // M / 16
}

// ---------------------------------------------------------------------------------------------
// tcgen05.mma (single thread issues), commit
// ---------------------------------------------------------------------------------------------
// D[tmem] (+)= A[smem] . B[smem]^T
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate,
                                       bool elected = true) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate), "r"((uint32_t)elected)
);
}
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate,
                                       bool elected = true) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate), "r"((uint32_t)elected)
);
}
// arrive on an mbarrier when all tcgen05.mma issued so far by this thread have completed
__device__ __forceinline__ void mma_commit(uint32_t bar, bool elected = true) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "setp.ne.b32 e, %1, 0;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar), "r"((uint32_t)elected)
);
}

// ---------------------------------------------------------------------------------------------
// TMEM <-> registers.  32x32b shape: thread i of the warp owns TMEM lane (warp%4)*32 + i and receives N
// consecutive 32-bit columns.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
);
}
// pointer forms (r[0..N) must be compile-time resolvable after inlining so the values stay in registers)
__device__ __forceinline__ void tmem_ld16p(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8p(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
);
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;"); }

}  // namespace ptx
}  // namespace aft
