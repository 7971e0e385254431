// sm_100a PTX wrappers used by the HyperNeRF hot-path kernels: mbarrier, bulk async copy (TMA 1-D),
// tcgen05 (UMMA / TMEM) and the proxy fences between them.  Nothing here is generic: every wrapper is
// the exact instruction form the kernels in this directory issue.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdio.h>
#include <stdint.h>

namespace hn {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin on try_wait (itself a bounded hardware sleep).  HN_WATCHDOG bounds the spin so a protocol bug
// traps instead of hanging the GPU box.
#ifndef HN_WATCHDOG
#define HN_WATCHDOG 1
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#if HN_WATCHDOG
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      printf("hn: mbarrier watchdog block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
#else
  while (!mbar_try_wait(bar, parity)) {
  }
#endif
}

// generic-proxy writes (st.shared) -> visible to the async proxy (UMMA / bulk copy reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// bulk async copy global -> shared (1-D TMA, no tensor map), completion on an mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// bulk async copy shared -> global (bulk group completion)
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------------------------
// TMEM allocation (one warp, .sync.aligned)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// UMMA descriptors.  Field layout per cute/arch/mma_sm100_desc.hpp (SmemDescriptor / InstrDescriptor).
// All operand tiles in this project use the un-swizzled "interleave" canonical layout:
//   core matrix = 8 (rows) x 16 bytes, 128 contiguous bytes
//   K-major  operand: rows = M/N index, 16 B = 8 K elements; LBO = byte stride between the two K chunks
//                     of one K=16 instruction, SBO = byte stride between 8-row groups
//   MN-major operand: 16 B = 8 consecutive M/N elements, rows = K index; LBO = byte stride between 8-row
//                     K groups, SBO = byte stride between groups of 8 M/N elements
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (sm_100)
  // base_offset = 0, lbo_mode = 0, layout_type = 0 (SWIZZLE_NONE)
  return d;
}
// kind::f16, bf16 x bf16 -> fp32.  a_major / b_major: 0 = K-major, 1 = MN-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_major, uint32_t b_major) {
  return (1u << 4)                 // c_format = F32
         | (1u << 7)               // a_format = BF16
         | (1u << 10)              // b_format = BF16
         | (a_major << 15) | (b_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; one thread issues.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued UMMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- CTA-pair (cta_group::2) forms: one UMMA spans the two CTAs of a cluster (M = 256: 128 rows per CTA, each CTA
// supplying its own A rows and N/2 rows of B from the SAME shared-memory offsets; cute/atom/mma_traits_sm100.hpp,
// SM100_MMA_F16BF16_2x1SM_SS).  Issued by the leader CTA (cluster rank 0) only.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at the same shared-memory offset in every CTA of `cta_mask` when all previously issued
// UMMAs of this thread have completed
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
// TMEM -> registers: 32 lanes x 32 bit, N consecutive columns per thread (thread t <- lane base+t)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// One elected lane of a CONVERGED warp.  The UMMA issuer must run its loop with all 32 lanes (warp-uniform control
// flow and operands) and guard only the tcgen05 instructions with this predicate: ptxas then keeps descriptors in
// uniform registers.  Issuing from a divergent `if (lane == 0)` region makes it wrap every UTCHMMA in an
// ELECT/BRA.U.ANY loop fed by R2UR moves (~240 cycles per instruction, measured with profiles/umma_rate.py).
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xFFFFFFFF;\n\t"
      "@px mov.s32 %0, 1;\n\t}"
      : "+r"(pred));
  return pred;
}

// register re-balancing between warpgroups (all 4 warps of the warpgroup execute it)
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
#ifndef HN_NO_SETMAXNREG
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
#endif
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
#ifndef HN_NO_SETMAXNREG
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
#endif
}

// pack two fp32 -> bf16x2 (lo = a, hi = b), round-to-nearest-even
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t pack_bf16_relu(float a, float b) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// ReLU gate words.  The forward epilogue records, per row and per block of 32 output columns, the SIGN bits of the 32
// fp32 pre-activations (sign set <=> ReLU closed; relu(+0) = 0 either way): even columns 0,2,..,30 in bits 15..0
// (column 2j at bit 15-j), odd columns 1,3,..,31 in bits 31..16 (column 2j+1 at bit 31-j).  gate_push shifts one sign
// in with a single funnel shift; after 16 pushes per half the word is complete.  The data gradient masks the packed
// bf16 pair j with gate_pair_mask: (w << j) puts the pair's signs at bits 15 and 31, PRMT (selector nibble 8|b =
// "replicate the top bit of byte b") widens them to halfword masks of the CLOSED gates.
__device__ __forceinline__ uint32_t gate_push(uint32_t acc, float v) { return __funnelshift_l(__float_as_uint(v), acc, 1); }
__device__ __forceinline__ uint32_t gate_word_of(uint32_t even_bits, uint32_t odd_bits) { return __byte_perm(even_bits, odd_bits, 0x5410); }
template <int J>
__device__ __forceinline__ uint32_t gate_pair_closed(uint32_t w) {
  uint32_t m;
  asm("prmt.b32 %0, %1, %1, 0xBB99;" : "=r"(m) : "r"(w << J));
  return m;
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

// 16-byte vector reduction into global memory (sm_90+): four fp32 adds in one L2 transaction
__device__ __forceinline__ void red_add_v4(float* addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(__uint_as_float(a)),
               "f"(__uint_as_float(b)), "f"(__uint_as_float(c)), "f"(__uint_as_float(d))
               : "memory");
}

}  // namespace hn
