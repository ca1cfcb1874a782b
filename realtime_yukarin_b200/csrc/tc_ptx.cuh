// tc_ptx.cuh -- inline-PTX wrappers shared by the tcgen05 convolution kernels (conv_tc.cu: one CTA per tile;
// conv_tc3.cu: persistent halo kernel): mbarriers, TMA loads, UMMA issue / commit, smem descriptors, PDL.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace ryk {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;          // fp16 elements = 128 bytes = one swizzle row
constexpr int kUmmaK = 16;
constexpr int kTcThreads = 192;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Programmatic dependent launch: every kernel of a U-Net forward is a dependent of the one before it in the stream.
// pdl_trigger() lets the NEXT kernel's CTAs be scheduled as soon as all CTAs of this grid have started (they run their
// prologue -- barrier init, TMEM allocation, tensor-map prefetch, scale/shift staging -- in the shadow of this grid's
// tail); pdl_wait() blocks until the PREVIOUS grid has completed and its memory is visible, and must precede every
// access to activations / workspaces.  Both are no-ops for launches without the programmatic attribute.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// One elected lane of a fully active warp.  The TMA / MMA issuing warps run their loops WARP-UNIFORMLY (all 32 lanes compute the same
// coordinates and descriptors) and guard only the issuing instruction with elect_one(): ptxas then keeps the operands in uniform
// registers.  Issuing from an `if (lane == 0)` region instead makes it wrap EVERY UTCHMMA / UTMALDG in an ELECT + 5 x R2UR.BROADCAST +
// BRA.U.ANY loop (~100 clocks per instruction: the tensor pipe then runs at ~60 % behind its issuer -- profiles/r02_halo_timeline.txt).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// rank of this CTA in its thread-block cluster
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }

// K-major, 128B-swizzled operand: 8-row atoms of 1024 B (SBO), LBO unused, descriptor version 1 (sm_100)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((1024u >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}


}  // namespace ryk
