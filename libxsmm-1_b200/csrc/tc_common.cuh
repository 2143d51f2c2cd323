// tcgen05 / TMEM helpers shared by the tensor-core kernels (sm_100a inline PTX).
#pragma once
#include "ptx.cuh"

namespace xb {

__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type)
{
  // reference for the field layout: CUTLASS cute/arch/mma_sm100_desc.hpp (SmemDescriptor)
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;        // descriptor version (Blackwell)
  d |= (uint64_t)layout_type << 61;   // 2 = SWIZZLE_128B, 1 = SWIZZLE_128B_BASE32B
  return d;
}

__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t.reg .pred p;\n\t"
    "setp.ne.b32 p, %4, 0;\n\t"
    "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
    ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar)
{
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32])
{
  asm volatile(
    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
      "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
      "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
    : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}


__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16])
{
  asm volatile(
    "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
    : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// eight columns, no wait: several loads can be in flight before one tc_wait_ld(); tc_pin8() after the wait ties the registers to it
__device__ __forceinline__ void tc_ld8_nowait(uint32_t taddr, uint32_t (&r)[8])
{
  asm volatile(
    "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
    : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void tc_pin8(uint32_t (&r)[8])
{
  asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]) :: "memory");
}

__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t.reg .pred p;\n\t"
    "setp.ne.b32 p, %4, 0;\n\t"
    "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
    ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// ---- CTA pairs (cta_group::2): the two CTAs of a cluster on one TPC share every MMA ---------------------------------
__device__ __forceinline__ uint32_t cluster_rank()
{
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// shared::cluster address of `p` (a shared::cta pointer of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank)
{
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];\n" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity)
{
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  }
}
// TMA load whose completion bytes are counted on a barrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint32_t leader_bar)
{
  asm volatile(
    "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
    ::"r"(smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(leader_bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t.reg .pred p;\n\t"
    "setp.ne.b32 p, %4, 0;\n\t"
    "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
    ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs of the pair once all earlier MMAs have completed
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar)
{
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

// 2:4 structured-sparse A (compressed, common.cuh: xb_sp_*); tmem_e: the tensor-memory column holding the metadata
__device__ __forceinline__ void tc_mma_bf16_sp_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t tmem_e, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t.reg .pred p;\n\t"
    "setp.ne.b32 p, %5, 0;\n\t"
    "tcgen05.mma.sp.cta_group::2.kind::f16 [%0], %1, %2, [%3], %4, p;\n\t}\n"
    ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(tmem_e), "r"(idesc), "r"(accumulate) : "memory");
}
// the same with 8-bit A and B (e4m3 / e5m2, named by the instruction descriptor): K = 64 per instruction, the metadata of
// row r in tensor-memory lane r, two columns per instruction (tools/umma_probe/probe_sp8.cu)
__device__ __forceinline__ void tc_mma_f8_sp_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t tmem_e, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t.reg .pred p;\n\t"
    "setp.ne.b32 p, %5, 0;\n\t"
    "tcgen05.mma.sp.cta_group::2.kind::f8f6f4 [%0], %1, %2, [%3], %4, p;\n\t}\n"
    ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(tmem_e), "r"(idesc), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void tc_mma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t.reg .pred p;\n\t"
    "setp.ne.b32 p, %4, 0;\n\t"
    "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
    ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

}  // namespace xb
