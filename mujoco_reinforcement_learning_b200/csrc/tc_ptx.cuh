// The Blackwell (sm_100a) PTX primitives of the tensor-core kernels and the bulk-copy gather, each written once:
// mbarriers, TMA and bulk copies, tcgen05 (TMEM, MMA, fences, descriptors), CTA-pair clusters, and wide or swizzled
// memory accesses.  Operands the instruction takes as immediates (CTA group, TMEM columns, wait-group depths) are
// template parameters, so they stay immediates.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace b200ppo {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarrier ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// makes the initialised barriers visible to the other threads, the async proxy and the peer CTA
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on a barrier of another CTA of the cluster (address from mapa_u32).  Relaxed: no release fence in front of it
// (a release is a MEMBAR.ALL.GPU); callers order their shared-memory writes with fence_proxy_async_smem() first.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}

// ---- TMA and bulk copies -------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// TMA load whose completion bytes are counted on an mbarrier of the pair's leader CTA (shared::cluster address)
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
// shared -> global through a tensor map (rows and columns outside the tensor are clipped); joins the bulk group
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
// plain bulk copy global -> this CTA's shared memory (shared address dst), bytes counted on a local mbarrier (16-byte
// granules)
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
// plain bulk copy shared (shared address src) -> global; joins the bulk group
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N bulk groups of this thread still pending
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// at most N bulk groups of this thread still reading their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (bulk copies, tensor-core operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 -----------------------------------------------------------------------------------------------------
// allocate COLS TMEM columns (a power of two >= 32) for CTA group CG, address written to *slot; one warp calls it
template <int CG, uint32_t COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::%2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS), "n"(CG) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::%0.sync.aligned;" ::"n"(CG) : "memory");
}
template <int CG, uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::%2.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS), "n"(CG) : "memory");
}
// order tcgen05 operations before / after a thread synchronisation (barrier, mbarrier arrive or wait)
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 64-bit shared-memory matrix descriptor (sm_100): 128-byte swizzle, version 1.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3FFFF) >> 4);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= uint64_t(1) << 46;  // descriptor version (Blackwell)
  d |= uint64_t(2) << 61;  // SWIZZLE_128B
  return d;
}
// 32-bit instruction descriptor of kind::f16: D fp32, A and B bf16 (f16: fp16), the operands' majors, N >> 3, M >> 4
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, bool a_mn_major, bool b_mn_major, bool f16 = false) {
  const uint32_t fmt = f16 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (uint32_t(a_mn_major) << 15) | (uint32_t(b_mn_major) << 16) | (uint32_t(N >> 3) << 17) |
         (uint32_t(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma2_commit(uint64_t* bar) {  // arrives on the barrier at this offset in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(uint16_t(3))
               : "memory");
}
// 32x32b loads: this thread's TMEM lane, 8 / 16 consecutive columns.  The _nowait form leaves the wait to the caller.
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
  tmem_ld_wait();
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  tmem_ld16_nowait(taddr, v);
  tmem_ld_wait();
}

// ---- clusters (CTA pairs) -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// this CTA's shared-memory address -> the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- wide and swizzled accesses ------------------------------------------------------------------------------------
// 256-bit global accesses: one full 32-byte sector per thread
__device__ __forceinline__ void ldg256(const void* p, uint32_t (&r)[8]) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p));
}
__device__ __forceinline__ void ldg256_na(const void* p, uint32_t (&r)[8]) {  // coherent 256-bit load that does not linger in L1
  asm volatile("ld.global.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p)
               : "memory");
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&r)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]),
               "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// 16 bf16 (8 words) <-> the 16-byte units 2s and 2s + 1 of a 128-byte shared-memory row whose units are XOR-swizzled by
// sw (row & 7): the layout of the 128-byte-swizzle TMA boxes and tcgen05 operands
__device__ __forceinline__ void sts_unit_pair(uint32_t row, uint32_t sw, int s, const uint32_t (&o)[8]) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row + (((2 * s) ^ sw) << 4)), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row + (((2 * s + 1) ^ sw) << 4)), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
}
__device__ __forceinline__ void lds_unit_pair(uint32_t row, uint32_t sw, int s, uint32_t (&h)[8]) {
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(h[0]), "=r"(h[1]), "=r"(h[2]), "=r"(h[3]) : "r"(row + (((2 * s) ^ sw) << 4)) : "memory");
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(h[4]), "=r"(h[5]), "=r"(h[6]), "=r"(h[7]) : "r"(row + (((2 * s + 1) ^ sw) << 4)) : "memory");
}

}  // namespace b200ppo
