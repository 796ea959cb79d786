// Thin inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / ld / commit / fences).
// Nothing here is generic: bf16 operands, fp32 accumulators, cta_group::1.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ------------------------------------------------- explicit shared-space 16-byte accesses
// (pointers carved out of the dynamic smem block decay to generic addresses; a generic LD/ST is a
// long-scoreboard operation, a LDS/STS is not)
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (try_wait may suspend the thread for a while; a thread that polls several barriers must not be)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> launch error the host reports) instead of hanging the GPU.  The bound
// is wall time (%globaltimer): 4 s, orders of magnitude above any legitimate wait in these kernels.
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
#pragma unroll 1
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 64; ++i)
      if (mbar_try_wait(bar, parity)) return;
    if (globaltimer_ns() - t0 > 4000000000ull) __trap();
  }
}

// ----------------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// 1-D bulk copy global -> shared (bytes a multiple of 16, both addresses 16-byte aligned), completion on an mbarrier
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// TMA store: smem tile (written by generic-proxy stores + fence_proxy_async) -> global, tracked by bulk groups.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// same, source given as a shared-space address
__device__ __forceinline__ void tma_store_2d_s(const CUtensorMap* m, uint32_t saddr, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(saddr), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d_s(const CUtensorMap* m, uint32_t saddr, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(saddr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N of this thread's most recent bulk groups still READING their smem source
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
// generic-proxy smem writes -> visible to the async proxy (TMA store, tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------- warp-uniform issue ("_e": elect one lane inside the wrapper)
// tcgen05.mma / commit / TMA take their operands from UNIFORM registers.  Issued from a `lane == 0` branch the
// operands live in vector registers of divergent code, and ptxas wraps every instruction in a scalarisation loop
// (ELECT + R2UR x4 + BRA.U.ANY): ~150 cycles per MMA whatever its N (measured, profiles/r1b_gemm_roles.md section 3).  With
// the whole warp converged and one lane elected inside the asm block, descriptors stay in uniform registers.
// elect.sync picks the same lane for the same mask every time, so commit / bulk-group tracking stays per thread.
#define TT_ELECT_PRED "elect.sync _|q, 0xffffffff;\n\t"
__device__ __forceinline__ void mbar_arrive_expect_tx_e(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(
                   smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_e(uint64_t* bar) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED "@q mbarrier.arrive.shared::cta.b64 _, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d_e(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(
                   smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d_e(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}" ::"r"(
                   smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_e(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(
                   smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair_e(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1, int c2, int c3) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}" ::"r"(
                   smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_store_2d_e(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n\t}" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit_e() {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED "@q cp.async.bulk.commit_group;\n\t}" ::: "memory");
}
// wait_group is not predicable in one asm block without a branch: the elected lane waits, the others fall through
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED "selp.u32 %0, 1, 0, q;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mma_bf16_e(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p, q;\n\t" TT_ELECT_PRED
               "setp.ne.b32 p, %4, 0;\n\t"
               "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc),
               "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_bf16_pair_e(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p, q;\n\t" TT_ELECT_PRED
               "setp.ne.b32 p, %4, 0;\n\t"
               "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc),
               "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit_e(uint64_t* bar) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mma_commit_pair_e(uint64_t* bar, uint16_t mask) {
  asm volatile("{\n\t.reg .pred q;\n\t" TT_ELECT_PRED
               "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}" ::"r"(
                   smem_u32(bar)), "h"(mask) : "memory");
}

// ------------------------------------------------------------------- tcgen05
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// One full warp allocates `ncols` (power of two >= 32) TMEM columns; base address lands in smem.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------- CTA pairs (cta_group::2)
// Two CTAs of a 2-CTA cluster (one TPC) run one M=256 tcgen05.mma: each CTA stages its own 128 rows
// of A and half of the B rows, the even ("leader") CTA issues the instruction, each CTA's TMEM
// receives its 128 accumulator rows.  Cross-CTA signalling goes through shared::cluster addresses.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem location in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads whose completion bytes are credited to a barrier given as a shared::cluster address
// (the leader CTA's), destination in the executing CTA's smem.
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair_only(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  tmem_alloc_pair_only(smem_dst, ncols);
  tmem_relinquish_pair();
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 per CTA] * B[N rows: N/2 per CTA]^T, issued by the leader CTA.
__device__ __forceinline__ void mma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once all previously issued MMAs completed) on the barrier at this smem offset in every CTA of `mask`.
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// TMEM -> registers: this thread's lane (row), 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// TMEM -> registers, N consecutive fp32 columns of this thread's lane (N = 16 or 32), and the matching
// wait that names the destination registers (see tmem_ld_wait(uint32_t(&)[16]) below).
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&r)[N]);
template <>
__device__ __forceinline__ void tmem_ld<16>(uint32_t taddr, uint32_t (&r)[16]) { tmem_ld16(taddr, r); }
template <>
__device__ __forceinline__ void tmem_ld<32>(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
      "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM: 32 consecutive fp32 columns of this thread's lane (the mirror of tmem_ld<32>); tmem_st_wait()
// before the values may be read back or accumulated on by a later tcgen05.mma (after the usual thread-sync fences).
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
      "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// named barrier `id` over `threads` threads (a multiple of 32) of the CTA
// (barrier.sync without .aligned: the participating warps arrive from different instructions -- the MMA issuer's and the
// row owners' -- and a warp may still be re-converging from an mbarrier spin loop; __syncwarp first keeps it whole)
template <int ID, int THREADS>
__device__ __forceinline__ void named_bar_sync() {
  __syncwarp();
  asm volatile("barrier.sync %0, %1;" ::"n"(ID), "n"(THREADS) : "memory");
}
// Same, but names the destination registers of the outstanding load as in/out operands so the compiler
// cannot schedule a read of them above the wait (the load completes asynchronously).
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// Shared-memory matrix descriptor for a K-major operand tile whose rows are `row_bytes`
// (128 -> SWIZZLE_128B, 64 -> SWIZZLE_64B) wide, 8-row groups `8*row_bytes` apart
// (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout_type [61,64): 2 = SW128, 4 = SW64).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t row_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;                        // LBO (ignored for swizzled K-major)
  d |= static_cast<uint64_t>((8 * row_bytes) >> 4) << 32;     // SBO
  d |= static_cast<uint64_t>(1) << 46;                        // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(row_bytes == 128 ? 2 : 4) << 61; // swizzle mode
  return d;
}
// Same for a SWIZZLE_128B / SWIZZLE_64B K-major tile whose 8-row groups are `sbo_bytes` apart.  Used by the halo convolution:
// a tap's A operand is the staged (TH+2) x 16-pixel tile read at a pixel offset, so the start address is NOT
// 1024-byte aligned.  Measured on B200 (tests/test_gemm_gpu.py::test_conv_halo): the tensor core applies the
// 128B-swizzle XOR to the absolute smem address bits, exactly as TMA wrote the tile, and the descriptor's
// matrix-base-offset field (bits [49,52)) must stay 0 -- setting it to the row offset gives wrong products.
__device__ __forceinline__ uint64_t make_smem_desc_sbo(uint32_t saddr, uint32_t row_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(row_bytes == 128 ? 2 : 4) << 61;
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accum, bf16 A/B, both K-major.
__device__ __forceinline__ uint32_t make_idesc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace ptx
