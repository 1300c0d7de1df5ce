// Thin inline-PTX wrappers for the Blackwell tensor-core path (sm_100a):
// tcgen05.mma with shared-memory operand descriptors, TMEM allocation / loads,
// mbarriers and the bulk-copy (TMA, 1-D) engine.
//
// Operand layout used throughout this library: K-major, NO swizzle ("interleave").
// A tile is a set of 8x16-byte "core matrices": 8 consecutive rows (M or N index)
// of 8 16-bit elements (16 bytes) each, rows 16 bytes apart.  The descriptor carries
//   SBO = byte distance between consecutive 8-row groups        (M/N direction)
//   LBO = byte distance between consecutive 16-byte K chunks    (K direction)
// and a start address that only needs 16-byte alignment, which is what lets a
// 3x3 convolution tap be expressed as "the same activation tile, start address
// moved by (dy*pitch + dx) rows" (conv.cu).
#pragma once
#include <cstdint>
#include <cuda_bf16.h>

namespace mz {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ---------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
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
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- CTA pairs (2-CTA clusters, tcgen05 .cta_group::2) ------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// every thread of both CTAs; orders each CTA's earlier shared-memory writes (barrier inits included) before the
// peer's later accesses
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the wait of a barrier that also receives arrivals from the peer CTA: acquire at cluster scope
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster; release at cluster scope makes
// everything this thread has observed (a completed local barrier phase included) visible to the peer's acquire
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
}
// the same without release semantics (no MEMBAR): forwards the completion of a barrier whose only payload is
// bulk-copy bytes in the forwarding CTA's own shared memory (conv.cu, w_full of SM-pair launches)
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint64_t* bar, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
}
// 16 bytes at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ uint4 ld_shared_peer_v4(const void* p, uint32_t cta) {
  uint32_t r;
  uint4 v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(cta));
  asm volatile("ld.shared::cluster.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(r) : "memory");
  return v;
}

// ---- proxies / fences ---------------------------------------------------------
// generic-proxy writes to smem (st.shared) -> visible to the async proxy (tcgen05.mma, TMA)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM ---------------------------------------------------------------------
// whole warp; ncols power of two >= 32; the base address lands in *smem_dst
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// CTA-pair forms: one warp in EACH CTA of the pair
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane (base lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- descriptors ----------------------------------------------------------------
// shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor):
//   [0,14) start>>4   [16,30) LBO>>4   [32,46) SBO>>4   [46,48) version=1   [61,64) layout=0
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}
// instruction descriptor for kind::f16, BF16 x BF16 -> FP32, both operands K-major
// (cute::UMMA::InstrDescriptor): c_format[4,6)=1 a_format[7,10)=1 b_format[10,13)=1 n>>3 [17,23) m>>4 [24,29)
__host__ __device__ constexpr uint32_t instr_desc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// same with FP16 x FP16 operands (a_format = b_format = 0)
__host__ __device__ constexpr uint32_t instr_desc_f16(uint32_t M, uint32_t N) {
  return (1u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The same, executed by a WHOLE converged warp: one lane is elected inside the asm statement.  With the
// election here (instead of an `if (lane == 0)` around mma_f16) ptxas emits a predicated UTCHMMA with no
// per-MMA convergence loop (ELECT / R2UR.BROADCAST / BRA.U.ANY), which otherwise costs ~100 cycles per MMA
// on the single issuing warp -- more than the 64 cycles an M128 N128 K16 MMA lasts.
__device__ __forceinline__ void mma_f16_elect(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with the disable-output-lane vector: bit j of word i keeps TMEM lane 32*i + j (row 32*i + j of D) from
// being written by this MMA.  conv3x3 uses it to drop, per tap, the output rows whose neighbour lies across a board edge
// (halo-free activation layout).
__device__ __forceinline__ void mma_f16_elect_masked(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                     uint32_t accumulate, uint32_t m0, uint32_t m1, uint32_t m2,
                                                     uint32_t m3) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
      : "memory");
}
// four K-steps under ONE election: ptxas moves every register operand of an elected tcgen05.mma into uniform
// registers (R2UR.BROADCAST) once per asm statement, so issuing the four MMAs of a 64-channel weight stage from one
// statement pays for the election, the accumulator address, the instruction descriptor and the lane masks once
// instead of four times (the issue loop, not the tensor pipe, bounds the halo-free conv kernel: 158 cycles per MMA
// and warp measured against the 128 the pipe needs).
__device__ __forceinline__ void mma4_f16_elect_masked(uint32_t d_tmem, uint64_t a0, uint64_t a1, uint64_t a2, uint64_t a3,
                                                      uint64_t b0, uint64_t b1, uint64_t b2, uint64_t b3, uint32_t idesc,
                                                      uint32_t accumulate, uint32_t m0, uint32_t m1, uint32_t m2,
                                                      uint32_t m3) {
  asm volatile(
      "{\n\t.reg .pred p, q, t;\n\t"
      "setp.ne.b32 p, %10, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %5, %9, {%11, %12, %13, %14}, p;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %2, %6, %9, {%11, %12, %13, %14}, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %3, %7, %9, {%11, %12, %13, %14}, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %4, %8, %9, {%11, %12, %13, %14}, t;\n\t}"
      ::"r"(d_tmem), "l"(a0), "l"(a1), "l"(a2), "l"(a3), "l"(b0), "l"(b1), "l"(b2), "l"(b3), "r"(idesc),
        "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
      : "memory");
}
// the same without lane masks (training kernels: padded grid, every tap unmasked)
__device__ __forceinline__ void mma4_f16_elect(uint32_t d_tmem, uint64_t a0, uint64_t a1, uint64_t a2, uint64_t a3, uint64_t b0,
                                               uint64_t b1, uint64_t b2, uint64_t b3, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q, t;\n\t"
      "setp.ne.b32 p, %10, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %5, %9, p;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %2, %6, %9, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %3, %7, %9, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %4, %8, %9, t;\n\t}"
      ::"r"(d_tmem), "l"(a0), "l"(a1), "l"(a2), "l"(a3), "l"(b0), "l"(b1), "l"(b2), "l"(b3), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The SM-pair form (cta_group::2, M = 256, issued by the even CTA of a 2-CTA cluster only): rows 0-127 of D are
// the issuing CTA's, rows 128-255 the peer's, each in its own TMEM at d_tmem; each CTA supplies its 128 rows of A and
// half of the N rows of B from its own shared memory at the descriptors' addresses.  Mask words 0-3 are the issuing
// CTA's TMEM lanes, words 4-7 the peer's.
__device__ __forceinline__ void mma4_f16_pair_elect_masked(uint32_t d_tmem, uint64_t a0, uint64_t a1, uint64_t a2,
                                                           uint64_t a3, uint64_t b0, uint64_t b1, uint64_t b2, uint64_t b3,
                                                           uint32_t idesc, uint32_t accumulate, const uint4& m,
                                                           const uint4& n) {
  asm volatile(
      "{\n\t.reg .pred p, q, t;\n\t"
      "setp.ne.b32 p, %10, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %5, %9, {%11, %12, %13, %14, %15, %16, %17, %18}, p;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %2, %6, %9, {%11, %12, %13, %14, %15, %16, %17, %18}, t;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %3, %7, %9, {%11, %12, %13, %14, %15, %16, %17, %18}, t;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %4, %8, %9, {%11, %12, %13, %14, %15, %16, %17, %18}, t;\n\t}"
      ::"r"(d_tmem), "l"(a0), "l"(a1), "l"(a2), "l"(a3), "l"(b0), "l"(b1), "l"(b2), "l"(b3), "r"(idesc),
        "r"(accumulate), "r"(m.x), "r"(m.y), "r"(m.z), "r"(m.w), "r"(n.x), "r"(n.y), "r"(n.z), "r"(n.w)
      : "memory");
}
// arrive on `bar` in BOTH CTAs of the pair once every MMA this thread issued before has completed
__device__ __forceinline__ void commit_pair_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}" ::"r"(
          smem_u32(bar)), "h"((unsigned short)3)
      : "memory");
}
__device__ __forceinline__ void commit_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
      : "memory");
}
// arrive on `bar` once every previously issued MMA has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- bulk copy (TMA, 1-D): global -> shared, completion on an mbarrier -----------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void bulk_g2s_u32(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

}  // namespace umma
}  // namespace mz
