// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (TMEM
// alloc / UMMA / commit / ld) and the shared-memory + instruction descriptors they consume.
// Everything here is device-only plumbing used by igemm.cu; no reference counterpart (the
// reference delegates all arithmetic to TF 1.13 kernels, SURVEY.md §0).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace bsl {

// Global "something deadlocked" flag. Every bounded spin in the pipeline sets it on timeout and
// every other spin polls it, so a wrong barrier protocol ends the kernel in ~seconds instead of
// hanging the GPU. Host code reads it back after the launch (bsl_ctx keeps a device copy).
struct DeviceStatus {
  int error;      // 0 ok; otherwise a BSL_DEV_* site code
  int block;      // linear block id that raised it
  int site;       // which wait
  int pad;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 %%rx;\n\t"
      ".reg .pred %%px;\n\t"
      "elect.sync %%rx|%%px, %1;\n\t"
      "@%%px mov.s32 %0, 1;\n\t"
      "}\n"
      : "+r"(pred)
      : "r"(0xffffffffu));
  return pred != 0;
}

// ------------------------------------------------------------------- programmatic dependent launch
// A kernel enqueued with cudaLaunchAttributeProgrammaticStreamSerialization (bsl_launch, internal.h) may become
// resident while its predecessor in the stream still runs. pdl_wait() returns once the predecessor grid has completed
// and its writes are visible. Nothing may read or write global data the predecessor touches before pdl_wait().
// It is a no-op in a launch without the attribute. No kernel issues the early trigger (griddepcontrol.launch_dependents):
// it made the training step 0.8-1.0 ms slower on B200 (profiles/r01_ab_experiments.md).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ----------------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}

#ifndef BSL_WAIT_TIMEOUT_NS
#define BSL_WAIT_TIMEOUT_NS 2000000000ull  // 2 s: far beyond any legitimate wait in these kernels
#endif

// Bounded wait. Returns false if the pipeline is (or has been declared) dead.
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, DeviceStatus* st, int site) {
  if (mbar_try_wait(bar, parity)) return true;
  uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (true) {
    if (mbar_try_wait(bar, parity)) return true;
    if ((++spins & 0xff) == 0) {
      if (*reinterpret_cast<volatile int*>(&st->error) != 0) return false;
      if (globaltimer_ns() - t0 > BSL_WAIT_TIMEOUT_NS) {
        if (atomicCAS(&st->error, 0, 1) == 0) {
          st->block = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
          st->site = site;
        }
        return false;
      }
    }
  }
}

// 256-bit global store (sm_100: STG.E.256), 32-byte aligned address.
__device__ __forceinline__ void st_global_v8(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t e,
                                             uint32_t f, uint32_t g, uint32_t h) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d), "r"(e),
               "r"(f), "r"(g), "r"(h)
               : "memory");
}

// ----------------------------------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0,
                                            int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
      "r"(c4)
      : "memory");
}

// TMA store of a shared-memory tile (written in the tensor map's swizzle) into a 4-D global tensor; bulk async group.
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed groups of this thread have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ------------------------------------------------------------------------------------- tcgen05
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "n"(NCOLS)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every previously issued UMMA of this thread has completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread t = lane base + t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
      " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// --------------------------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, SWIZZLE_128B (layout_type 2), descriptor version 1 (sm_100).
// Byte offsets are stored >>4. Field positions per the sm_100 UMMA descriptor (bits: start [0,14),
// LBO [16,30), SBO [32,46), version [46,48), base_offset [49,52), layout [61,64)).
//  K-major  operand: rows (M or N) are 128 B apart, 8-row groups SBO apart; LBO is not used.
//  MN-major operand: K rows are 128 B apart, 8-row K groups SBO apart, and successive 64-element
//                    blocks along M/N are LBO apart.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                         uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffff) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}

// ------------------------------------------------------------------------------------------ CTA pairs (cta_group::2)
// Primitives validated on sm_100a by tools/umma2_probe.cu (profiles/r01_umma_2cta_probe.log): a cluster of two CTAs
// issues ONE 256 x N x 16 MMA from the even CTA; each CTA holds its 128 rows of A and HALF of B (N / 2 rows) in its own
// shared memory at the same offsets, and its 128 accumulator rows in its own tensor memory.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc2(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on the barrier at offset `bar` in BOTH CTAs of the pair once every MMA issued so far has completed.
__device__ __forceinline__ void umma2_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
// TMA loads of a CTA pair: the data lands in THIS CTA's shared memory, the bytes are counted on `cluster_bar`, a
// shared::cluster barrier address that may belong to the peer (the even CTA, whose thread issues the MMAs).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* m, uint32_t cluster_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(cluster_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(uint32_t dst, const CUtensorMap* m, uint32_t cluster_bar, int c0, int c1,
                                                 int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
      "r"(c4)
      : "memory");
}

// Instruction descriptor for kind::f16 with bf16 inputs and fp32 accumulation.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                                   // D format: fp32
         | (1u << 7)                                 // A format: bf16
         | (1u << 10)                                // B format: bf16
         | (static_cast<uint32_t>(a_mn_major) << 15)
         | (static_cast<uint32_t>(b_mn_major) << 16)
         | (static_cast<uint32_t>(N >> 3) << 17)
         | (static_cast<uint32_t>(M >> 4) << 24);
}

}  // namespace bsl
