// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Nothing here is generic CUDA; this file only compiles for compute_100a.
#pragma once
#include <cstdint>
#include <cuda.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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
// Bounded wait: a protocol bug must surface as a CUDA error (trap), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

// ------------------------------------------------------------------ proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load global -> shared, completion signalled on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// L2 eviction-priority policy for TMA traffic (createpolicy): evict_last keeps a producer/consumer ring resident until its
// slots are overwritten (dirty lines that are evicted early cost a DRAM write-back each).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
// 2-D tiled store shared -> global (bulk async-group completion) with an L2 cache policy.  The box is read from shared
// memory through the async proxy: generic-proxy writes to it need fence.proxy.async first; the source may be reused after
// wait_group.read.
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* m, uint32_t src_smem, int c0, int c1, uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src_smem), "r"(c0), "r"(c1), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// at most N of this thread's most recent bulk groups still pending (older ones complete, writes performed)
template <int N>
__device__ __forceinline__ void bulk_wait_group_le() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// full cross-proxy fence (generic <-> async, every state space): orders TMA traffic to GLOBAL memory against flags that
// are written / read with ordinary loads and stores
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ------------------------------------------------------------------ inter-CTA flags in global memory (gpu scope)
__device__ __forceinline__ void red_release_gpu_add(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Bounded spin until *p >= want: a protocol bug must surface as a CUDA error (trap), never as a hung GPU.
__device__ __forceinline__ void spin_until_ge(const uint32_t* p, uint32_t want) {
  uint32_t spins = 0;
  while (ld_acquire_gpu(p) < want) {
    __nanosleep(64);
    if (++spins > (1u << 26)) __trap();
  }
}

// system-scope flag reads (flags written by PEER GPUs over NVLink) and the global nanosecond timer for bounded waits
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ------------------------------------------------------------------ clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::f16 (bf16 x bf16 -> f32), single CTA.
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (count 1) on an mbarrier once every tcgen05.mma issued so far by this thread has completed.
// Implies tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// Software-pipelined issue blocks.  An mbarrier.try_wait costs ~170 clk even when the phase has already
// completed (measured, tools/umma_bench.cu) -- more than the four 128xNx16 MMAs of one K=64 box take to issue.  These
// blocks start the try_wait for the NEXT stage first, issue the current stage's work, and only then read the
// predicate, so the wait latency hides behind the issue.  Returns 1 if the next stage is already complete.

// Four MMAs over one K=64 box (descriptor start addresses advance by 32 B = 2 units per K=16 step).
__device__ __forceinline__ uint32_t mma_box_prefetch(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                     uint32_t accumulate_first, uint32_t next_bar, uint32_t next_parity) {
  uint32_t ready;
  asm volatile(
      "{\n\t"
      ".reg .pred P, PA, PT;\n\t"
      ".reg .b64 a1, b1, a2, b2, a3, b3;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%6], %7;\n\t"
      "setp.ne.b32 PA, %5, 0;\n\t"
      "setp.eq.u32 PT, %1, %1;\n\t"
      "add.u64 a1, %2, 2;\n\t"
      "add.u64 b1, %3, 2;\n\t"
      "add.u64 a2, %2, 4;\n\t"
      "add.u64 b2, %3, 4;\n\t"
      "add.u64 a3, %2, 6;\n\t"
      "add.u64 b3, %3, 6;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], %2, %3, %4, PA;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], a1, b1, %4, PT;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], a2, b2, %4, PT;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], a3, b3, %4, PT;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(ready)
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(next_bar), "r"(next_parity)
      : "memory");
  return ready;
}

// Arm `full_bar` for `bytes` and issue one TMA box load; try_wait on the next stage's EMPTY barrier overlaps.
__device__ __forceinline__ uint32_t tma_box_prefetch(uint32_t dst_smem, const CUtensorMap* m, uint32_t full_bar,
                                                     uint32_t bytes, int c0, int c1, uint32_t next_bar,
                                                     uint32_t next_parity) {
  uint32_t ready;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%7], %8;\n\t"
      "mbarrier.arrive.expect_tx.shared::cta.b64 _, [%3], %4;\n\t"
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%1], [%2, {%5, %6}], [%3];\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(ready)
      : "r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(full_bar), "r"(bytes), "r"(c0), "r"(c1), "r"(next_bar),
        "r"(next_parity)
      : "memory");
  return ready;
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive 32-bit columns (lane l gets its own row).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ CTA pairs (cta_group::2)
// A pair = cluster of two CTAs on the two SMs of one TPC.  One tcgen05.mma issued by the leader (cluster rank 0)
// reads A (its M/2 rows) and B (its N/2 rows) from the shared memory of BOTH CTAs at the same offsets and writes the
// accumulator rows of each CTA into that CTA's own TMEM.  All four primitives below were validated on a B200 with
// tools/umma_probe.cu (numerics against a CPU GEMM for K-/MN-major operands, 4x1 and 2x2 accumulator layouts).

// shared::cluster address of `addr` (a shared::cta address of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// arrive (count 1) on an mbarrier of ANY CTA of the cluster.  Default semantics (release at CTA scope): what the
// arrive orders is either nothing in memory (a drained TMEM buffer) or this CTA's OWN shared memory, which the
// peer never reads through the generic proxy -- the tensor core does, after fence.proxy.async.  The .release.cluster
// form compiles to MEMBAR.ALL.GPU + ERRBAR per arrive (26 % of all stall samples in the first version, ncu).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {   // same warp id in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA box load into THIS CTA's shared memory whose completion bytes are counted on the LEADER's mbarrier at the same
// offset (bit 24 of a shared-window address selects the CTA within a pair)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_hint(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                                      uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
// arrive on the barrier at this offset in BOTH CTAs once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void mma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
}
// Four pair-MMAs over one K = 64 slab; descriptor start addresses advance by a_step / b_step (16-byte units) per K = 16
// (2 for a K-major operand, 128 for an MN-major one whose 8-row groups are 1 KiB apart).  The try_wait on the NEXT
// stage's barrier overlaps the issue (see mma_box_prefetch); returns 1 if that stage is already complete.
__device__ __forceinline__ uint32_t mma_box_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t a_step,
                                                 uint32_t b_step, uint32_t idesc, uint32_t accumulate_first,
                                                 uint32_t next_bar, uint32_t next_parity) {
  uint32_t ready;
  asm volatile(
      "{\n\t"
      ".reg .pred P, PA, PT;\n\t"
      ".reg .b64 sa, sb, a1, b1, a2, b2, a3, b3;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%8], %9;\n\t"
      "setp.ne.b32 PA, %7, 0;\n\t"
      "setp.eq.u32 PT, %1, %1;\n\t"
      "cvt.u64.u32 sa, %4;\n\t"
      "cvt.u64.u32 sb, %5;\n\t"
      "add.u64 a1, %2, sa;\n\t"
      "add.u64 b1, %3, sb;\n\t"
      "add.u64 a2, a1, sa;\n\t"
      "add.u64 b2, b1, sb;\n\t"
      "add.u64 a3, a2, sa;\n\t"
      "add.u64 b3, b2, sb;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%1], %2, %3, %6, PA;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%1], a1, b1, %6, PT;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%1], a2, b2, %6, PT;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%1], a3, b3, %6, PT;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(ready)
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(a_step), "r"(b_step), "r"(idesc), "r"(accumulate_first),
        "r"(next_bar), "r"(next_parity)
      : "memory");
  return ready;
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor for a K-major bf16 operand tile stored as rows of 128 B
// (64 bf16) with the 128-byte swizzle, 8-row groups 1024 B apart -- exactly what a TMA box
// {64 elements, R rows} with CU_TENSOR_MAP_SWIZZLE_128B writes.  Field layout (PTX ISA,
// "tcgen05 shared memory descriptor"): [0,14) start>>4, [16,30) LBO>>4 (ignored for swizzled
// K-major), [32,46) SBO>>4, [46,48) version=1, [61,64) layout type (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t smem_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// The same physical tile read as an MN-major operand: a TMA box {64 elements, R rows} of a row-major [k][mn] matrix
// holds 64 consecutive MN elements per 128-byte row and consecutive K per row; the canonical SWIZZLE_128B MN-major
// layout is ((64 mn, groups) , (8 k, groups)) with LBO = byte distance between 64-element MN groups (the next box)
// and SBO = 1 KiB between 8-row K groups.  One K = 16 instruction step advances the start address by 2 KiB.
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// kind::f16 instruction descriptor with explicit operand majors (bit 15: A is MN-major, bit 16: B is MN-major)
__host__ __device__ constexpr uint32_t idesc_bf16_f32_major(int m, int n, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// Instruction descriptor, kind::f16: bf16 A and B (both K-major), f32 accumulate, shape M x N.
// [4,6) D fmt (1=f32), [7,10) A fmt (1=bf16), [10,13) B fmt, bit 15/16 A/B major (0=K),
// [17,23) N>>3, [24,29) M>>4.
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

}  // namespace ptx
