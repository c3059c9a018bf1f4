// Hand-written sm_100a PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc/mma/commit/ld/st),
// UMMA shared-memory and instruction descriptors.  No CuTe / CUTLASS: everything here is inline PTX plus the
// bit layouts of the two descriptor words.
//
// Replaces (on the reference side) the Ampere-era PTX macro sets
//   kernels/hgemm/mma/basic/hgemm_mma_stage.cu:L29-51   (cp.async / ldmatrix / mma.sync m16n8k16)
//   kernels/flash-attn/utils/utils.h:L32-59              (same set for the attention kernels)
//   ffpa-attn-mma/include/cuffpa/{mma,cp_async}.cuh
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace b200k {

#ifndef B200K_SPIN_LIMIT_CYCLES
// A protocol bug in an mbarrier pipeline shows up as a hang.  Every spin-wait below gives up after this many
// SM cycles (~5 s), prints which barrier it was waiting on and traps, so a bug becomes a CUDA error instead
// of a dead GPU box.  The check is only reached after a failed try_wait (slow path).
#define B200K_SPIN_LIMIT_CYCLES (10LL * 1000 * 1000 * 1000)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(pred));
  return pred;
}
// Address of `local_smem_addr` inside CTA `rank` of this cluster (shared::cluster window).
__device__ __forceinline__ uint32_t mapa(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_arrive() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_sync() {
  cluster_arrive();
  cluster_wait();
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Register re-allocation between warpgroups (all 4 warps of an aligned warpgroup must execute it).
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// ---------------------------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// generic-proxy writes (st.shared) -> visible to the async proxy (TMA store, tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on a barrier that lives in another CTA of the cluster (address from mapa())
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// Remote arrive WITHOUT release semantics, for hand-shakes that order nothing but tensor-memory accesses which have already
// completed (tcgen05.wait::ld / ::st + tcgen05.fence::before_thread_sync in front of it).  The .release.cluster form costs a
// GPU-wide memory fence per arrive (MEMBAR.ALL.GPU + ERRBAR in SASS, 1-1.5 k cycles measured inside the FFPA O^T kernel).
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// non-blocking probe (mbarrier.test_wait): has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
static __device__ __noinline__ void mbar_timeout_trap(uint32_t bar, uint32_t parity) {
  printf("[b200k] mbarrier wait timed out: block (%d,%d) thread %d bar 0x%x parity %u\n", blockIdx.x, blockIdx.y,
         threadIdx.x, bar, parity);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > B200K_SPIN_LIMIT_CYCLES) mbar_timeout_trap(bar, parity);
  }
}

// ---------------------------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// L2 cache-policy words (createpolicy fractional encodings; same constants every TMA user passes)
constexpr uint64_t kPolicyEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kPolicyEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kPolicyEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int32_t c0,
                                            int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
// cta_group::2 form: data lands in THIS CTA's smem, the complete_tx is signalled on `cluster_bar`, which may
// live in the peer (leader) CTA of the pair (shared::cluster address from mapa()).
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst_smem, const CUtensorMap* m, uint32_t cluster_bar,
                                                int32_t c0, int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(cluster_bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int32_t c0,
                                            int32_t c1, int32_t c2, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst_smem, const CUtensorMap* m, uint32_t cluster_bar,
                                                int32_t c0, int32_t c1, int32_t c2, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t src_smem, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src_smem, int32_t c0, int32_t c1,
                                             int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src_smem), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {  // smem source may be overwritten afterwards
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {  // global writes are complete
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------------------------------------- tcgen05 / TMEM
template <int CTA_GROUP>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  if constexpr (CTA_GROUP == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
                 : "memory");
}
template <int CTA_GROUP>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (CTA_GROUP == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int CTA_GROUP>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (CTA_GROUP == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]       (kind::f16: fp16/bf16 operands, f32 or f16 accumulate)
template <int CTA_GROUP, bool TF32 = false>
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  if constexpr (TF32 && CTA_GROUP == 1)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else if constexpr (TF32)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else if constexpr (CTA_GROUP == 1)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]   (the "TS" form: A operand read from tensor memory)
template <int CTA_GROUP>
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  if constexpr (CTA_GROUP == 1)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Make `bar` (this CTA) observe completion of all prior tcgen05 ops issued by this thread.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// cta_group::2: arrive on the barrier at the same smem offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(cta_mask)
      : "memory");
}

// TMEM address: bits [31:16] lane, [15:0] column.  A warp may only touch lanes 32*(warp_id%4) .. +31.
__device__ __forceinline__ uint32_t tmem_addr(uint32_t base, uint32_t lane, uint32_t col) {
  return base + (lane << 16) + col;
}
// 32 lanes x 32-bit, N consecutive columns: thread t of the warp receives lane (base_lane+t), columns c..c+N-1.
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
          taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

// ---------------------------------------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor (64 bit):
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4 (LBO)
//   [32,46) stride-dim byte offset >> 4 (SBO)      [46,48) version = 1 (Blackwell)
//   [49,52) base offset = 0           [61,64) swizzle: 0 none, 2 = 128B, 4 = 64B, 6 = 32B
// Canonical layouts with 128B swizzle and 16-bit elements (units: 16-byte chunks):
//   K-major  ("row = M/N index, 64 K-elements = 128 B per row"):   rows at 128 B, groups of 8 rows at SBO (=1024 B
//            when the tile is one TMA box of 64 x rows), LBO unused.  A K step of 16 elements = +32 B on the address.
//   MN-major ("row = K index, 64 M/N-elements = 128 B per row"):   8 K-rows form a 1024 B atom, next 8 K-rows at
//            SBO, next 64 M/N-elements at LBO.  A K step of 16 = +2*SBO on the address.
constexpr uint32_t kSwizzle128B = 2;
__host__ __device__ constexpr uint64_t make_smem_desc_hi(uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t swizzle) {
  return (uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16) | (uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32) |
         (uint64_t(1) << 46) | (uint64_t(swizzle & 7) << 61);
}
__device__ __forceinline__ uint64_t smem_desc(uint64_t hi_template, uint32_t smem_addr) {
  return hi_template | uint64_t((smem_addr >> 4) & 0x3FFF);
}

// Instruction descriptor for kind::f16 (32 bit):
//   [4,6) D format: 0 = f16, 1 = f32      [7,10) A format: 0 = f16, 1 = bf16     [10,13) B format
//   [13] negate A  [14] negate B  [15] A major: 0 = K, 1 = MN   [16] B major      [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t m, uint32_t n, bool acc_f32, bool a_mn_major,
                                                      bool b_mn_major, bool bf16 = false) {
  return (uint32_t(acc_f32 ? 1 : 0) << 4) | (uint32_t(bf16 ? 1 : 0) << 7) | (uint32_t(bf16 ? 1 : 0) << 10) |
         (uint32_t(a_mn_major ? 1 : 0) << 15) | (uint32_t(b_mn_major ? 1 : 0) << 16) | ((n >> 3) << 17) |
         ((m >> 4) << 24);
}

// Same descriptor with the operand format spelled out: 0 = f16, 1 = bf16 (kind::f16), 2 = tf32 (kind::tf32); fp32
// accumulation.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t m, uint32_t n, int fmt, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (uint32_t(fmt) << 7) | (uint32_t(fmt) << 10) | (uint32_t(a_mn_major ? 1 : 0) << 15) |
         (uint32_t(b_mn_major ? 1 : 0) << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// ---------------------------------------------------------------------------------------------- small helpers
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf162(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_shared_u16(uint32_t addr, uint16_t a) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(a) : "memory");
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Blackwell packed fp32x2 arithmetic (FFMA2 / FADD2): two fp32 lanes per instruction and issue slot.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  ra = (unsigned long long)__float_as_uint(a.x) | ((unsigned long long)__float_as_uint(a.y) << 32);
  rb = (unsigned long long)__float_as_uint(b.x) | ((unsigned long long)__float_as_uint(b.y) << 32);
  rc = (unsigned long long)__float_as_uint(c.x) | ((unsigned long long)__float_as_uint(c.y) << 32);
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return make_float2(__uint_as_float((unsigned)rd), __uint_as_float((unsigned)(rd >> 32)));
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  unsigned long long ra, rb, rd;
  ra = (unsigned long long)__float_as_uint(a.x) | ((unsigned long long)__float_as_uint(a.y) << 32);
  rb = (unsigned long long)__float_as_uint(b.x) | ((unsigned long long)__float_as_uint(b.y) << 32);
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  return make_float2(__uint_as_float((unsigned)rd), __uint_as_float((unsigned)(rd >> 32)));
}

// 2^x on the FMA/ALU pipes (no MUFU): Cody-Waite split x = n + f, f in [-0.5, 0.5], degree-3 minimax polynomial for
// 2^f (max relative error 1.0e-4, below the 4.9e-4 rounding step of the fp16 P it feeds), exponent patched in with
// an integer multiply-add.  Used for a fraction of the softmax exponentials so that the MUFU pipe (16 ex2/clk/SM) is
// not the only source of exponentials (the FlashAttention-4 trick).
__device__ __forceinline__ float exp2_poly3(float x) {
  x = fmaxf(x, -126.0f);                       // also maps -inf (masked keys) to 2^-126 -> 0 in fp16
  const float magic = 12582912.0f;             // 1.5 * 2^23: x + magic has round(x) in its low mantissa bits
  const float t = x + magic;
  const float f = x - (t - magic);
  float p = fmaf(f, 5.500892858e-02f, 2.422109601e-01f);
  p = fmaf(p, f, 6.932829276e-01f);
  p = fmaf(p, f, 1.0f);
  // (bits(t) << 23) == n << 23 (mod 2^32): the low 9 bits of bits(magic) are zero
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}

// Packed (fp32x2) version of exp2_poly3: two exponentials per instruction slot on the FMA pipe.
__device__ __forceinline__ float2 exp2_poly3_x2(float2 x) {
  x.x = fmaxf(x.x, -126.0f);
  x.y = fmaxf(x.y, -126.0f);
  const float2 magic = make_float2(12582912.0f, 12582912.0f);
  const float2 t = fadd2(x, magic);
  const float2 nnf = ffma2(t, make_float2(-1.0f, -1.0f), magic);  // magic - t = -round(x), exact
  const float2 f = fadd2(x, nnf);
  float2 p = ffma2(f, make_float2(5.500892858e-02f, 5.500892858e-02f), make_float2(2.422109601e-01f, 2.422109601e-01f));
  p = ffma2(p, f, make_float2(6.932829276e-01f, 6.932829276e-01f));
  p = ffma2(p, f, make_float2(1.0f, 1.0f));
  // exponent patch: bits(p) + (bits(t) << 23), one LEA per element on the ALU pipe
  uint32_t rx, ry;
  asm("{\n\t.reg .b32 u;\n\tshl.b32 u, %2, 23;\n\tadd.s32 %0, %1, u;\n\t}" : "=r"(rx) : "r"(__float_as_uint(p.x)), "r"(__float_as_uint(t.x)));
  asm("{\n\t.reg .b32 u;\n\tshl.b32 u, %2, 23;\n\tadd.s32 %0, %1, u;\n\t}" : "=r"(ry) : "r"(__float_as_uint(p.y)), "r"(__float_as_uint(t.y)));
  return make_float2(__uint_as_float(rx), __uint_as_float(ry));
}

// tcgen05.st of N consecutive 32-bit columns (N = 8, 16, 32 or 64) from registers r[0..N)
template <int N>
__device__ __forceinline__ void tmem_st_n(uint32_t taddr, const uint32_t* r) {
  static_assert(N == 8 || N == 16 || N == 32 || N == 64, "tmem_st_n");
  if constexpr (N == 8) tmem_st_32x32b_x8(taddr, r);
  if constexpr (N == 16) tmem_st_32x32b_x16(taddr, r);
  if constexpr (N == 32) tmem_st_32x32b_x32(taddr, r);
  if constexpr (N == 64) {
    tmem_st_32x32b_x32(taddr, r);
    tmem_st_32x32b_x32(taddr + 32, r + 32);
  }
}

// 3-input max (FMNMX3): half the ALU-pipe slots of a 2-input max chain
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// max of s[0..N) with four independent FMNMX3 chains (N % 8 == 4 or N % 8 == 0, N >= 12)
template <int N>
__device__ __forceinline__ float row_max(const float* s) {
  static_assert(N >= 12 && N % 4 == 0, "row_max");
  float m0 = s[0], m1 = s[1], m2 = s[2], m3 = s[3];
  constexpr int FULL = 4 + ((N - 4) / 8) * 8;
#pragma unroll
  for (int c = 4; c < FULL; c += 8) {
    m0 = fmax3(m0, s[c], s[c + 1]);
    m1 = fmax3(m1, s[c + 2], s[c + 3]);
    m2 = fmax3(m2, s[c + 4], s[c + 5]);
    m3 = fmax3(m3, s[c + 6], s[c + 7]);
  }
  if constexpr (FULL < N) {
    m0 = fmax3(m0, s[FULL], s[FULL + 1]);
    m1 = fmax3(m1, s[FULL + 2], s[FULL + 3]);
  }
  return fmax3(m0, m1, fmaxf(m2, m3));
}

}  // namespace b200k
