// Inline-PTX wrappers for the Blackwell (sm_100a) tensor-core path: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 alloc / mma / commit / ld / st, UMMA descriptors.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace ge2e {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// One try_wait (hardware-suspended up to a time limit); the common case in a running pipeline.
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
// Slow path, out of line so that the hot loops stay small.  A wait that never completes is a
// programming error in the pipeline: trap after 2 s of wall time instead of hanging the GPU.
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  uint64_t t0 = 0;
  for (uint32_t spins = 0;; ++spins) {
    if (mbar_try_wait(bar, parity)) return;
    if ((spins & 255u) == 255u) {
      const uint64_t t = globaltimer_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > 2000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity);
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int x, int y, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* tmap, int x, int y, int z, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(z), "r"(bar)
      : "memory");
}

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, int x, int y, int z, int w, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(z), "r"(w), "r"(bar)
      : "memory");
}

// plain 1-D bulk copy global -> shared (16-byte aligned, size a multiple of 16), bytes counted on `bar`
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
               : "memory");
}

// multicast variants: the box lands at the same CTA-relative offset in every CTA of `mask` and
// completes tx bytes on the mbarrier at the same offset in each of them
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const void* tmap, int x, int y, uint32_t bar,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster "
      "[%0], [%1, {%2, %3}], [%4], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(bar), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_mc(uint32_t dst, const void* tmap, int x, int y, int z, uint32_t bar,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster "
      "[%0], [%1, {%2, %3, %4}], [%5], %6;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(z), "r"(bar), "h"(mask)
      : "memory");
}


// ---------------------------------------------------------------- TMA stores (shared -> global)
// generic-proxy writes to shared memory become visible to the async proxy (TMA) after this fence
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_store_2d(const void* tmap, int x, int y, uint32_t src) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(src)
               : "memory");
}
// element-wise fp32 add into global memory, performed at the L2 (no read-back to the SM)
__device__ __forceinline__ void tma_reduce_add_2d(const void* tmap, int x, int y, uint32_t src) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(src)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores of this thread have finished READING shared memory
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the `pending` most recent bulk groups of this thread have finished reading shared memory
// (groups complete in commit order; the count is an immediate operand)
__device__ __forceinline__ void tma_store_wait_read_pending(int pending) {
  switch (pending) {
    case 0: asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.bulk.wait_group.read 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.bulk.wait_group.read 5;" ::: "memory"); break;
    case 6: asm volatile("cp.async.bulk.wait_group.read 6;" ::: "memory"); break;
    default: asm volatile("cp.async.bulk.wait_group.read 7;" ::: "memory"); break;
  }
}

// ---------------------------------------------------------------- clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the two halves of cluster_sync_all, for work that fits between them
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05: TMEM management
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t holder_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(holder_smem), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05: MMA
// Shared-memory matrix descriptors (version 1 = Blackwell).
//   K-major operand  [rows][32 tf32], SWIZZLE_128B (16-byte chunks XOR row, 8-row atoms of 1024 B):
//       SBO = 1024 (next 8 rows), LBO unused.  TMA: CU_TENSOR_MAP_SWIZZLE_128B.
//   MN-major TF32 operand [k][32 tf32], SWIZZLE_128B_BASE32B -- the only MN-major layout the
//   hardware accepts for 32-bit operands (32-byte chunks XOR row, 4-row atoms of 512 B):
//       LBO = stride between 32-element MN chunks, SBO = 512 (next 4 k-rows).
//       TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
constexpr uint32_t kLayoutSw128 = 2, kLayoutSw128Base32 = 1;
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;   // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(layout_type) << 61;
  return d;
}
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return smem_desc(addr, lbo_bytes, sbo_bytes, kLayoutSw128);
}
// Instruction descriptor for kind::tf32, fp32 accumulate.
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void umma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued MMAs of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// same, arriving on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"(mask)
      : "memory");
}


// ---------------------------------------------------------------- warp election, cluster addressing
// One lane of a fully converged warp.  Gating tcgen05 / TMA issue with elect.sync (instead of
// `lane == 0`) lets ptxas keep descriptors in uniform registers and emit the instruction once;
// a plain lane test costs a per-lane ELECT loop around every UTCHMMA (probe: 87 vs <35 clk/MMA).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// arrive on an mbarrier given by a shared::cluster address (own or peer CTA)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}

// ---------------------------------------------------------------- cta_group::2 (CTA pair) variants
template <int COLS>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t holder_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(holder_smem), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void umma_tf32_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_ts_2cta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this CTA-relative offset in every CTA of `mask` once all MMAs issued
// so far by this thread have completed
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"(mask)
      : "memory");
}
// TMA loads of a CTA pair: the data lands in this CTA's shared memory, the transaction bytes are
// counted on `cluster_bar`, an mbarrier of the pair's leader CTA (shared::cluster address)
__device__ __forceinline__ void tma_load_2d_2cta(uint32_t dst, const void* tmap, int x, int y, uint32_t cluster_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(cluster_bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2cta(uint32_t dst, const void* tmap, int x, int y, int z,
                                                 uint32_t cluster_bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(z), "r"(cluster_bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2cta(uint32_t dst, const void* tmap, int x, int y, int z, int w,
                                                 uint32_t cluster_bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(z), "r"(w), "r"(cluster_bar)
      : "memory");
}

// ---------------------------------------------------------------- one ring stage per asm block
// The MMA warp's loop is instruction-bound: a ring stage has to be issued in less than the ~520 clk
// its MMAs run, and an mbarrier.try_wait on an already-complete barrier alone costs ~200 clk.  These
// helpers issue, from ONE asm block, (1) a non-blocking probe of the NEXT stage's FULL barrier,
// (2) the stage's MMAs and (3) the commit that releases the stage; the probe's latency overlaps
// with the MMA issue and the caller skips the blocking wait when the probe already succeeded.
// All return the probe result.  Descriptors advance by 2 (= 32 bytes >> 4) per K step of 8.
#define GE2E_MMA_SS(CGS) "tcgen05.mma.cta_group::" CGS ".kind::tf32 [%1], a, b, %6, "
#define GE2E_STAGE_SS_BODY(CGS, COMMIT)                                                             \
  "{\n\t.reg .pred pn, pa, pt;\n\t.reg .b64 a, b, sa, sb;\n\t"                                       \
  "mbarrier.test_wait.parity.shared::cta.b64 pn, [%9], %10;\n\t"                                     \
  "setp.ne.b32 pa, %7, 0;\n\tsetp.eq.b32 pt, %7, %7;\n\t"                                            \
  "cvt.u64.u32 sa, %4;\n\tcvt.u64.u32 sb, %5;\n\t"                                                   \
  "mov.b64 a, %2;\n\tmov.b64 b, %3;\n\t" GE2E_MMA_SS(CGS) "pa;\n\t"                                  \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"                              \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"                              \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"
#define GE2E_STAGE_SS_SLAB2(CGS)                                                                    \
  "add.u64 a, %2, sa;\n\tadd.u64 b, %3, sb;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"                          \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"                              \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"                              \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_SS(CGS) "pt;\n\t"
#define GE2E_COMMIT_1 "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%8];\n\t"
#define GE2E_COMMIT_2 \
  "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%8], %11;\n\t"
#define GE2E_STAGE_END "selp.u32 %0, 1, 0, pn;\n\t}"

// NSLAB (1 or 2) K-slabs of 32 columns, both operands from shared memory (K-major, 128B swizzle):
// 4 * NSLAB MMAs.  a_step / b_step: descriptor distance (bytes >> 4) between the two slabs.
template <int CG, int NSLAB>
__device__ __forceinline__ uint32_t umma_stage_ss(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t a_step,
                                                  uint32_t b_step, uint32_t idesc, uint32_t acc_first,
                                                  uint32_t empty_bar, uint32_t probe_bar, uint32_t probe_parity) {
  uint32_t ready;
  const uint16_t mask = 3;
  if (CG == 1 && NSLAB == 1)
    asm volatile(GE2E_STAGE_SS_BODY("1", 1) GE2E_COMMIT_1 GE2E_STAGE_END
                 : "=r"(ready) : "r"(d_tmem), "l"(da), "l"(db), "r"(a_step), "r"(b_step), "r"(idesc), "r"(acc_first),
                   "r"(empty_bar), "r"(probe_bar), "r"(probe_parity), "h"(mask) : "memory");
  else if (CG == 1)
    asm volatile(GE2E_STAGE_SS_BODY("1", 1) GE2E_STAGE_SS_SLAB2("1") GE2E_COMMIT_1 GE2E_STAGE_END
                 : "=r"(ready) : "r"(d_tmem), "l"(da), "l"(db), "r"(a_step), "r"(b_step), "r"(idesc), "r"(acc_first),
                   "r"(empty_bar), "r"(probe_bar), "r"(probe_parity), "h"(mask) : "memory");
  else if (NSLAB == 1)
    asm volatile(GE2E_STAGE_SS_BODY("2", 2) GE2E_COMMIT_2 GE2E_STAGE_END
                 : "=r"(ready) : "r"(d_tmem), "l"(da), "l"(db), "r"(a_step), "r"(b_step), "r"(idesc), "r"(acc_first),
                   "r"(empty_bar), "r"(probe_bar), "r"(probe_parity), "h"(mask) : "memory");
  else
    asm volatile(GE2E_STAGE_SS_BODY("2", 2) GE2E_STAGE_SS_SLAB2("2") GE2E_COMMIT_2 GE2E_STAGE_END
                 : "=r"(ready) : "r"(d_tmem), "l"(da), "l"(db), "r"(a_step), "r"(b_step), "r"(idesc), "r"(acc_first),
                   "r"(empty_bar), "r"(probe_bar), "r"(probe_parity), "h"(mask) : "memory");
  return ready;
}

// 4 MMAs with A from tensor memory (8 columns = 8 k per MMA) and B MN-major from shared memory
// (descriptor advances by 64 = 1024 bytes >> 4 per 8 k-rows).
#define GE2E_MMA_TS(CGS) "tcgen05.mma.cta_group::" CGS ".kind::tf32 [%1], [ta], b, %6, "
#define GE2E_STAGE_TS_BODY(CGS)                                                                     \
  "{\n\t.reg .pred pn, pa, pt;\n\t.reg .b64 b;\n\t.reg .b32 ta;\n\t"                                 \
  "mbarrier.test_wait.parity.shared::cta.b64 pn, [%9], %10;\n\t"                                     \
  "setp.ne.b32 pa, %7, 0;\n\tsetp.eq.b32 pt, %7, %7;\n\t"                                            \
  "mov.b32 ta, %2;\n\tmov.b64 b, %3;\n\t" GE2E_MMA_TS(CGS) "pa;\n\t"                                 \
  "add.u32 ta, ta, 8;\n\tadd.u64 b, b, 64;\n\t" GE2E_MMA_TS(CGS) "pt;\n\t"                           \
  "add.u32 ta, ta, 8;\n\tadd.u64 b, b, 64;\n\t" GE2E_MMA_TS(CGS) "pt;\n\t"                           \
  "add.u32 ta, ta, 8;\n\tadd.u64 b, b, 64;\n\t" GE2E_MMA_TS(CGS) "pt;\n\t"
template <int CG>
__device__ __forceinline__ uint32_t umma_stage_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t db, uint32_t idesc,
                                                  uint32_t acc_first, uint32_t empty_bar, uint32_t probe_bar,
                                                  uint32_t probe_parity) {
  uint32_t ready;
  const uint16_t mask = 3;
  const uint32_t unused = 0;
  if (CG == 1)
    asm volatile(GE2E_STAGE_TS_BODY("1") GE2E_COMMIT_1 GE2E_STAGE_END
                 : "=r"(ready) : "r"(d_tmem), "r"(a_tmem), "l"(db), "r"(unused), "r"(unused), "r"(idesc), "r"(acc_first),
                   "r"(empty_bar), "r"(probe_bar), "r"(probe_parity), "h"(mask) : "memory");
  else
    asm volatile(GE2E_STAGE_TS_BODY("2") GE2E_COMMIT_2 GE2E_STAGE_END
                 : "=r"(ready) : "r"(d_tmem), "r"(a_tmem), "l"(db), "r"(unused), "r"(unused), "r"(idesc), "r"(acc_first),
                   "r"(empty_bar), "r"(probe_bar), "r"(probe_parity), "h"(mask) : "memory");
  return ready;
}

// ---------------------------------------------------------------- kind::f16 (split-precision path)
// fp32 operands travel as two fp16 planes (hi = fp16(x), lo = fp16(x - hi)); a product is three MMAs
// (hi hi, hi lo, lo hi) into the same fp32 accumulator.  Same byte geometry as the TF32 path: a K step is
// 16 elements = 32 bytes (descriptor + 2), an MN-major K step is 16 rows = 2048 bytes (descriptor + 128),
// an A operand in tensor memory takes 8 columns per K step (two fp16 per 32-bit cell).
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (static_cast<uint32_t>(a_mn_major) << 15) | (static_cast<uint32_t>(b_mn_major) << 16) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// non-blocking probe of an mbarrier phase
__device__ __forceinline__ uint32_t mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  return done;
}
#define GE2E_MMA_F16_SS(CGS) "tcgen05.mma.cta_group::" CGS ".kind::f16 [%0], a, b, %3, "
#define GE2E_F16_SS4(CGS)                                                                           \
  "{\n\t.reg .pred pa, pt;\n\t.reg .b64 a, b;\n\t"                                               \
  "setp.ne.b32 pa, %4, 0;\n\tsetp.eq.b32 pt, %4, %4;\n\t"                                         \
  "mov.b64 a, %1;\n\tmov.b64 b, %2;\n\t" GE2E_MMA_F16_SS(CGS) "pa;\n\t"                          \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_F16_SS(CGS) "pt;\n\t"                      \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_F16_SS(CGS) "pt;\n\t"                      \
  "add.u64 a, a, 2;\n\tadd.u64 b, b, 2;\n\t" GE2E_MMA_F16_SS(CGS) "pt;\n\t}"
// 4 MMAs over one [rows x 64 fp16] K-major slab pair (K = 64): D (+)= A_slab . B_slab^T
template <int CG>
__device__ __forceinline__ void umma_f16_ss4(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc,
                                             uint32_t acc_first) {
  if (CG == 1)
    asm volatile(GE2E_F16_SS4("1") ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(acc_first) : "memory");
  else
    asm volatile(GE2E_F16_SS4("2") ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(acc_first) : "memory");
}
// 2 MMAs (32 k-rows): A from tensor memory (16 columns), B MN-major from shared memory
#define GE2E_MMA_F16_TS(CGS) "tcgen05.mma.cta_group::" CGS ".kind::f16 [%0], [ta], b, %3, "
#define GE2E_F16_TS2(CGS)                                                                           \
  "{\n\t.reg .pred pa, pt;\n\t.reg .b64 b;\n\t.reg .b32 ta;\n\t"                                \
  "setp.ne.b32 pa, %4, 0;\n\tsetp.eq.b32 pt, %4, %4;\n\t"                                         \
  "mov.b32 ta, %1;\n\tmov.b64 b, %2;\n\t" GE2E_MMA_F16_TS(CGS) "pa;\n\t"                         \
  "add.u32 ta, ta, 8;\n\tadd.u64 b, b, 128;\n\t" GE2E_MMA_F16_TS(CGS) "pt;\n\t}"
template <int CG>
__device__ __forceinline__ void umma_f16_ts2(uint32_t d_tmem, uint32_t a_tmem, uint64_t db, uint32_t idesc,
                                             uint32_t acc_first) {
  if (CG == 1)
    asm volatile(GE2E_F16_TS2("1") ::"r"(d_tmem), "r"(a_tmem), "l"(db), "r"(idesc), "r"(acc_first) : "memory");
  else
    asm volatile(GE2E_F16_TS2("2") ::"r"(d_tmem), "r"(a_tmem), "l"(db), "r"(idesc), "r"(acc_first) : "memory");
}

// elect.sync with the leader's lane id (the same for every lane of the warp)
__device__ __forceinline__ bool elect_leader(uint32_t& leader) {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync %1|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(pred), "=r"(leader));
  return pred != 0;
}

// ---------------------------------------------------------------- tcgen05: TMEM <-> registers
// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp gets lane (base_lane + t).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- misc
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ptx
}  // namespace ge2e
