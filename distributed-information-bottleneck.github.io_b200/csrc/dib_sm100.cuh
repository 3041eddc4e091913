// dib_sm100.cuh -- thin inline-PTX wrappers for the Blackwell (sm_100a) async machinery used by the tensor-core
// kernels: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (TMEM alloc / mma / commit / ld) and the UMMA shared-memory
// and instruction descriptors.  Bit layouts follow the PTX ISA / CUTLASS cute/arch/mma_sm100_desc.hpp.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sm100 {

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link); nullptr where the driver lacks it
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn tensor_map_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  // (no suspend-time hint: a 10 ms hint removes the poll loops' instructions -- 17 % of the forward kernel's issue slots,
  //  profiles/r02_enc_fwd_source_summary.txt -- but measured no gain there and +30 us in the latency-bound backward kernel:
  //  warps parked with a long limit wake up later)
  return ok != 0;
}
// non-blocking probe: a loop around it never parks the warp (fastest wake-up, costs issue slots while waiting)
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#ifdef DIB_MBAR_SPIN
  while (!mbar_test_wait(bar, parity)) {}
#else
  while (!mbar_try_wait(bar, parity)) {}
#endif
}
// for a lone control thread that shares its scheduler with working warps: back off between polls
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) {
#ifdef DIB_MBAR_SPIN
  while (!mbar_test_wait(bar, parity)) {}
  return;
#endif
  while (!mbar_try_wait(bar, parity)) {}   // try_wait itself suspends for a bounded time; an extra nanosleep only adds hop latency
}

// ------------------------------------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (tcgen05.mma / TMA store reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------ TMEM / tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {   // whole warp, ncols = 2^k >= 32
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {    // whole warp (the allocating one)
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; one thread issues on behalf of the CTA.
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
template <bool BF16>
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  umma_bf16(d_tmem, adesc, bdesc, idesc, accumulate);   // kind::f16 covers fp16 and bf16; the idesc selects the format
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns: thread `lane` of the warp gets row (quarter*32 + lane), r[j] = column j.
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ CTA pair (cta_group::2)
// Two CTAs of a cluster (same TPC) execute ONE tcgen05.mma with M = 256: each CTA holds its 128 rows of A, HALF of B (N / 2) in its
// own shared memory and its 128 rows of the accumulator in its own TMEM.  Only the even CTA issues MMAs; both issue TMA loads
// that signal the even CTA's mbarrier (CUTLASS SM100_TMA_2SM_LOAD / SM100_MMA_F16BF16_2x1SM_SS / umma_arrive_multicast_2x1SM).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {            // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of THIS CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {      // arrive on a (possibly remote) mbarrier
  // relaxed: the only thing the waiter consumes is TMEM that tcgen05.wait::ld has already finished reading -- a release here would
  // also wait for this warp's outstanding global stores (MEMBAR + ERRBAR: 12 % of the CTA-pair kernel's stall samples)
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// TMA loads of a CTA pair: data lands in THIS CTA's shared memory, the bytes are counted on `cluster_bar` (the even CTA's barrier)
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const void* map, uint32_t cluster_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(cluster_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma2_load_3d(uint32_t dst, const void* map, uint32_t cluster_bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tmem2_alloc(uint32_t smem_dst, uint32_t ncols) {   // the same warp id in BOTH CTAs of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem2_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem2_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B with M = 256 (instruction descriptor built with m = 256); issued by one thread of the even CTA
__device__ __forceinline__ void umma2_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on the mbarrier at this shared-memory offset in every CTA of `cta_mask` when all MMAs issued so far have completed
__device__ __forceinline__ void umma2_commit(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask) : "memory");
}

// ---- warp-uniform issue: the WHOLE warp runs the issue loop (uniform control flow lets ptxas keep descriptors, barrier
// addresses and loop state in uniform registers) and one elected lane executes the instruction.  With `if (lane == 0)` around the
// loop every tcgen05 operand went through an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall (~15 instructions per MMA).
__device__ __forceinline__ void umma_f16_w(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_w(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma2_f16_w(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma2_commit_w(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
      ::"r"(bar), "h"(cta_mask) : "memory");
}

// ------------------------------------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): SWIZZLE_128B, sm_100 version bit.
//   K-major  operand tile [rows x 128 B]: 8-row groups of 1024 B;  SBO = 1024 (next 8 rows), LBO unused (=16 B).
//   MN-major operand tile: panels of [k-rows x 128 B] (128 B = 32 fp32 / 64 bf16 along M/N);
//                          SBO = 1024 (next 8 k-rows), LBO = panel stride (next 128 B worth of M/N).
//   fp32/tf32 MN-major operands must use LayoutType::SWIZZLE_128B_BASE32B (CUTLASS sm100_common.inl: "for mn-major
//   tf32 operands, SW128_32B is the only available smem layout"): atoms of 4 k-rows x 128 B in which the 32-byte
//   chunk index is XORed with (k-row % 4)  (cute Swizzle<2,5,2>; TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
//   SBO = 512 (next 4 k-rows), LBO = panel stride.
constexpr uint32_t kLayoutSw128 = 2, kLayoutSw128Base32 = 1, kLayoutNone = 0;
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t layout_type = kLayoutSw128) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
  d |= (uint64_t)layout_type << 61;
  return d;
}

// the same from an address in 16-byte units: `(base >> 4) + constant` folds to ONE add per descriptor in an unrolled issue sequence
// (the byte-address form costs add + shift + mask + or for each of the two descriptors of every MMA; a lone issuing thread then
// issues MMAs more slowly than the tensor pipe retires them)
__device__ __forceinline__ uint64_t umma_desc16(uint32_t addr16, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type = kLayoutSw128) {
  const uint32_t lo = addr16 + (((lbo_bytes >> 4) & 0x3FFF) << 16);
  const uint32_t hi = ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (layout_type << 29);
  return ((uint64_t)hi << 32) | lo;
}
// The same descriptor split in two words for issue loops: only the 14-bit start-address field (bits 0..13 of the low word, units
// of 16 bytes) changes between the MMAs of a kernel, so a loop advances `lo` by (byte offset >> 4) and keeps `hi` -- a single
// issuing thread otherwise spends more time rebuilding 64-bit descriptors than the tensor pipe spends on the MMA.
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr & 0x3FFFF) >> 4) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
__device__ __forceinline__ uint32_t umma_desc_hi(uint32_t sbo_bytes, uint32_t layout_type = kLayoutSw128) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (layout_type << 29);
}
__device__ __forceinline__ uint64_t umma_desc_join(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// Instruction descriptor (cute::UMMA::InstrDescriptor), dense, fp32 accumulate, M = 128.
//   fmt: 0 = f16, 1 = bf16, 2 = tf32;  a_mn / b_mn: 1 = MN-major operand
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t fmt, uint32_t a_mn, uint32_t b_mn, uint32_t n, uint32_t m = 128) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn << 15) | (b_mn << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

}  // namespace sm100
