// Inline-PTX wrappers for the Blackwell (sm_100a) async machinery: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (UMMA) + TMEM.  Hand-written; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace sv {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Watchdog: a pipeline bug must fail loudly, never hang the GPU box.  ~2 s of no progress -> trap.
#ifndef SV_MBAR_TIMEOUT_CYCLES
#define SV_MBAR_TIMEOUT_CYCLES 4000000000LL
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > SV_MBAR_TIMEOUT_CYCLES) {
      printf("[surgvid] mbarrier timeout: block %d thread %d bar@%u parity %u\n", blockIdx.x, threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// One leader lane of a CONVERGED warp (the same lane every time for the full mask).  tcgen05.mma / tcgen05.commit / TMA instructions take
// their operands from uniform registers: issued under `if (lane == 0)` the compiler wraps every one of them in a serialising
// BRA.U.ANY loop with R2UR moves, issued under elect.sync inside warp-uniform control flow they are emitted back to back
// (scripts/ubench/umma_rate.cu: 570 -> 512 cycles per 4-MMA group at N = 256, 571 -> 457 at N = 160).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load global -> shared, completion signalled on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// cp.async.bulk.wait_group.read takes an immediate: at most n (0..3) of this thread's bulk store groups may still be reading shared memory
__device__ __forceinline__ void bulk_wait_group_read(int n) {
  switch (n) {
    case 0: asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); break;
    default: asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory"); break;
  }
}
// Ask the TMA unit to pull a tile into L2 only (no shared-memory destination, no barrier): used to run the HBM stream well
// ahead of the shared-memory ring, whose depth alone cannot cover DRAM latency for short-K GEMMs.
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* map, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1) : "memory");
}

// 4-D tile load (e.g. NHWC activation tile with halo); out-of-bounds coordinates (negative or past the extent) are zero-filled.
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// im2col-mode load from an NHWC tensor (map from cuTensorMapEncodeIm2col): pixelsPerColumn pixels, channelsPerPixel channels from c,
// starting at pixel (w, h, n) and walking the map's bounding box with its element strides (row by row, then image by image); each
// pixel is read at (w + off_w, h + off_h).  Pixels outside the tensor (conv padding, images past the last) are zero-filled.
__device__ __forceinline__ void tma_load_im2col_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c, int32_t w, int32_t h, int32_t n,
                                                   uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (bf16/fp16 in, fp32 accumulate). One thread issues.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued tcgen05.mma of this thread arrive on `bar` when complete (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns (thread t gets lane base+t).
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- CTA pairs (cluster of 2, tcgen05 cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory variable in another CTA of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
// Arrive on a (possibly remote) CTA's barrier.  Default semantics (.release at CTA scope) on purpose: a .release.cluster arrive
// makes the thread wait until all of its earlier writes are visible cluster-wide — measured ~1 800 cycles per call in the GEMM
// epilogue (profiles/r02/gemm_trace_cta0.log) — and the only ordering the accumulator hand-back needs is the tcgen05 one, which
// tcgen05.fence::before_thread_sync in front of the arrive provides.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// In a CTA pair the transaction bytes of BOTH CTAs' loads are counted on the leader (rank 0) CTA's barrier: clearing the
// CTA-rank bit of the shared::cluster address of our own barrier names the leader's copy.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c, int32_t w, int32_t h,
                                                        int32_t n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c), "r"(w), "r"(h), "r"(n),
        "h"(off_w), "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A (128 rows from each CTA's smem) * B (N/2 rows from each CTA's smem); issued by the leader CTA.
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the leader's MMAs arrives on the barrier at the same offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle (tile rows are 128 B = 64 bf16,
// 8-row swizzle atoms of 1024 B stacked contiguously): start>>4 | LBO(ignored)=1 | SBO=1024>>4 | version=1 | SWIZZLE_128B=2.
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // [0,14)
  d |= static_cast<uint64_t>(1) << 16;                      // [16,30) leading byte offset (unused for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // [32,46) stride byte offset between 8-row groups
  d |= static_cast<uint64_t>(1) << 46;                      // [46,48) descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                      // [61,64) SWIZZLE_128B
  return d;
}

// Instruction descriptor for kind::f16: D=f32, A=B=bf16, both K-major, M x N tile.
__host__ __device__ inline uint32_t make_idesc_bf16_f32(int M, int N) {
  uint32_t d = 0;
  d |= 1u << 4;                        // c_format = F32
  d |= 1u << 7;                        // a_format = BF16
  d |= 1u << 10;                       // b_format = BF16
  d |= static_cast<uint32_t>(N >> 3) << 17;
  d |= static_cast<uint32_t>(M >> 4) << 24;
  return d;
}

}  // namespace ptx
}  // namespace sv
