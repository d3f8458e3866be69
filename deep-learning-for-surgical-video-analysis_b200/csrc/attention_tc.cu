// softmax(Q K^T * scale) V on the 5th-generation tensor cores (tcgen05 + TMEM) for head_dim 64 and N_kv <= 448:
// every encoder block of mit_b1..b5_evp (mix_transformer_evp.py:123-127; N_kv = 49 at 224x224, 390/405 at 480x854).
//
// One CTA = one (frame, head) and a run of 128-row query tiles; K and V of the (frame, head) stay resident in shared memory.
//   warp 8     TMA loads: K/V tiles once, Q tiles through a 2-deep ring that is refilled as soon as the S MMAs of a tile have read it
//              (3-D tensor maps [C, N, frames]: rows past the frame's last token are zero-filled on load and clipped on store, so
//              tiles never bleed into the next frame).
//   warp 10    TMA stores of the finished output tiles (staged in the P buffer the tile's PV MMAs have consumed).
//   warp 9     one thread issues tcgen05.mma: S = Q K^T (M=128, N=64 per key tile, K = 64) into TMEM, then O += P_t V_t per key tile
//              (A = P from shared memory, B = V as an MN-major operand: V is used as stored, no transpose).
//   warps 0-7  two softmax groups of 4 warps; thread = query row (TMEM lane).  tcgen05.ld of the S row, scale in the log2 domain, mask
//              keys >= N_kv, row max, exp2, row sum; P as bf16 into the 128B-swizzled K-major A tile (generic-proxy stores +
//              fence.proxy.async); after the PV MMAs: O row from TMEM, * 1/l, bf16, into the (consumed) P buffer in the swizzled
//              layout of the TMA store.
// N_kv <= 64 (one key tile; 224x224): the groups PING-PONG over query tiles — S and O are double-buffered in TMEM (256 columns), so
// the MMAs and TMEM round trips of one tile hide behind the exponentials of the other.
// 64 < N_kv <= 448 (480x854): all of S (up to 448 columns) sits in TMEM at once — exact two-pass softmax, no online rescaling of O.
// Both groups work on the SAME query tile: group g takes the key tiles t = g (mod 2) and owns P buffer g of the 2-deep ring (the PV
// MMA of tile t overlaps the exponentials of tile t+1); row max and row sum are exchanged through shared memory; each group
// normalises and stages one half of the output columns.
#include <stdlib.h>

#include <string>

#include "host.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sv {
namespace {

constexpr int kHD = 64;                 // head dim == one 128-byte swizzle row of bf16
constexpr int kQRows = 128;             // query rows per tile == UMMA M == TMEM lanes
constexpr int kKeys = 64;               // keys per tile == UMMA N of S == K extent of one PV step group
constexpr int kMaxKt = 7;               // 7 * 64 S columns + 64 O columns = 512 TMEM columns
constexpr int kQBytes = kQRows * kHD * 2;   // 16 KB
constexpr int kKBytes = kKeys * kHD * 2;    // 8 KB
constexpr int kThreads = 384;               // 8 softmax warps + a control warpgroup: Q/K/V loader, MMA issuer, output store (+ 1 idle)

struct AttnTcParams {
  int Nq, Nkv, kt, tpc, qtiles;
  float scale_log2;
  unsigned tmem_cols;
};

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               :
               : "r"(ptx::smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// MN-major B operand (V tile: rows = keys = K index, 128 B of head dim = N index per row), 128-byte swizzle, N = 64 = one atom:
// start>>4 | LBO (one N atom: unused) | SBO = 1024 B between 8-key groups | version 1 | SWIZZLE_128B
__device__ __forceinline__ uint64_t make_sw128_mnmajor_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// chunks [c_begin, c_begin + 4) (32 bf16) of row `row` of a 128B-swizzled tile: chunk c lives at row*128 + ((c ^ (row & 7)) << 4)
__device__ __forceinline__ void store_half_row_sw128(uint8_t* tile, int row, int c_begin, const uint32_t (&w)[16]) {
  uint8_t* rp = tile + row * 128;
  const int x = row & 7;
#pragma unroll
  for (int c = 0; c < 4; ++c)
    *reinterpret_cast<uint4*>(rp + (((c_begin + c) ^ x) << 4)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// max over the valid keys of 32 raw scores (key index kbase + i)
__device__ __forceinline__ float max32(const uint32_t (&r)[32], int kbase, int Nkv, float m) {
  if (kbase + 32 <= Nkv) {
#pragma unroll
    for (int i = 0; i < 32; ++i) m = fmaxf(m, __uint_as_float(r[i]));
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) m = fmaxf(m, (kbase + i < Nkv) ? __uint_as_float(r[i]) : -INFINITY);
  }
  return m;
}
// p = exp2(s * scale - m) for 32 scores -> 16 packed bf16x2 words; returns the partial row sum
__device__ __forceinline__ float exp32(const uint32_t (&r)[32], int kbase, int Nkv, float scale_log2, float m, uint32_t (&w)[16]) {
  float l0 = 0.f, l1 = 0.f;
  if (kbase + 32 <= Nkv) {
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      const float a0 = sv_ex2(fmaf(__uint_as_float(r[i]), scale_log2, -m));       // arguments <= 0: ex2.approx.ftz, 2 ulp
      const float a1 = sv_ex2(fmaf(__uint_as_float(r[i + 1]), scale_log2, -m));
      l0 += a0; l1 += a1;
      w[i >> 1] = pack_bf16x2(a0, a1);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      const float a0 = (kbase + i < Nkv) ? sv_ex2(fmaf(__uint_as_float(r[i]), scale_log2, -m)) : 0.f;
      const float a1 = (kbase + i + 1 < Nkv) ? sv_ex2(fmaf(__uint_as_float(r[i + 1]), scale_log2, -m)) : 0.f;
      l0 += a0; l1 += a1;
      w[i >> 1] = pack_bf16x2(a0, a1);
    }
  }
  return l0 + l1;
}

template <bool MULTI>
__global__ void __launch_bounds__(kThreads, MULTI ? 1 : 2)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k, const __grid_constant__ CUtensorMap tmap_v,
                    const __grid_constant__ CUtensorMap tmap_o, const AttnTcParams p) {
  extern __shared__ uint8_t attn_tc_smem[];
  __shared__ __align__(8) uint64_t kv_full, q_full[2], q_empty[2], s_full[2], p_full[2], p_empty[2], o_full[2], o_staged[2], st_done[2];
  __shared__ float xch[2][2][kQRows];   // MULTI: [row max | row sum][group][row]
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int head = blockIdx.y, b = blockIdx.z;
  const int tile0 = blockIdx.x * p.tpc;
  const int ntiles = min(p.tpc, p.qtiles - tile0);
  const int kt = MULTI ? p.kt : 1;
  uint8_t* smem = attn_tc_smem + ((1024u - (ptx::smem_u32(attn_tc_smem) & 1023u)) & 1023u);
  uint8_t* Qs = smem;                       // [2][16 KB]
  uint8_t* Ks = Qs + 2 * kQBytes;           // [kt][8 KB]
  uint8_t* Vs = Ks + kt * kKBytes;          // [kt][8 KB]
  uint8_t* Ps = Vs + kt * kKBytes;          // [2][16 KB]; a consumed P buffer doubles as the staging tile of the output

  if (warp == 8 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_q);
    ptx::prefetch_tensormap(&tmap_k);
    ptx::prefetch_tensormap(&tmap_v);
    ptx::prefetch_tensormap(&tmap_o);
  }
  if (warp == 9) {
    if (lane == 0) {
      ptx::mbar_init(&kv_full, 1);
      for (int i = 0; i < 2; ++i) {
        ptx::mbar_init(&q_full[i], 1);
        ptx::mbar_init(&q_empty[i], 1);
        ptx::mbar_init(&st_done[i], 1);
        ptx::mbar_init(&s_full[i], 1);
        ptx::mbar_init(&p_full[i], 128);
        ptx::mbar_init(&p_empty[i], 1);
        ptx::mbar_init(&o_full[i], 1);
        ptx::mbar_init(&o_staged[i], MULTI ? 256 : 128);
      }
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(&tmem_slot, p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  // TMEM columns.  one key tile: S of group g at 64g, O of group g at 128 + 64g.  several: S tile t at 64t, O at 64*kt.
  const uint32_t tmem_o = tmem_base + static_cast<uint32_t>(MULTI ? kt * kKeys : 2 * kKeys);
  const int c0 = head * kHD;

  // register budget: the control warpgroup gives registers back, the two softmax warpgroups take them.  setmaxnreg moves registers
  // inside the CTA's LAUNCH allocation only (384 threads x 80 at one key tile): 8 * 96 + 4 * 48 = 12 * 80.
  if (warp >= 8) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");   // one instruction for the whole control warpgroup (warps 8-11)
  if (warp == 8) {
    // ------------------------------------------------------------------ TMA loads
    // (all three control warps: the whole warp runs the loop and polls the barriers, ONE ELECTED lane issues the TMA / tcgen05
    // instructions — issued under `if (lane == 0)` every one of them is wrapped in a serialising BRA.U.ANY loop, see ptx::elect_one)
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx(&kv_full, static_cast<uint32_t>(2 * kt * kKBytes));
      for (int t = 0; t < kt; ++t) {
        tma_load_3d(Ks + t * kKBytes, &tmap_k, &kv_full, c0, t * kKeys, b);
        tma_load_3d(Vs + t * kKBytes, &tmap_v, &kv_full, c0, t * kKeys, b);
      }
    }
    __syncwarp();
    for (int j = 0; j < ntiles; ++j) {
      const int qb = j & 1;
      if (j >= 2) ptx::mbar_wait(&q_empty[qb], static_cast<uint32_t>(((j - 2) >> 1) & 1));   // the S MMAs of tile j-2 have read this buffer
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&q_full[qb], kQBytes);
        tma_load_3d(Qs + qb * kQBytes, &tmap_q, &q_full[qb], c0, (tile0 + j) * kQRows, b);
      }
      __syncwarp();
    }
  } else if (warp == 10) {
    // ------------------------------------------------------------------ TMA stores of the output tiles (warp 11 idles)
    for (int j = 0; j < ntiles; ++j) {
      const int sb = MULTI ? 0 : (j & 1);
      ptx::mbar_wait(&o_staged[sb], static_cast<uint32_t>((MULTI ? j : (j >> 1)) & 1));   // the rows of O_j are staged in P buffer sb (and fenced)
      if (ptx::elect_one()) {
        tma_store_3d(&tmap_o, Ps + sb * kQBytes, c0, (tile0 + j) * kQRows, b);
        tma_store_commit();
        tma_store_wait_read();                  // the store has read the buffer: P may be overwritten / the CTA may exit
        ptx::mbar_arrive(&st_done[sb]);
      }
      __syncwarp();
    }
  } else if (warp == 9) {
    // ------------------------------------------------------------------ MMA issuer (converged warp, one elected lane issues)
    {
      const uint32_t idesc_s = ptx::make_idesc_bf16_f32(kQRows, kKeys);                 // A, B K-major
      const uint32_t idesc_pv = ptx::make_idesc_bf16_f32(kQRows, kHD) | (1u << 16);     // B (= V) MN-major
      ptx::mbar_wait(&kv_full, 0u);
      if (!MULTI) {
        // issue order S_0, S_1, PV_0, S_2, PV_1, ...: the S MMA of the next tile is in flight while a group does its exponentials
        const uint64_t dk = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Ks));
        const uint64_t dv = make_sw128_mnmajor_desc(ptx::smem_u32(Vs));
        for (int j = 0; j <= ntiles; ++j) {
          if (j < ntiles) {
            const int g = j & 1;
            ptx::mbar_wait(&q_full[g], static_cast<uint32_t>((j >> 1) & 1));
            ptx::tc_fence_after();
            const uint64_t dq = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Qs + g * kQBytes));
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < kHD / 16; ++ks)
                ptx::umma_f16(tmem_base + static_cast<uint32_t>(g * kKeys), dq + static_cast<uint64_t>(ks * 2), dk + static_cast<uint64_t>(ks * 2), idesc_s, ks ? 1u : 0u);
              ptx::umma_commit(&s_full[g]);
              ptx::umma_commit(&q_empty[g]);
            }
            __syncwarp();
          }
          if (j >= 1) {
            const int jj = j - 1, g = jj & 1;
            // P_jj is in shared memory; the same arrivals order the group's reads of S_jj and of O_{jj-2} before this point
            ptx::mbar_wait(&p_full[g], static_cast<uint32_t>((jj >> 1) & 1));
            ptx::tc_fence_after();
            const uint64_t dp = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Ps + g * kQBytes));
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < kKeys / 16; ++ks)   // 16 keys per step: +32 B along P's rows, +2 swizzle atoms (2048 B) down V
                ptx::umma_f16(tmem_o + static_cast<uint32_t>(g * kHD), dp + static_cast<uint64_t>(ks * 2), dv + static_cast<uint64_t>(ks * (2048 >> 4)), idesc_pv,
                              ks ? 1u : 0u);
              ptx::umma_commit(&o_full[g]);
            }
            __syncwarp();
          }
        }
      } else {
        uint32_t n_pf[2] = {0u, 0u};
        for (int j = 0; j < ntiles; ++j) {
          const int qb = j & 1;
          ptx::mbar_wait(&q_full[qb], static_cast<uint32_t>((j >> 1) & 1));
          ptx::tc_fence_after();
          const uint64_t dq = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Qs + qb * kQBytes));
          if (ptx::elect_one()) {
            for (int t = 0; t < kt; ++t) {
              const uint64_t dk = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Ks + t * kKBytes));
#pragma unroll
              for (int ks = 0; ks < kHD / 16; ++ks)
                ptx::umma_f16(tmem_base + static_cast<uint32_t>(t * kKeys), dq + static_cast<uint64_t>(ks * 2), dk + static_cast<uint64_t>(ks * 2), idesc_s, ks ? 1u : 0u);
            }
            ptx::umma_commit(&s_full[0]);
            ptx::umma_commit(&q_empty[qb]);
          }
          __syncwarp();
          for (int t = 0; t < kt; ++t) {
            const int pb = t & 1;
            const uint32_t par = (pb ? n_pf[1] : n_pf[0]) & 1u;
            ptx::mbar_wait(&p_full[pb], par);
            if (pb) ++n_pf[1]; else ++n_pf[0];
            if (t == 0 && j > 0) ptx::mbar_wait(&o_staged[0], static_cast<uint32_t>((j - 1) & 1));   // O_{j-1} has left TMEM
            ptx::tc_fence_after();
            const uint64_t dp = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Ps + pb * kQBytes));
            const uint64_t dv = make_sw128_mnmajor_desc(ptx::smem_u32(Vs + t * kKBytes));
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < kKeys / 16; ++ks)
                ptx::umma_f16(tmem_o, dp + static_cast<uint64_t>(ks * 2), dv + static_cast<uint64_t>(ks * (2048 >> 4)), idesc_pv, (t | ks) ? 1u : 0u);
              ptx::umma_commit(&p_empty[pb]);
              if (t == kt - 1) ptx::umma_commit(&o_full[0]);
            }
            __syncwarp();
          }
        }
      }
    }
  }
  } else {
    // ------------------------------------------------------------------ softmax + output rows (thread = query row = TMEM lane)
    if (MULTI) asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 96;");
    const int grp = warp >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_sel = static_cast<uint32_t>(quarter * 32) << 16;
    if (!MULTI) {
      const uint32_t t_s = tmem_base + static_cast<uint32_t>(grp * kKeys) + lane_sel;
      const uint32_t t_o = tmem_o + static_cast<uint32_t>(grp * kHD) + lane_sel;
      uint8_t* Pg = Ps + grp * kQBytes;
      for (int j = grp; j < ntiles; j += 2) {
        const uint32_t par = static_cast<uint32_t>((j >> 1) & 1);
        const bool active = (tile0 + j) * kQRows + quarter * 32 < p.Nq;   // warp-uniform: rows past the frame's last query do no math
        ptx::mbar_wait(&s_full[grp], par);
        ptx::tc_fence_after();
        float l = 1.f;
        if (active) {
          uint32_t r0[32], r1[32];
          ptx::tmem_ld_x32(t_s, r0);
          ptx::tmem_ld_x32(t_s + 32u, r1);
          ptx::tmem_ld_wait();
          float m = max32(r0, 0, p.Nkv, -INFINITY);
          m = max32(r1, 32, p.Nkv, m) * p.scale_log2;   // scale > 0: max commutes with it
          uint32_t w[16];
          l = exp32(r0, 0, p.Nkv, p.scale_log2, m, w);
          // P buffer `grp` is free: the PV MMAs of this group's previous tile retired before its o_full, and the TMA store of that
          // tile's output (staged in the same buffer) has finished reading it
          if (j >= 2) ptx::mbar_wait(&st_done[grp], static_cast<uint32_t>(((j - 2) >> 1) & 1));
          store_half_row_sw128(Pg, row, 0, w);
          l += exp32(r1, 32, p.Nkv, p.scale_log2, m, w);
          store_half_row_sw128(Pg, row, 4, w);
        }
        ptx::fence_proxy_async_smem();   // generic-proxy stores of P -> visible to the tensor core
        ptx::tc_fence_before();          // this thread's TMEM reads of S are complete
        ptx::mbar_arrive(&p_full[grp]);
        ptx::mbar_wait(&o_full[grp], par);
        ptx::tc_fence_after();
        if (active) {
          uint32_t r0[32], r1[32];
          ptx::tmem_ld_x32(t_o, r0);
          ptx::tmem_ld_x32(t_o + 32u, r1);
          ptx::tmem_ld_wait();
          const float inv = 1.0f / l;
          uint32_t w[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) w[i >> 1] = pack_bf16x2(__uint_as_float(r0[i]) * inv, __uint_as_float(r0[i + 1]) * inv);
          store_half_row_sw128(Pg, row, 0, w);
#pragma unroll
          for (int i = 0; i < 32; i += 2) w[i >> 1] = pack_bf16x2(__uint_as_float(r1[i]) * inv, __uint_as_float(r1[i + 1]) * inv);
          store_half_row_sw128(Pg, row, 4, w);
        }
        ptx::fence_proxy_async_smem();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&o_staged[grp]);
      }
    } else {
      const uint32_t t_s = tmem_base + lane_sel;
      const uint32_t t_o = tmem_o + static_cast<uint32_t>(grp * 32) + lane_sel;
      uint8_t* Pg = Ps + grp * kQBytes;
      uint32_t n_pe = 0u;
      for (int j = 0; j < ntiles; ++j) {
        const bool active = (tile0 + j) * kQRows + quarter * 32 < p.Nq;
        ptx::mbar_wait(&s_full[0], static_cast<uint32_t>(j & 1));
        ptx::tc_fence_after();
        float m = -INFINITY;
        if (active) {
          for (int t = grp; t < kt; t += 2) {
            uint32_t r[32];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              ptx::tmem_ld_x32(t_s + static_cast<uint32_t>(t * kKeys + h * 32), r);
              ptx::tmem_ld_wait();
              m = max32(r, t * kKeys + h * 32, p.Nkv, m);
            }
          }
        }
        xch[0][grp][row] = m;
        named_bar_sync(1, 256);
        m = fmaxf(xch[0][0][row], xch[0][1][row]) * p.scale_log2;   // finite for active rows: key 0 is valid and belongs to group 0
        float l = 0.f;
        for (int t = grp; t < kt; t += 2) {
          if (n_pe > 0u) ptx::mbar_wait(&p_empty[grp], (n_pe - 1u) & 1u);   // the PV MMA that read this group's P buffer last has retired
          ++n_pe;
          if (grp == 0 && t == 0 && j > 0) ptx::mbar_wait(&st_done[0], static_cast<uint32_t>((j - 1) & 1));   // ... and the store of O_{j-1}, staged in P[0]
          if (active) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t r[32], w[16];
              ptx::tmem_ld_x32(t_s + static_cast<uint32_t>(t * kKeys + h * 32), r);
              ptx::tmem_ld_wait();
              l += exp32(r, t * kKeys + h * 32, p.Nkv, p.scale_log2, m, w);
              store_half_row_sw128(Pg, row, 4 * h, w);
            }
          }
          ptx::fence_proxy_async_smem();
          ptx::tc_fence_before();
          ptx::mbar_arrive(&p_full[grp]);
        }
        xch[1][grp][row] = l;
        ptx::mbar_wait(&o_full[0], static_cast<uint32_t>(j & 1));
        ptx::tc_fence_after();
        named_bar_sync(2, 256);
        if (active) {
          const float inv = 1.0f / (xch[1][0][row] + xch[1][1][row]);
          uint32_t r[32], w[16];
          ptx::tmem_ld_x32(t_o, r);        // this group's half of the output columns
          ptx::tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i += 2) w[i >> 1] = pack_bf16x2(__uint_as_float(r[i]) * inv, __uint_as_float(r[i + 1]) * inv);
          store_half_row_sw128(Ps, row, 4 * grp, w);     // P[0]: every PV MMA of the tile has retired (o_full)
        }
        ptx::fence_proxy_async_smem();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&o_staged[0]);
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---- N_kv <= 64, persistent: a CTA walks a contiguous range of (frame, head, query tile) work items, so the per-CTA set-up (TMEM
// allocation, barrier init, descriptor prefetch) is paid once per SM slot instead of once per one or two tiles (stages 3 and 4 have
// 196 / 49 queries per frame and head), and the K/V tiles of the NEXT (frame, head) are prefetched into a second buffer while the
// current one is being used.  Tile j of the CTA belongs to softmax group j & 1 (ping-pong, S and O double-buffered in TMEM).
struct AttnTcSingleParams {
  int Nq, Nkv, heads, qtiles, tiles_total;
  int order;   // 1: head fastest, items dealt round-robin (several heads); 0: contiguous (frame, head, tile) ranges
  float scale_log2;
};

__global__ void __launch_bounds__(kThreads, 2)
attention_tc_single_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k, const __grid_constant__ CUtensorMap tmap_v,
                           const __grid_constant__ CUtensorMap tmap_o, const AttnTcSingleParams p) {
  extern __shared__ uint8_t attn_tc_smem[];
  __shared__ __align__(8) uint64_t kv_full[2], kv_empty[2], q_full[2], q_empty[2], s_full[2], p_full[2], o_full[2], o_staged[2], st_done[2];
  __shared__ uint32_t tmem_slot;
  constexpr uint32_t kTmemCols = 256;   // S of group g at 64g, O of group g at 128 + 64g

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per = p.tiles_total / static_cast<int>(gridDim.x), extra = p.tiles_total % static_cast<int>(gridDim.x);
  const int ntiles = per + (static_cast<int>(blockIdx.x) < extra ? 1 : 0);
  // Work-item order.  One head: a contiguous range of (frame, query tile) items per CTA (K/V loaded once per frame).  Several heads: the
  // head index runs FASTEST and items are dealt round-robin, so the CTAs running at the same time read / write all heads of the same
  // token rows (whole C-wide rows per DRAM page instead of one 128-byte head slice of every row: with the head outermost the achieved
  // bandwidth fell with the head count, 4.5 / 3.4 / 2.3 / 1.6 TB/s at 1 / 2 / 5 / 8 heads); K/V (16 KB, L2-resident) are then loaded per item.
  const bool rr = p.order != 0 && p.heads > 1;
  const int t_first = rr ? static_cast<int>(blockIdx.x) : static_cast<int>(blockIdx.x) * per + min(static_cast<int>(blockIdx.x), extra);
  const int t_stride = rr ? static_cast<int>(gridDim.x) : 1;
  auto item = [&](int j, int& bh, int& qt) {   // j-th item of this CTA -> (frame * heads + head, query tile)
    const int t = t_first + j * t_stride;
    if (rr) {
      const int head = t % p.heads, r = t / p.heads;
      qt = r % p.qtiles;
      bh = (r / p.qtiles) * p.heads + head;
    } else {
      bh = t / p.qtiles;
      qt = t - bh * p.qtiles;
    }
  };
  uint8_t* smem = attn_tc_smem + ((1024u - (ptx::smem_u32(attn_tc_smem) & 1023u)) & 1023u);
  uint8_t* Qs = smem;                       // [2][16 KB]
  uint8_t* Ks = Qs + 2 * kQBytes;           // [2][8 KB]  K of the current / the next (frame, head)
  uint8_t* Vs = Ks + 2 * kKBytes;           // [2][8 KB]
  uint8_t* Ps = Vs + 2 * kKBytes;           // [2][16 KB]; a consumed P buffer doubles as the staging tile of the output

  if (warp == 8 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_q);
    ptx::prefetch_tensormap(&tmap_k);
    ptx::prefetch_tensormap(&tmap_v);
    ptx::prefetch_tensormap(&tmap_o);
  }
  if (warp == 9) {
    if (lane == 0) {
      for (int i = 0; i < 2; ++i) {
        ptx::mbar_init(&kv_full[i], 1);
        ptx::mbar_init(&kv_empty[i], 1);
        ptx::mbar_init(&q_full[i], 1);
        ptx::mbar_init(&q_empty[i], 1);
        ptx::mbar_init(&s_full[i], 1);
        ptx::mbar_init(&p_full[i], 128);
        ptx::mbar_init(&o_full[i], 1);
        ptx::mbar_init(&o_staged[i], 128);
        ptx::mbar_init(&st_done[i], 1);
      }
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(&tmem_slot, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t tmem_o = tmem_base + 2u * kKeys;

  if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");   // one instruction for the whole control warpgroup; 8 * 96 + 4 * 48 = 12 * 80
    if (warp == 8) {
      // ---------------------------------------------------------------- TMA loads
      // (control warps: the whole warp runs the loop and polls, one elected lane issues — see ptx::elect_one)
      {
        int prev_bh = -1, n_kv = 0;
        for (int j = 0; j < ntiles; ++j) {
          int bh, qt;
          item(j, bh, qt);
          const int b = bh / p.heads, c0 = (bh - b * p.heads) * kHD;
          if (bh != prev_bh) {
            const int kb = n_kv & 1;
            if (n_kv >= 2) ptx::mbar_wait(&kv_empty[kb], static_cast<uint32_t>(((n_kv - 2) >> 1) & 1));   // every MMA on the pair two back has retired
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&kv_full[kb], 2 * kKBytes);
              tma_load_3d(Ks + kb * kKBytes, &tmap_k, &kv_full[kb], c0, 0, b);
              tma_load_3d(Vs + kb * kKBytes, &tmap_v, &kv_full[kb], c0, 0, b);
            }
            __syncwarp();
            ++n_kv;
            prev_bh = bh;
          }
          const int qb = j & 1;
          if (j >= 2) ptx::mbar_wait(&q_empty[qb], static_cast<uint32_t>(((j - 2) >> 1) & 1));   // the S MMAs of tile j-2 have read this buffer
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(&q_full[qb], kQBytes);
            tma_load_3d(Qs + qb * kQBytes, &tmap_q, &q_full[qb], c0, qt * kQRows, b);
          }
          __syncwarp();
        }
      }
    } else if (warp == 10) {
      // ---------------------------------------------------------------- TMA stores of the output tiles (warp 11 idles)
      for (int j = 0; j < ntiles; ++j) {
        int bh, qt;
        item(j, bh, qt);
        const int b = bh / p.heads, c0 = (bh - b * p.heads) * kHD;
        const int sb = j & 1;
        ptx::mbar_wait(&o_staged[sb], static_cast<uint32_t>((j >> 1) & 1));   // the rows of O_j are staged in P buffer sb (and fenced)
        if (ptx::elect_one()) {
          tma_store_3d(&tmap_o, Ps + sb * kQBytes, c0, qt * kQRows, b);
          tma_store_commit();
          tma_store_wait_read();                  // the store has read the buffer: P may be overwritten / the CTA may exit
          ptx::mbar_arrive(&st_done[sb]);
        }
        __syncwarp();
      }
    } else if (warp == 9) {
      // ---------------------------------------------------------------- MMA issuer (converged warp, one elected lane issues)
      {
        const uint32_t idesc_s = ptx::make_idesc_bf16_f32(kQRows, kKeys);                 // A, B K-major
        const uint32_t idesc_pv = ptx::make_idesc_bf16_f32(kQRows, kHD) | (1u << 16);     // B (= V) MN-major
        // issue order S_0, S_1, PV_0, S_2, PV_1, ...: the S MMA of the next tile is in flight while a group does its exponentials
        int n_kv = 0, bh_s = -1, kb_s = 0;   // K/V buffer of the tile whose S is being issued
        int bh_pv = -1, kb_pv = 0;           // ... and of the tile whose PV is being issued (one tile behind)
        for (int j = 0; j <= ntiles; ++j) {
          if (j < ntiles) {
            int bh, qt_unused;
            item(j, bh, qt_unused);
            if (bh != bh_s) {
              kb_s = n_kv & 1;
              ptx::mbar_wait(&kv_full[kb_s], static_cast<uint32_t>((n_kv >> 1) & 1));
              ++n_kv;
              bh_s = bh;
            }
            const int g = j & 1;
            ptx::mbar_wait(&q_full[g], static_cast<uint32_t>((j >> 1) & 1));
            ptx::tc_fence_after();
            const uint64_t dq = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Qs + g * kQBytes));
            const uint64_t dk = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Ks + kb_s * kKBytes));
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < kHD / 16; ++ks)
                ptx::umma_f16(tmem_base + static_cast<uint32_t>(g * kKeys), dq + static_cast<uint64_t>(ks * 2), dk + static_cast<uint64_t>(ks * 2), idesc_s, ks ? 1u : 0u);
              ptx::umma_commit(&s_full[g]);
              ptx::umma_commit(&q_empty[g]);
            }
            __syncwarp();
          }
          if (j >= 1) {
            const int jj = j - 1, g = jj & 1;
            int bh, qt_unused;
            item(jj, bh, qt_unused);
            if (bh != bh_pv) { kb_pv = (bh_pv < 0) ? 0 : (kb_pv ^ 1); bh_pv = bh; }   // pairs alternate buffers in issue order
            // P_jj is in shared memory; the same arrivals order the group's reads of S_jj and of O_{jj-2} before this point
            ptx::mbar_wait(&p_full[g], static_cast<uint32_t>((jj >> 1) & 1));
            ptx::tc_fence_after();
            const uint64_t dp = ptx::make_sw128_kmajor_desc(ptx::smem_u32(Ps + g * kQBytes));
            const uint64_t dv = make_sw128_mnmajor_desc(ptx::smem_u32(Vs + kb_pv * kKBytes));
            // last tile of its (frame, head): once everything issued so far has retired, the K/V buffer may be refilled
            int bh_next = -1;
            if (j < ntiles) item(j, bh_next, qt_unused);
            const bool last_of_pair = j == ntiles || bh_next != bh;
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < kKeys / 16; ++ks)   // 16 keys per step: +32 B along P's rows, +2 swizzle atoms (2048 B) down V
                ptx::umma_f16(tmem_o + static_cast<uint32_t>(g * kHD), dp + static_cast<uint64_t>(ks * 2), dv + static_cast<uint64_t>(ks * (2048 >> 4)), idesc_pv,
                              ks ? 1u : 0u);
              ptx::umma_commit(&o_full[g]);
              if (last_of_pair) ptx::umma_commit(&kv_empty[kb_pv]);
            }
            __syncwarp();
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax + output rows (thread = query row = TMEM lane)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 96;");
    const int grp = warp >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_sel = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t t_s = tmem_base + static_cast<uint32_t>(grp * kKeys) + lane_sel;
    const uint32_t t_o = tmem_o + static_cast<uint32_t>(grp * kHD) + lane_sel;
    uint8_t* Pg = Ps + grp * kQBytes;
    for (int j = grp; j < ntiles; j += 2) {
      const uint32_t par = static_cast<uint32_t>((j >> 1) & 1);
      int bh_unused, qt;
      item(j, bh_unused, qt);
      const bool active = qt * kQRows + quarter * 32 < p.Nq;   // warp-uniform: rows past the frame's last query do no math
      ptx::mbar_wait(&s_full[grp], par);
      ptx::tc_fence_after();
      float l = 1.f;
      if (active) {
        uint32_t r0[32], r1[32];
        ptx::tmem_ld_x32(t_s, r0);
        ptx::tmem_ld_x32(t_s + 32u, r1);
        ptx::tmem_ld_wait();
        float m = max32(r0, 0, p.Nkv, -INFINITY);
        m = max32(r1, 32, p.Nkv, m) * p.scale_log2;   // scale > 0: max commutes with it
        uint32_t w[16];
        l = exp32(r0, 0, p.Nkv, p.scale_log2, m, w);
        // P buffer `grp` is free: the PV MMAs of this group's previous tile retired before its o_full, and the TMA store of that
        // tile's output (staged in the same buffer) has finished reading it
        if (j >= 2) ptx::mbar_wait(&st_done[grp], static_cast<uint32_t>(((j - 2) >> 1) & 1));
        store_half_row_sw128(Pg, row, 0, w);
        l += exp32(r1, 32, p.Nkv, p.scale_log2, m, w);
        store_half_row_sw128(Pg, row, 4, w);
      }
      ptx::fence_proxy_async_smem();   // generic-proxy stores of P -> visible to the tensor core
      ptx::tc_fence_before();          // this thread's TMEM reads of S are complete
      ptx::mbar_arrive(&p_full[grp]);
      ptx::mbar_wait(&o_full[grp], par);
      ptx::tc_fence_after();
      if (active) {
        uint32_t r0[32], r1[32];
        ptx::tmem_ld_x32(t_o, r0);
        ptx::tmem_ld_x32(t_o + 32u, r1);
        ptx::tmem_ld_wait();
        const float inv = 1.0f / l;
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) w[i >> 1] = pack_bf16x2(__uint_as_float(r0[i]) * inv, __uint_as_float(r0[i + 1]) * inv);
        store_half_row_sw128(Pg, row, 0, w);
#pragma unroll
        for (int i = 0; i < 32; i += 2) w[i >> 1] = pack_bf16x2(__uint_as_float(r1[i]) * inv, __uint_as_float(r1[i + 1]) * inv);
        store_half_row_sw128(Pg, row, 4, w);
      } else if (j >= 2) {
        ptx::mbar_wait(&st_done[grp], static_cast<uint32_t>(((j - 2) >> 1) & 1));   // keep the phase bookkeeping of idle warps in step
      }
      ptx::fence_proxy_async_smem();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&o_staged[grp]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// [frames, N, ld] bf16 (token-major, row stride ld) seen as a 3-D tensor {cols, N, frames}; box = 64 columns x rows x 1 frame, 128B swizzle
int encode_tokens_map(CUtensorMap* map, const bf16* base, int cols, int N, int B, int64_t ld, int box_rows) {
  cuuint64_t gdim[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(B)};
  cuuint64_t gstr[2] = {static_cast<cuuint64_t>(ld) * 2, static_cast<cuuint64_t>(N) * static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(kHD), static_cast<cuuint32_t>(box_rows), 1};
  return encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      "attention");
}

}  // namespace

bool attention_tc_enabled() {
  static const bool on = [] { const char* e = getenv("SURGVID_ATTN_TC"); return !(e && atoi(e) == 0); }();
  return on;
}

bool attention_tc_supported(int hd, int Nkv, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, const void* q, const void* k, const void* v, const void* o) {
  if (hd != kHD || Nkv < 1 || Nkv > kMaxKt * kKeys) return false;
  if (ldq % 8 || ldk % 8 || ldv % 8 || ldo % 8) return false;
  return ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(o)) & 15) == 0;
}

int attention_tc_plan(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, const bf16* v, int64_t ldv, bf16* o, int64_t ldo, int B, int heads,
                      int Nq, int Nkv, float scale, AttnTcPlan* plan) {
  SV_CHECK(attention_tc_supported(kHD, Nkv, ldq, ldk, ldv, ldo, q, k, v, o), "attention_tc: unsupported shape / alignment");
  SV_CHECK(B > 0 && B <= 65535 && heads > 0 && heads <= 65535 && Nq > 0, "attention_tc dims");
  const int cols = heads * kHD;
  SV_CHECK(ldq >= cols && ldk >= cols && ldv >= cols && ldo >= cols, "attention_tc leading dims");
  SV_TRY(encode_tokens_map(&plan->tmap_q, q, cols, Nq, B, ldq, kQRows));
  SV_TRY(encode_tokens_map(&plan->tmap_k, k, cols, Nkv, B, ldk, kKeys));
  SV_TRY(encode_tokens_map(&plan->tmap_v, v, cols, Nkv, B, ldv, kKeys));
  SV_TRY(encode_tokens_map(&plan->tmap_o, o, cols, Nq, B, ldo, kQRows));
  plan->B = B; plan->heads = heads; plan->Nq = Nq; plan->Nkv = Nkv;
  plan->kt = ceil_div(Nkv, kKeys);
  plan->qtiles = ceil_div(Nq, kQRows);
  plan->scale_log2 = scale * 1.4426950408889634f;
  // query tiles per CTA: as many as still leave a few CTAs per SM-slot (K/V are loaded once per CTA)
  int tpc = 1;
  const long long want = 8LL * std::max(1, device_sm_count());
  while (tpc < 8 && tpc * 2 <= plan->qtiles && static_cast<long long>(ceil_div(plan->qtiles, tpc * 2)) * heads * B >= want) tpc *= 2;
  if (plan->kt == 1 && tpc == 1 && plan->qtiles >= 2) tpc = 2;   // the two softmax groups ping-pong over a CTA's tiles
  plan->tpc = tpc;
  const int need_cols = plan->kt > 1 ? plan->kt * kKeys + kHD : 4 * kKeys;   // one key tile: S and O double-buffered (ping-pong groups)
  plan->tmem_cols = need_cols <= 256 ? 256 : 512;
  plan->smem_bytes = 2 * kQBytes + 2 * plan->kt * kKBytes + 2 * kQBytes + 1024;
  return SV_OK;
}

int attention_tc_launch(const AttnTcPlan& plan, cudaStream_t st) {
  AttnTcParams p;
  p.Nq = plan.Nq; p.Nkv = plan.Nkv; p.kt = plan.kt; p.tpc = plan.tpc; p.qtiles = plan.qtiles; p.scale_log2 = plan.scale_log2;
  p.tmem_cols = static_cast<unsigned>(plan.tmem_cols);
  dim3 grid(ceil_div(plan.qtiles, plan.tpc), plan.heads, plan.B);
  if (plan.kt > 1) {
    SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(attention_tc_kernel<true>), 2 * kQBytes + 2 * kMaxKt * kKBytes + 2 * kQBytes + 1024));
    attention_tc_kernel<true><<<grid, kThreads, plan.smem_bytes, st>>>(plan.tmap_q, plan.tmap_k, plan.tmap_v, plan.tmap_o, p);
  } else {
    AttnTcSingleParams sp;
    sp.Nq = plan.Nq; sp.Nkv = plan.Nkv; sp.heads = plan.heads; sp.qtiles = plan.qtiles; sp.scale_log2 = plan.scale_log2;
    static const int order_env = [] { const char* e = getenv("SURGVID_ATTN_ORDER"); return e ? atoi(e) : 0; }();
    sp.order = order_env;
    const long long total = static_cast<long long>(plan.B) * plan.heads * plan.qtiles;
    if (total >= (1LL << 31)) return fail(SV_ERR_INVALID, "attention_tc: more than 2^31 query tiles");
    sp.tiles_total = static_cast<int>(total);
    const int smem_single = 4 * kQBytes + 4 * kKBytes + 1024;
    SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(attention_tc_single_kernel), smem_single));
    // persistent: two CTAs per SM, each walking a contiguous range of >= 2 tiles (one per softmax group)
    const int grid1 = static_cast<int>(std::min<long long>(std::max<long long>(1, (total + 1) / 2), 2LL * std::max(1, device_sm_count())));
    attention_tc_single_kernel<<<grid1, kThreads, smem_single, st>>>(plan.tmap_q, plan.tmap_k, plan.tmap_v, plan.tmap_o, sp);
  }
  return launch_status("attention_tc_kernel");
}

}  // namespace sv
