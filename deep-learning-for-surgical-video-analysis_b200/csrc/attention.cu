// Fused softmax(Q K^T * scale) V for spatial-reduction attention (mix_transformer_evp.py:123-127) and the
// flow cross-attention (nn.MultiheadAttention, mix_transformer_evp.py:868-883).  One CTA = 64 query rows of one
// (frame, head); K/V are streamed through shared memory in 64-key tiles with an online softmax, so the
// [B, heads, N, N_kv] attention matrix the reference materialises never exists.  bf16 operands, fp32 softmax and
// accumulation.  Tensor-core path: mma.sync m16n8k16 (round-1 implementation; 2.6 % of the path's FLOPs).
#include <mutex>

#include "kernels.cuh"

namespace sv {

namespace {

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

constexpr int kTile = 64;  // query rows per CTA and keys per smem tile

template <int HD>
struct AttnShape {
  static constexpr int HDP = (HD + 15) / 16 * 16;  // head dim padded to the MMA K granularity
  static constexpr int KS = HDP / 16;              // k-steps of Q K^T
  static constexpr int NTO = HDP / 8;              // n-tiles of the output
  static constexpr int LDS = HDP + 8;              // smem row stride (elements): odd multiple of 16 B -> conflict-free ldmatrix
};

// rows [r0, r0+64) x HD columns of a bf16 matrix -> smem tile [64][LDS], zero-filling OOB rows and pad columns
template <int HD>
__device__ __forceinline__ void load_tile(bf16* __restrict__ dst, const bf16* __restrict__ src, int64_t ld, int r0, int rows_total) {
  using S = AttnShape<HD>;
  if constexpr (HD % 8 == 0) {
    constexpr int CH = S::HDP / 8;
    for (int i = threadIdx.x; i < kTile * CH; i += blockDim.x) {
      const int r = i / CH, c = i % CH;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (r0 + r < rows_total && c * 8 < HD) v = __ldg(reinterpret_cast<const uint4*>(src + static_cast<int64_t>(r0 + r) * ld + c * 8));
      *reinterpret_cast<uint4*>(dst + r * S::LDS + c * 8) = v;
    }
  } else {  // head_dim 20 (mit_b0_evp flow cross-attention): a head starts 8-byte aligned only, so move 8-byte chunks
    constexpr int CH = S::HDP / 4;
    for (int i = threadIdx.x; i < kTile * CH; i += blockDim.x) {
      const int r = i / CH, c = i % CH;
      uint2 v = make_uint2(0u, 0u);
      if (r0 + r < rows_total && c * 4 < HD) v = __ldg(reinterpret_cast<const uint2*>(src + static_cast<int64_t>(r0 + r) * ld + c * 4));
      *reinterpret_cast<uint2*>(dst + r * S::LDS + c * 4) = v;
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(128) attention_kernel(const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ k, int64_t ldk,
                                                        const bf16* __restrict__ v, int64_t ldv, bf16* __restrict__ o, int64_t ldo,
                                                        int Nq, int Nkv, float scale_log2) {
  using S = AttnShape<HD>;
  __shared__ __align__(16) bf16 Qs[kTile * S::LDS];
  __shared__ __align__(16) bf16 Ks[kTile * S::LDS];
  __shared__ __align__(16) bf16 Vs[kTile * S::LDS];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int head = blockIdx.y, b = blockIdx.z;
  const int q0 = blockIdx.x * kTile;
  const bf16* qb = q + static_cast<int64_t>(b) * Nq * ldq + head * HD;
  const bf16* kb = k + static_cast<int64_t>(b) * Nkv * ldk + head * HD;
  const bf16* vb = v + static_cast<int64_t>(b) * Nkv * ldv + head * HD;
  bf16* ob = o + static_cast<int64_t>(b) * Nq * ldo + head * HD;

  load_tile<HD>(Qs, qb, ldq, q0, Nq);
  __syncthreads();

  // Q fragments of this warp's 16 rows stay in registers for the whole kernel
  uint32_t qf[S::KS][4];
  {
    const int mi = lane >> 3;
    const int row = warp * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
    for (int ks = 0; ks < S::KS; ++ks) {
      const int col = ks * 16 + (mi >> 1) * 8;
      ldmatrix_x4(qf[ks], static_cast<uint32_t>(__cvta_generic_to_shared(Qs + row * S::LDS + col)));
    }
  }

  float m_run[2] = {-INFINITY, -INFINITY};
  float l_run[2] = {0.f, 0.f};
  float oacc[S::NTO][4];
#pragma unroll
  for (int i = 0; i < S::NTO; ++i) { oacc[i][0] = oacc[i][1] = oacc[i][2] = oacc[i][3] = 0.f; }

  for (int kv0 = 0; kv0 < Nkv; kv0 += kTile) {
    __syncthreads();  // previous tile fully consumed
    load_tile<HD>(Ks, kb, ldk, kv0, Nkv);
    load_tile<HD>(Vs, vb, ldv, kv0, Nkv);
    __syncthreads();

    // S = Q K^T for 64 keys: 8 n-tiles
    float sacc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { sacc[i][0] = sacc[i][1] = sacc[i][2] = sacc[i][3] = 0.f; }
    {
      const int mi = lane >> 3;
#pragma unroll
      for (int ks = 0; ks < S::KS; ++ks) {
#pragma unroll
        for (int np = 0; np < 4; ++np) {  // pairs of key n-tiles
          const int key = np * 16 + (mi >> 1) * 8 + (lane & 7);
          const int col = ks * 16 + (mi & 1) * 8;
          uint32_t kf[4];
          ldmatrix_x4(kf, static_cast<uint32_t>(__cvta_generic_to_shared(Ks + key * S::LDS + col)));
          mma_bf16_16816(sacc[np * 2], qf[ks], kf[0], kf[1]);
          mma_bf16_16816(sacc[np * 2 + 1], qf[ks], kf[2], kf[3]);
        }
      }
    }
    // scale (log2 domain), mask keys beyond Nkv, online softmax
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = kv0 + nt * 8 + t * 2 + (e & 1);
        float s = sacc[nt][e] * scale_log2;
        if (key >= Nkv) s = -INFINITY;
        sacc[nt][e] = s;
        mx[e >> 1] = fmaxf(mx[e >> 1], s);
      }
    }
    float corr[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float m_new = fmaxf(m_run[r], mx[r]);  // finite: every tile has >= 1 valid key
      corr[r] = exp2f(m_run[r] - m_new);
      m_run[r] = m_new;
      l_run[r] *= corr[r];
    }
#pragma unroll
    for (int i = 0; i < S::NTO; ++i) {
      oacc[i][0] *= corr[0]; oacc[i][1] *= corr[0];
      oacc[i][2] *= corr[1]; oacc[i][3] *= corr[1];
    }
    uint32_t pf[4][4];  // P as A-fragments for the 4 key k-steps
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float p0 = exp2f(sacc[nt][0] - m_run[0]);
      const float p1 = exp2f(sacc[nt][1] - m_run[0]);
      const float p2 = exp2f(sacc[nt][2] - m_run[1]);
      const float p3 = exp2f(sacc[nt][3] - m_run[1]);
      l_run[0] += p0 + p1;
      l_run[1] += p2 + p3;
      const int kk = nt >> 1;
      if ((nt & 1) == 0) { pf[kk][0] = pack_bf16x2(p0, p1); pf[kk][1] = pack_bf16x2(p2, p3); }
      else               { pf[kk][2] = pack_bf16x2(p0, p1); pf[kk][3] = pack_bf16x2(p2, p3); }
    }
    // O += P V
    {
      const int mi = lane >> 3;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
        for (int dp = 0; dp < S::NTO / 2; ++dp) {
          const int key = kk * 16 + (mi & 1) * 8 + (lane & 7);
          const int col = (dp * 2 + (mi >> 1)) * 8;
          uint32_t vf[4];
          ldmatrix_x4_trans(vf, static_cast<uint32_t>(__cvta_generic_to_shared(Vs + key * S::LDS + col)));
          mma_bf16_16816(oacc[dp * 2], pf[kk], vf[0], vf[1]);
          mma_bf16_16816(oacc[dp * 2 + 1], pf[kk], vf[2], vf[3]);
        }
      }
    }
  }

#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
  const float inv0 = 1.0f / l_run[0], inv1 = 1.0f / l_run[1];
  const int row0 = q0 + warp * 16 + g, row1 = row0 + 8;
#pragma unroll
  for (int i = 0; i < S::NTO; ++i) {
    const int col = i * 8 + t * 2;
    if (col < HD) {
      if (row0 < Nq) *reinterpret_cast<uint32_t*>(ob + static_cast<int64_t>(row0) * ldo + col) = pack_bf16x2(oacc[i][0] * inv0, oacc[i][1] * inv0);
      if (row1 < Nq) *reinterpret_cast<uint32_t*>(ob + static_cast<int64_t>(row1) * ldo + col) = pack_bf16x2(oacc[i][2] * inv1, oacc[i][3] * inv1);
    }
  }
}

// ---- N_kv <= 64 (every encoder block at 224x224: N_kv = 49): K and V of one (frame, head) stay resident in shared memory
// while the CTA walks over several 64-row query tiles; query tiles are double-buffered with cp.async, the softmax is single
// pass (all keys at once), and the output tile goes back through shared memory so that global stores are 16-byte coalesced.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  const int bytes = valid ? 16 : 0;  // src-size 0 -> zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  const int bytes = valid ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int HD>
__device__ __forceinline__ void load_tile_async(bf16* __restrict__ dst, const bf16* __restrict__ src, int64_t ld, int r0, int rows_total) {
  using S = AttnShape<HD>;
  if constexpr (HD % 8 == 0) {
    constexpr int CH = S::HDP / 8;
    for (int i = threadIdx.x; i < kTile * CH; i += blockDim.x) {
      const int r = i / CH, c = i % CH;
      const bool ok = (r0 + r < rows_total) && (c * 8 < HD);
      const bf16* g = ok ? src + static_cast<int64_t>(r0 + r) * ld + c * 8 : src;
      cp_async16(dst + r * S::LDS + c * 8, g, ok);
    }
  } else {
    constexpr int CH = S::HDP / 4;
    for (int i = threadIdx.x; i < kTile * CH; i += blockDim.x) {
      const int r = i / CH, c = i % CH;
      const bool ok = (r0 + r < rows_total) && (c * 4 < HD);
      const bf16* g = ok ? src + static_cast<int64_t>(r0 + r) * ld + c * 4 : src;
      cp_async8(dst + r * S::LDS + c * 4, g, ok);
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(128) attention_resident_kv_kernel(const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ k, int64_t ldk,
                                                                    const bf16* __restrict__ v, int64_t ldv, bf16* __restrict__ o, int64_t ldo,
                                                                    int Nq, int Nkv, float scale_log2, int tiles_per_cta) {
  using S = AttnShape<HD>;
  __shared__ __align__(16) bf16 Qs[2][kTile * S::LDS];
  __shared__ __align__(16) bf16 Ks[kTile * S::LDS];
  __shared__ __align__(16) bf16 Vs[kTile * S::LDS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int head = blockIdx.y, b = blockIdx.z;
  const int tile0 = blockIdx.x * tiles_per_cta;
  const int ntiles = min(tiles_per_cta, (Nq + kTile - 1) / kTile - tile0);
  const bf16* qb = q + static_cast<int64_t>(b) * Nq * ldq + head * HD;
  const bf16* kb = k + static_cast<int64_t>(b) * Nkv * ldk + head * HD;
  const bf16* vb = v + static_cast<int64_t>(b) * Nkv * ldv + head * HD;
  bf16* ob = o + static_cast<int64_t>(b) * Nq * ldo + head * HD;

  load_tile_async<HD>(Ks, kb, ldk, 0, Nkv);
  load_tile_async<HD>(Vs, vb, ldv, 0, Nkv);
  load_tile_async<HD>(Qs[0], qb, ldq, tile0 * kTile, Nq);
  cp_async_commit();

  const int mi = lane >> 3;
  for (int j = 0; j < ntiles; ++j) {
    const int q0 = (tile0 + j) * kTile;
    bf16* Qc = Qs[j & 1];
    if (j + 1 < ntiles) load_tile_async<HD>(Qs[(j + 1) & 1], qb, ldq, q0 + kTile, Nq);  // overlaps this tile's math
    cp_async_commit();
    cp_async_wait<1>();  // everything except the group just committed has landed (K, V, Q(j))
    __syncthreads();

    if (q0 + warp * 16 < Nq) {   // a warp whose 16 rows lie beyond the last query (196 = 3 x 64 + 4) has nothing to do for this tile
    uint32_t qf[S::KS][4];
    {
      const int row = warp * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
      for (int ks = 0; ks < S::KS; ++ks)
        ldmatrix_x4(qf[ks], static_cast<uint32_t>(__cvta_generic_to_shared(Qc + row * S::LDS + ks * 16 + (mi >> 1) * 8)));
    }
    float sacc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { sacc[i][0] = sacc[i][1] = sacc[i][2] = sacc[i][3] = 0.f; }
#pragma unroll
    for (int ks = 0; ks < S::KS; ++ks) {
#pragma unroll
      for (int np = 0; np < 4; ++np) {
        const int key = np * 16 + (mi >> 1) * 8 + (lane & 7);
        uint32_t kf[4];
        ldmatrix_x4(kf, static_cast<uint32_t>(__cvta_generic_to_shared(Ks + key * S::LDS + ks * 16 + (mi & 1) * 8)));
        mma_bf16_16816(sacc[np * 2], qf[ks], kf[0], kf[1]);
        mma_bf16_16816(sacc[np * 2 + 1], qf[ks], kf[2], kf[3]);
      }
    }
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = nt * 8 + t * 2 + (e & 1);
        float sv = sacc[nt][e] * scale_log2;
        if (key >= Nkv) sv = -INFINITY;
        sacc[nt][e] = sv;
        mx[e >> 1] = fmaxf(mx[e >> 1], sv);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
    }
    float l[2] = {0.f, 0.f};
    uint32_t pf[4][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float p0 = exp2f(sacc[nt][0] - mx[0]), p1 = exp2f(sacc[nt][1] - mx[0]);
      const float p2 = exp2f(sacc[nt][2] - mx[1]), p3 = exp2f(sacc[nt][3] - mx[1]);
      l[0] += p0 + p1;
      l[1] += p2 + p3;
      const int kk = nt >> 1;
      if ((nt & 1) == 0) { pf[kk][0] = pack_bf16x2(p0, p1); pf[kk][1] = pack_bf16x2(p2, p3); }
      else               { pf[kk][2] = pack_bf16x2(p0, p1); pf[kk][3] = pack_bf16x2(p2, p3); }
    }
    float oacc[S::NTO][4];
#pragma unroll
    for (int i = 0; i < S::NTO; ++i) { oacc[i][0] = oacc[i][1] = oacc[i][2] = oacc[i][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
      for (int dp = 0; dp < S::NTO / 2; ++dp) {
        const int key = kk * 16 + (mi & 1) * 8 + (lane & 7);
        uint32_t vf[4];
        ldmatrix_x4_trans(vf, static_cast<uint32_t>(__cvta_generic_to_shared(Vs + key * S::LDS + (dp * 2 + (mi >> 1)) * 8)));
        mma_bf16_16816(oacc[dp * 2], pf[kk], vf[0], vf[1]);
        mma_bf16_16816(oacc[dp * 2 + 1], pf[kk], vf[2], vf[3]);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l[r] += __shfl_xor_sync(0xffffffffu, l[r], 1);
      l[r] += __shfl_xor_sync(0xffffffffu, l[r], 2);
    }
    const float inv0 = 1.0f / l[0], inv1 = 1.0f / l[1];
    // this warp's 16 output rows go back through its own rows of the (now consumed) query tile, then out 16 bytes per lane
    __syncwarp();
#pragma unroll
    for (int i = 0; i < S::NTO; ++i) {
      const int col = i * 8 + t * 2;
      *reinterpret_cast<uint32_t*>(Qc + (warp * 16 + g) * S::LDS + col) = pack_bf16x2(oacc[i][0] * inv0, oacc[i][1] * inv0);
      *reinterpret_cast<uint32_t*>(Qc + (warp * 16 + g + 8) * S::LDS + col) = pack_bf16x2(oacc[i][2] * inv1, oacc[i][3] * inv1);
    }
    __syncwarp();
    if constexpr (HD % 8 == 0) {
      constexpr int CH = HD / 8;  // 16-byte chunks per output row
      for (int i = lane; i < 16 * CH; i += 32) {
        const int r = i / CH, c = i % CH;
        const int row = q0 + warp * 16 + r;
        if (row < Nq)
          *reinterpret_cast<uint4*>(ob + static_cast<int64_t>(row) * ldo + c * 8) = *reinterpret_cast<const uint4*>(Qc + (warp * 16 + r) * S::LDS + c * 8);
      }
    } else {
      constexpr int CH = HD / 4;  // 8-byte chunks
      for (int i = lane; i < 16 * CH; i += 32) {
        const int r = i / CH, c = i % CH;
        const int row = q0 + warp * 16 + r;
        if (row < Nq)
          *reinterpret_cast<uint2*>(ob + static_cast<int64_t>(row) * ldo + c * 4) = *reinterpret_cast<const uint2*>(Qc + (warp * 16 + r) * S::LDS + c * 4);
      }
    }
    }
    __syncthreads();  // Qc may be refilled by the prefetch issued at the top of the next-but-one iteration
  }
  cp_async_wait<0>();
}

// ---- 64 < N_kv <= 256 (the flow cross-attention at 224x224: N_kv = 196, head_dim 40): K and V of one (frame, head) are still small
// enough to stay resident (dynamic shared memory); the CTA walks over its query tiles as above and, per tile, over the resident
// 64-key tiles with the online softmax of the streaming kernel — no reloads of K/V per query tile, no load/compute serialisation.
template <int HD>
__global__ void __launch_bounds__(128) attention_resident_multi_kernel(const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ k, int64_t ldk,
                                                                       const bf16* __restrict__ v, int64_t ldv, bf16* __restrict__ o, int64_t ldo,
                                                                       int Nq, int Nkv, float scale_log2, int tiles_per_cta, int kv_tiles) {
  using S = AttnShape<HD>;
  extern __shared__ __align__(16) uint8_t attn_smem[];
  bf16* Qs0 = reinterpret_cast<bf16*>(attn_smem);
  bf16* Qs1 = Qs0 + kTile * S::LDS;
  bf16* Ks = Qs1 + kTile * S::LDS;
  bf16* Vs = Ks + kv_tiles * kTile * S::LDS;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int head = blockIdx.y, b = blockIdx.z;
  const int tile0 = blockIdx.x * tiles_per_cta;
  const int ntiles = min(tiles_per_cta, (Nq + kTile - 1) / kTile - tile0);
  const bf16* qb = q + static_cast<int64_t>(b) * Nq * ldq + head * HD;
  const bf16* kb = k + static_cast<int64_t>(b) * Nkv * ldk + head * HD;
  const bf16* vb = v + static_cast<int64_t>(b) * Nkv * ldv + head * HD;
  bf16* ob = o + static_cast<int64_t>(b) * Nq * ldo + head * HD;

  for (int kt = 0; kt < kv_tiles; ++kt) {
    load_tile_async<HD>(Ks + kt * kTile * S::LDS, kb, ldk, kt * kTile, Nkv);
    load_tile_async<HD>(Vs + kt * kTile * S::LDS, vb, ldv, kt * kTile, Nkv);
  }
  load_tile_async<HD>(Qs0, qb, ldq, tile0 * kTile, Nq);
  cp_async_commit();

  const int mi = lane >> 3;
  for (int j = 0; j < ntiles; ++j) {
    const int q0 = (tile0 + j) * kTile;
    bf16* Qc = (j & 1) ? Qs1 : Qs0;
    if (j + 1 < ntiles) load_tile_async<HD>((j & 1) ? Qs0 : Qs1, qb, ldq, q0 + kTile, Nq);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();

    if (q0 + warp * 16 < Nq) {
    uint32_t qf[S::KS][4];
    {
      const int row = warp * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
      for (int ks = 0; ks < S::KS; ++ks)
        ldmatrix_x4(qf[ks], static_cast<uint32_t>(__cvta_generic_to_shared(Qc + row * S::LDS + ks * 16 + (mi >> 1) * 8)));
    }
    float m_run[2] = {-INFINITY, -INFINITY};
    float l_run[2] = {0.f, 0.f};
    float oacc[S::NTO][4];
#pragma unroll
    for (int i = 0; i < S::NTO; ++i) { oacc[i][0] = oacc[i][1] = oacc[i][2] = oacc[i][3] = 0.f; }
    for (int kt = 0; kt < kv_tiles; ++kt) {
      const bf16* Kt = Ks + kt * kTile * S::LDS;
      const bf16* Vt = Vs + kt * kTile * S::LDS;
      float sacc[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { sacc[i][0] = sacc[i][1] = sacc[i][2] = sacc[i][3] = 0.f; }
#pragma unroll
      for (int ks = 0; ks < S::KS; ++ks) {
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          const int key = np * 16 + (mi >> 1) * 8 + (lane & 7);
          uint32_t kf[4];
          ldmatrix_x4(kf, static_cast<uint32_t>(__cvta_generic_to_shared(Kt + key * S::LDS + ks * 16 + (mi & 1) * 8)));
          mma_bf16_16816(sacc[np * 2], qf[ks], kf[0], kf[1]);
          mma_bf16_16816(sacc[np * 2 + 1], qf[ks], kf[2], kf[3]);
        }
      }
      float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = kt * kTile + nt * 8 + t * 2 + (e & 1);
          float sv = sacc[nt][e] * scale_log2;
          if (key >= Nkv) sv = -INFINITY;
          sacc[nt][e] = sv;
          mx[e >> 1] = fmaxf(mx[e >> 1], sv);
        }
      }
      float corr[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        const float m_new = fmaxf(m_run[r], mx[r]);  // finite: every key tile holds >= 1 valid key
        corr[r] = exp2f(m_run[r] - m_new);
        m_run[r] = m_new;
        l_run[r] *= corr[r];
      }
#pragma unroll
      for (int i = 0; i < S::NTO; ++i) {
        oacc[i][0] *= corr[0]; oacc[i][1] *= corr[0];
        oacc[i][2] *= corr[1]; oacc[i][3] *= corr[1];
      }
      uint32_t pf[4][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const float p0 = exp2f(sacc[nt][0] - m_run[0]), p1 = exp2f(sacc[nt][1] - m_run[0]);
        const float p2 = exp2f(sacc[nt][2] - m_run[1]), p3 = exp2f(sacc[nt][3] - m_run[1]);
        l_run[0] += p0 + p1;
        l_run[1] += p2 + p3;
        const int kk = nt >> 1;
        if ((nt & 1) == 0) { pf[kk][0] = pack_bf16x2(p0, p1); pf[kk][1] = pack_bf16x2(p2, p3); }
        else               { pf[kk][2] = pack_bf16x2(p0, p1); pf[kk][3] = pack_bf16x2(p2, p3); }
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
        for (int dp = 0; dp < S::NTO / 2; ++dp) {
          const int key = kk * 16 + (mi & 1) * 8 + (lane & 7);
          uint32_t vf[4];
          ldmatrix_x4_trans(vf, static_cast<uint32_t>(__cvta_generic_to_shared(Vt + key * S::LDS + (dp * 2 + (mi >> 1)) * 8)));
          mma_bf16_16816(oacc[dp * 2], pf[kk], vf[0], vf[1]);
          mma_bf16_16816(oacc[dp * 2 + 1], pf[kk], vf[2], vf[3]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
    const float inv0 = 1.0f / l_run[0], inv1 = 1.0f / l_run[1];
    __syncwarp();
#pragma unroll
    for (int i = 0; i < S::NTO; ++i) {
      const int col = i * 8 + t * 2;
      *reinterpret_cast<uint32_t*>(Qc + (warp * 16 + g) * S::LDS + col) = pack_bf16x2(oacc[i][0] * inv0, oacc[i][1] * inv0);
      *reinterpret_cast<uint32_t*>(Qc + (warp * 16 + g + 8) * S::LDS + col) = pack_bf16x2(oacc[i][2] * inv1, oacc[i][3] * inv1);
    }
    __syncwarp();
    if constexpr (HD % 8 == 0) {
      constexpr int CH = HD / 8;  // 16-byte chunks per output row
      for (int i = lane; i < 16 * CH; i += 32) {
        const int r = i / CH, c = i % CH;
        const int row = q0 + warp * 16 + r;
        if (row < Nq)
          *reinterpret_cast<uint4*>(ob + static_cast<int64_t>(row) * ldo + c * 8) = *reinterpret_cast<const uint4*>(Qc + (warp * 16 + r) * S::LDS + c * 8);
      }
    } else {
      constexpr int CH = HD / 4;  // 8-byte chunks
      for (int i = lane; i < 16 * CH; i += 32) {
        const int r = i / CH, c = i % CH;
        const int row = q0 + warp * 16 + r;
        if (row < Nq)
          *reinterpret_cast<uint2*>(ob + static_cast<int64_t>(row) * ldo + c * 4) = *reinterpret_cast<const uint2*>(Qc + (warp * 16 + r) * S::LDS + c * 4);
      }
    }
    }
    __syncthreads();
  }
  cp_async_wait<0>();
}

// the kernel launch_attention runs for these operands (SV_ATTN_*, include/surgvid.h)
int attention_kernel_for(int hd, int Nkv, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, const void* q, const void* k, const void* v,
                         const void* o) {
  if (attention_tc_enabled() && attention_tc_supported(hd, Nkv, ldq, ldk, ldv, ldo, q, k, v, o))
    return Nkv <= kTile ? SV_ATTN_TC_SINGLE : SV_ATTN_TC_MULTI;
  // the resident kernels store 16-byte chunks of output rows (heads of 20 columns stay 8-byte aligned under these)
  const bool o16 = ldo % 8 == 0 && (reinterpret_cast<uintptr_t>(o) & 15) == 0;
  if (o16 && Nkv <= kTile) return SV_ATTN_RESIDENT;
  if (o16 && Nkv <= 4 * kTile) return SV_ATTN_RESIDENT_MULTI;
  return SV_ATTN_STREAM;
}

template <int HD>
int attn_launch(int kernel, const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, const bf16* v, int64_t ldv, bf16* o, int64_t ldo, int B,
                int heads, int Nq, int Nkv, float scale, cudaStream_t st) {
  const float scale_log2 = scale * 1.4426950408889634f;
  const int qtiles = ceil_div(Nq, kTile);
  if (kernel == SV_ATTN_RESIDENT) {
    // enough CTAs to fill the machine a few times over, but as many query tiles per CTA as that allows (K/V loaded once per CTA)
    int tpc = 1;
    while (tpc < 8 && tpc < qtiles && static_cast<long long>(ceil_div(qtiles, tpc * 2)) * heads * B >= 4LL * 148 * 4) tpc *= 2;
    if (qtiles <= 4) tpc = qtiles;
    dim3 grid(ceil_div(qtiles, tpc), heads, B);
    attention_resident_kv_kernel<HD><<<grid, 128, 0, st>>>(q, ldq, k, ldk, v, ldv, o, ldo, Nq, Nkv, scale_log2, tpc);
    return launch_status("attention_resident_kv_kernel");
  }
  if (kernel == SV_ATTN_RESIDENT_MULTI) {
    using S = AttnShape<HD>;
    const int kv_tiles = ceil_div(Nkv, kTile);
    const int smem = (2 + 2 * kv_tiles) * kTile * S::LDS * static_cast<int>(sizeof(bf16));
    SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(attention_resident_multi_kernel<HD>), (2 + 2 * 4) * kTile * S::LDS * static_cast<int>(sizeof(bf16))));
    const int tpc = std::min(qtiles, 8);
    dim3 grid(ceil_div(qtiles, tpc), heads, B);
    attention_resident_multi_kernel<HD><<<grid, 128, smem, st>>>(q, ldq, k, ldk, v, ldv, o, ldo, Nq, Nkv, scale_log2, tpc, kv_tiles);
    return launch_status("attention_resident_multi_kernel");
  }
  dim3 grid(qtiles, heads, B);
  attention_kernel<HD><<<grid, 128, 0, st>>>(q, ldq, k, ldk, v, ldv, o, ldo, Nq, Nkv, scale_log2);
  return launch_status("attention_kernel");
}

}  // namespace

int launch_attention(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, const bf16* v, int64_t ldv, bf16* o, int64_t ldo, int B,
                     int heads, int Nq, int Nkv, int hd, float scale, cudaStream_t st) {
  SV_CHECK(B > 0 && heads > 0 && Nq > 0 && Nkv > 0, "attention dims");
  SV_CHECK(B <= 65535 && heads <= 65535, "attention grid limits");
  SV_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 2 == 0, "attention leading dims must keep 16-byte row alignment");
  SV_CHECK(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 15) == 0, "attention operand alignment");
  SV_CHECK((reinterpret_cast<uintptr_t>(o) & 3) == 0, "attention output must be 4-byte aligned (the kernels store bf16 pairs)");
  const int kernel = attention_kernel_for(hd, Nkv, ldq, ldk, ldv, ldo, q, k, v, o);
  if (kernel == SV_ATTN_TC_SINGLE || kernel == SV_ATTN_TC_MULTI) {
    AttnTcPlan plan;
    SV_TRY(attention_tc_plan(q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, scale, &plan));
    return attention_tc_launch(plan, st);
  }
  switch (hd) {
    case 20: return attn_launch<20>(kernel, q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, scale, st);
    case 32: return attn_launch<32>(kernel, q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, scale, st);
    case 40: return attn_launch<40>(kernel, q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, scale, st);
    case 64: return attn_launch<64>(kernel, q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, scale, st);
    default: return fail(SV_ERR_UNSUPPORTED, "attention head_dim must be 20, 32, 40 or 64");
  }
}

}  // namespace sv

extern "C" int sv_op_attention(const uint16_t* q, int64_t ldq, const uint16_t* k, int64_t ldk, const uint16_t* v, int64_t ldv, uint16_t* o,
                               int64_t ldo, int32_t B, int32_t heads, int32_t Nq, int32_t Nkv, int32_t hd, float scale, void* stream) {
  return sv::launch_attention(reinterpret_cast<const sv::bf16*>(q), ldq, reinterpret_cast<const sv::bf16*>(k), ldk,
                              reinterpret_cast<const sv::bf16*>(v), ldv, reinterpret_cast<sv::bf16*>(o), ldo, B, heads, Nq, Nkv, hd, scale,
                              static_cast<cudaStream_t>(stream));
}

extern "C" int sv_op_attention_kernel(const uint16_t* q, int64_t ldq, const uint16_t* k, int64_t ldk, const uint16_t* v, int64_t ldv,
                                      const uint16_t* o, int64_t ldo, int32_t Nkv, int32_t hd) {
  return sv::attention_kernel_for(hd, Nkv, ldq, ldk, ldv, ldo, q, k, v, o);
}
