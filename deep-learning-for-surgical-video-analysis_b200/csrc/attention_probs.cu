// Post-softmax attention maps P = softmax(Q K^T * scale) of the encoder blocks (mix_transformer_evp.py:123-125, the `attn` tensor the
// reference's `get_local('attn')` records), written to a contiguous fp32 [B, heads, Nq, Nkv] array.
//
// The kernel is bound by its stores (2*hd FLOP per 4-byte output), so S = Q K^T runs on tensor cores: mma.sync m16n8k16, one warp =
// 16 query rows, one CTA = 64 rows of one (frame, head), keys in 64-key chunks through shared memory.  N_kv <= 64 (every block at 224^2):
// one chunk, the exponentials stay in registers and are scaled by 1/rowsum.  N_kv > 64: pass 1 computes row max and row sum over all
// chunks (online rescaling), pass 2 recomputes each chunk and writes exp2(s - max) / sum.  A warp's rows go through a per-warp shared
// tile so that the stores are coalesced: with one chunk the warp's 16 rows are one contiguous run of the output (rows are N_kv * 4 bytes,
// not 16-byte multiples, so the tile is placed at the output's alignment and copied with 16-byte stores); with several chunks each row
// segment is written by consecutive lanes.
#include "kernels.cuh"

namespace sv {

namespace {

constexpr int kProbRows = 64;      // query rows per CTA (16 per warp)
constexpr int kProbKeys = 64;      // keys per chunk
constexpr int kStageLd = 72;       // row stride of a multi-chunk staging tile (floats): float2 fragment stores without bank conflicts
constexpr int kStageFloats = 16 * kStageLd;  // >= 16 * 64 + 3 (single chunk: 16 contiguous rows, shifted by up to 3 floats)

__device__ __forceinline__ void probs_ldmatrix_x4(uint32_t (&r)[4], const void* p) {
  const uint32_t addr = static_cast<uint32_t>(__cvta_generic_to_shared(p));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void probs_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows [r0, r0+64) x HD columns of a bf16 matrix -> smem [64][HD+8], rows past rows_total zero-filled
template <int HD>
__device__ __forceinline__ void probs_load_rows(bf16* __restrict__ dst, const bf16* __restrict__ src, int64_t ld, int r0, int rows_total) {
  constexpr int CH = HD / 8;
  for (int i = threadIdx.x; i < 64 * CH; i += blockDim.x) {
    const int r = i / CH, c = i % CH;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r0 + r < rows_total) v = __ldg(reinterpret_cast<const uint4*>(src + static_cast<int64_t>(r0 + r) * ld + c * 8));
    *reinterpret_cast<uint4*>(dst + r * (HD + 8) + c * 8) = v;
  }
}

// s = (Q K^T) * scale_log2 of this warp's 16 rows against the 64 keys in Ks (keys >= Nkv - c0 masked to -inf)
template <int HD>
__device__ __forceinline__ void probs_scores(float (&s)[8][4], const uint32_t (&qf)[HD / 16][4], const bf16* Ks, int lane, int kv_left,
                                             float scale_log2) {
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
  const int mi = lane >> 3;
#pragma unroll
  for (int ks = 0; ks < HD / 16; ++ks) {
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t kf[4];
      probs_ldmatrix_x4(kf, Ks + (np * 16 + (mi >> 1) * 8 + (lane & 7)) * (HD + 8) + ks * 16 + (mi & 1) * 8);
      probs_mma(s[np * 2], qf[ks], kf[0], kf[1]);
      probs_mma(s[np * 2 + 1], qf[ks], kf[2], kf[3]);
    }
  }
  const int t = lane & 3;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int e = 0; e < 4; ++e) s[nt][e] = nt * 8 + t * 2 + (e & 1) < kv_left ? s[nt][e] * scale_log2 : -INFINITY;
}

template <int HD>
__global__ void __launch_bounds__(128) attention_probs_kernel(const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ k, int64_t ldk,
                                                              float* __restrict__ p, int Nq, int Nkv, float scale_log2) {
  __shared__ __align__(16) bf16 Qs[kProbRows * (HD + 8)];
  __shared__ __align__(16) bf16 Ks[kProbKeys * (HD + 8)];
  __shared__ __align__(16) float stage_all[4][kStageFloats];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int head = blockIdx.y, b = blockIdx.z;
  const int row0 = blockIdx.x * kProbRows + warp * 16;  // this warp's first query row
  const bf16* qb = q + static_cast<int64_t>(b) * Nq * ldq + head * HD;
  const bf16* kb = k + static_cast<int64_t>(b) * Nkv * ldk + head * HD;
  // element offsets pass 2^31 at 480x854 from B = 19 on: 64-bit throughout
  float* out0 = p + ((static_cast<int64_t>(b) * gridDim.y + head) * Nq + row0) * Nkv;
  const int rows = min(16, Nq - row0);  // <= 0: a warp past the last query row (it still takes part in the CTA's barriers)
  const int nchunks = (Nkv + kProbKeys - 1) / kProbKeys;

  probs_load_rows<HD>(Qs, qb, ldq, blockIdx.x * kProbRows, Nq);
  if (nchunks == 1) probs_load_rows<HD>(Ks, kb, ldk, 0, Nkv);
  __syncthreads();

  uint32_t qf[HD / 16][4];
  {
    const int mi = lane >> 3;
#pragma unroll
    for (int ks = 0; ks < HD / 16; ++ks)
      probs_ldmatrix_x4(qf[ks], Qs + (warp * 16 + (mi & 1) * 8 + (lane & 7)) * (HD + 8) + ks * 16 + (mi >> 1) * 8);
  }

  // pass 1: row max and row sum (rows g and g + 8 of the warp's 16; each quad of lanes shares a row)
  float s[8][4];
  float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
  for (int c = 0; c < nchunks; ++c) {
    if (nchunks > 1) {
      __syncthreads();
      probs_load_rows<HD>(Ks, kb, ldk, c * kProbKeys, Nkv);
      __syncthreads();
    }
    probs_scores<HD>(s, qf, Ks, lane, Nkv - c * kProbKeys, scale_log2);
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) mx[e >> 1] = fmaxf(mx[e >> 1], s[nt][e]);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float m_new = fmaxf(m[r], mx[r]);  // finite: every chunk holds >= 1 valid key
      l[r] *= exp2f(m[r] - m_new);
      m[r] = m_new;
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float x = exp2f(s[nt][e] - m[e >> 1]);
        l[e >> 1] += x;
        if (nchunks == 1) s[nt][e] = x;  // the max is final: keep the exponentials for pass 2
      }
  }
  float inv[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l[r] += __shfl_xor_sync(0xffffffffu, l[r], 1);
    l[r] += __shfl_xor_sync(0xffffffffu, l[r], 2);
    inv[r] = 1.f / l[r];
  }

  // pass 2: normalise, stage, store
  float* st = stage_all[warp];
  if (nchunks == 1) {
    // the warp's rows are out0[0, rows * Nkv): stage them at out0's offset within 16 bytes, copy with aligned 16-byte stores
    const int sh = static_cast<int>((reinterpret_cast<uintptr_t>(out0) >> 2) & 3);
    float* sb = st + sh;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int col = nt * 8 + t * 2 + (e & 1);
        if (col < Nkv) sb[(g + (e >> 1) * 8) * Nkv + col] = s[nt][e] * inv[e >> 1];
      }
    __syncwarp();
    if (rows > 0) {
      const int T = rows * Nkv;
      const int lead = min(T, (4 - sh) & 3);
      if (lane < lead) __stcs(out0 + lane, sb[lane]);
      const int nvec = (T - lead) >> 2;
      const float4* sv = reinterpret_cast<const float4*>(sb + lead);
      float4* dv = reinterpret_cast<float4*>(out0 + lead);
      for (int i = lane; i < nvec; i += 32) __stcs(dv + i, sv[i]);
      const int done = lead + nvec * 4;
      if (done + lane < T) __stcs(out0 + done + lane, sb[done + lane]);
    }
    return;
  }
  for (int c = 0; c < nchunks; ++c) {
    const int c0 = c * kProbKeys, w = min(kProbKeys, Nkv - c0);
    __syncthreads();
    probs_load_rows<HD>(Ks, kb, ldk, c0, Nkv);
    __syncthreads();
    probs_scores<HD>(s, qf, Ks, lane, w, scale_log2);
    __syncwarp();  // the previous chunk's copy-out has read the staging tile
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int h = 0; h < 2; ++h)
        *reinterpret_cast<float2*>(st + (g + h * 8) * kStageLd + nt * 8 + t * 2) =
            make_float2(exp2f(s[nt][2 * h] - m[h]) * inv[h], exp2f(s[nt][2 * h + 1] - m[h]) * inv[h]);
    __syncwarp();
    for (int r = 0; r < rows; ++r)
      for (int j = lane; j < w; j += 32) __stcs(out0 + static_cast<int64_t>(r) * Nkv + c0 + j, st[r * kStageLd + j]);
  }
}

}  // namespace

int launch_attention_probs(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, int B, int heads, int Nq, int Nkv, int hd, float scale,
                           float* p, cudaStream_t st) {
  SV_CHECK(q && k && p, "attention_probs: null argument");
  SV_CHECK(B > 0 && heads > 0 && Nq > 0 && Nkv > 0, "attention_probs dims");
  SV_CHECK(B <= 65535 && heads <= 65535, "attention_probs grid limits");
  SV_CHECK(ldq % 8 == 0 && ldk % 8 == 0, "attention_probs leading dims must keep 16-byte row alignment");
  SV_CHECK(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k)) & 15) == 0, "attention_probs operand alignment");
  SV_CHECK((reinterpret_cast<uintptr_t>(p) & 3) == 0, "attention_probs output must be 4-byte aligned");
  const float scale_log2 = scale * 1.4426950408889634f;
  const dim3 grid(ceil_div(Nq, kProbRows), heads, B);
  switch (hd) {
    case 32: attention_probs_kernel<32><<<grid, 128, 0, st>>>(q, ldq, k, ldk, p, Nq, Nkv, scale_log2); break;
    case 64: attention_probs_kernel<64><<<grid, 128, 0, st>>>(q, ldq, k, ldk, p, Nq, Nkv, scale_log2); break;
    default: return fail(SV_ERR_UNSUPPORTED, "attention_probs head_dim must be 32 or 64");
  }
  return launch_status("attention_probs_kernel");
}

}  // namespace sv

extern "C" int sv_op_attention_probs(const uint16_t* q, int64_t ldq, const uint16_t* k, int64_t ldk, int32_t B, int32_t heads, int32_t Nq,
                                     int32_t Nkv, int32_t hd, float scale, float* p, void* stream) {
  return sv::launch_attention_probs(reinterpret_cast<const sv::bf16*>(q), ldq, reinterpret_cast<const sv::bf16*>(k), ldk, B, heads, Nq, Nkv,
                                    hd, scale, p, static_cast<cudaStream_t>(stream));
}
