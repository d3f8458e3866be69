// Trans-SVNet head (SURVEY.md 8f-1): the inner module of adapter_transformer.Transformer (adapter_transformer.py:317-325, 348),
//   output[t] = Transformer2_3_1(inputs[t] = the len_q-frame causal window of the MS-TCN logits ending at t, feas[t] = tanh(fc(LFB[t])))
// fused into ONE kernel that reads the channel-major MS-TCN logits and the query directly: the [T, len_q, 14] window tensor the
// reference builds with a Python loop is never materialised.
//
// The source of Transformer2_3_1 is NOT in the reference tree (SURVEY.md F7); the arithmetic here follows the published upstream
// architecture as restated in oracle/trans_head_oracle.py (PARITY UNPINNED): one encoder layer over the window (4-head self-attention,
// residual + LayerNorm, position-wise FFN with ReLU, residual + LayerNorm), one decoder layer whose single query cross-attends the
// encoder output (same blocks).  fp32 throughout (d_model = 14: nothing here is tensor-core shaped).
//
// d_k = d_v is a template parameter (32: mstcn_f_maps 32; 64: mstcn_f_maps >= 64, adapter_transformer.py:315), see HeadCfg.
//   d_k = 32: one persistent CTA = two groups of 128 threads (4 warps = 4 heads each); every group walks its own frames t with its own
//             Q/K/V tiles and named barriers, and both share the weights (86 KB, d_model padded to 16) in shared memory.
//   d_k = 64: the weights alone take 155 KB, so a CTA is one group, and it keeps no Q tile: a lane computes its window row's Q of its
//             head in registers right before the scores, and the self-attention context overwrites the head's own K columns, which no
//             other warp reads (228 936 B of shared memory in all).
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "host.cuh"
#include "kernels.cuh"

namespace sv {
namespace {

constexpr int kDP = 16;      // d_model padded
constexpr int kH = 4;        // heads
constexpr int kLMax = 32;    // len_q <= 32
constexpr int kFFMax = 64;   // d_ff <= 64

// blob layout of one FFN block (floats)
constexpr int kFfnW1 = 0, kFfnB1 = kFFMax * kDP, kFfnW2 = kFfnB1 + kFFMax, kFfnB2 = kFfnW2 + kDP * kFFMax, kFfnG = kFfnB2 + kDP, kFfnB = kFfnG + kDP,
              kFfnSize = kFfnB + kDP;

template <int DK>   // d_k = d_v
struct HeadCfg {
  static_assert(DK == 32 || DK == 64, "d_k = d_v = 32 or 64");
  static constexpr int kDK = DK;
  static constexpr int kHD = kH * kDK;
  static constexpr int kLdS = kHD + 1;  // row stride of the Q/K/V tiles (conflict-free row-wise reads)
  // blob layout of one attention block (floats)
  static constexpr int kAttnWQ = 0, kAttnBQ = kHD * kDP, kAttnWK = kAttnBQ + kHD, kAttnBK = kAttnWK + kHD * kDP, kAttnWV = kAttnBK + kHD,
                       kAttnBV = kAttnWV + kHD * kDP, kAttnWO = kAttnBV + kHD, kAttnBO = kAttnWO + kDP * kHD, kAttnG = kAttnBO + kDP,
                       kAttnB = kAttnG + kDP, kAttnSize = kAttnB + kDP;
  static constexpr int kBlobSize = 2 * (kAttnSize + kFfnSize);   // encoder attn | encoder ffn | decoder attn | decoder ffn
  static constexpr int kGroups = DK == 32 ? 2 : 1;               // 128-thread groups per CTA
  // per-group tiles: Q (d_k = 32 only), K, V [kLMax][kLdS]; X, Y, E [kLMax][kDP]; the decoder query [kDP]; d_k = 64 adds the decoder's
  // Q row and context row [2][kLdS] (d_k = 32 keeps both in the Q tile)
  static constexpr int kGroupFloats = (DK == 32 ? 3 : 2) * kLMax * kLdS + 3 * kLMax * kDP + kDP + (DK == 32 ? 0 : 2 * kLdS);
  static constexpr int kSmemBytes = (kBlobSize + kGroups * kGroupFloats) * static_cast<int>(sizeof(float));
};
static_assert(HeadCfg<32>::kSmemBytes <= 227 * 1024 && HeadCfg<64>::kSmemBytes <= 227 * 1024, "shared memory per block");

struct TransParams {
  int D, L, FF, n_videos;
  float scale;   // 1 / sqrt(d_k)
};

__device__ __forceinline__ void layer_norm_inplace(float (&v)[kDP], int D, const float* g, const float* b) {
  float m = 0.f;
#pragma unroll
  for (int c = 0; c < kDP; ++c) m += (c < D) ? v[c] : 0.f;
  m /= static_cast<float>(D);
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < kDP; ++c) { const float d = (c < D) ? v[c] - m : 0.f; q += d * d; }
  const float r = rsqrtf(q / static_cast<float>(D) + 1e-5f);
#pragma unroll
  for (int c = 0; c < kDP; ++c) v[c] = (c < D) ? (v[c] - m) * r * g[c] + b[c] : 0.f;
}

__device__ __forceinline__ void group_sync(int grp) { asm volatile("bar.sync %0, 128;" ::"r"(grp + 1) : "memory"); }

// Where a window row that precedes its video's (or stream chunk's) first frame in `logits` comes from.
//   OfflineWindow: logits hold whole videos, so such a row is the zero left padding.
//   StreamWindow:  logits hold one step of the streams (chunk k = stream ids[k], frames seen[s] .. seen[s]+count-1); a row at stream
//                  position q >= 0 comes from the stream's ring of the last len_q - 1 logits rows (slot q mod (len_q - 1)), q < 0 is zero.
struct OfflineWindow {
  static constexpr bool kStream = false;
};
struct StreamWindow {
  static constexpr bool kStream = true;
  const int64_t* __restrict__ ids;     // [n_ids] stream of each chunk
  const int64_t* __restrict__ seen;    // [n_streams]
  const float* __restrict__ ring;      // [n_streams][len_q - 1][D]
};

template <int DK, class Window>
__global__ void __launch_bounds__(128 * HeadCfg<DK>::kGroups) trans_head_kernel(const float* __restrict__ logits, int64_t ldx, const float* __restrict__ query,
                                                         const int64_t* __restrict__ offsets, int64_t T, const float* __restrict__ blob,
                                                         float* __restrict__ out, const TransParams p, const Window win) {
  using C = HeadCfg<DK>;
  constexpr int kDK = C::kDK, kHD = C::kHD, kLdS = C::kLdS, kGroups = C::kGroups, kBlobSize = C::kBlobSize;
  constexpr int kAttnWQ = C::kAttnWQ, kAttnBQ = C::kAttnBQ, kAttnWK = C::kAttnWK, kAttnBK = C::kAttnBK, kAttnWV = C::kAttnWV, kAttnBV = C::kAttnBV,
                kAttnWO = C::kAttnWO, kAttnBO = C::kAttnBO, kAttnG = C::kAttnG, kAttnB = C::kAttnB, kAttnSize = C::kAttnSize;
  extern __shared__ __align__(16) float sm[];
  float* Wb = sm;                              // kBlobSize
  const int grp = threadIdx.x >> 7;
  float* Qs = Wb + kBlobSize + grp * C::kGroupFloats;   // d_k = 32: [kLMax][kLdS]  Q, then the attention context
  float* Ks = Qs + (DK == 32 ? kLMax * kLdS : 0);       // d_k = 64: the attention context overwrites K (head h's columns by warp h)
  float* Vs = Ks + kLMax * kLdS;
  float* Xs = Vs + kLMax * kLdS;               // [kLMax][kDP]  window
  float* Ys = Xs + kLMax * kDP;                // [kLMax][kDP]
  float* Es = Ys + kLMax * kDP;                // [kLMax][kDP]  encoder output
  float* qv = Es + kLMax * kDP;                // [kDP] decoder query
  float* Cs = DK == 32 ? Qs : Ks;              // self-attention context [kLMax][kLdS]
  float* Qd = DK == 32 ? Qs : qv + kDP;        // decoder: row 0 its Q, row 1 the cross-attention context
  const int tid = threadIdx.x & 127, warp = tid >> 5, lane = tid & 31;
  const int D = p.D, L = p.L, FF = p.FF;
  for (int i = threadIdx.x; i < kBlobSize / 4; i += 128 * kGroups) reinterpret_cast<float4*>(Wb)[i] = __ldg(reinterpret_cast<const float4*>(blob) + i);
  const float* EA = Wb;
  const float* EF = EA + kAttnSize;
  const float* DA = EF + kFfnSize;
  const float* DF = DA + kAttnSize;
  __syncthreads();

  for (int64_t t = static_cast<int64_t>(blockIdx.x) * kGroups + grp; t < T; t += static_cast<int64_t>(gridDim.x) * kGroups) {
    // first frame of t's video (zero left padding of the window never crosses a video boundary, adapter_transformer.py:336-341)
    int lo = 0, hi = p.n_videos;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (offsets[mid] <= t) lo = mid; else hi = mid;
    }
    const int64_t start = offsets[lo];
    // ---- (1) window X [L, D] and the decoder query
    if constexpr (Window::kStream) {
      const int64_t s = win.ids[lo], pos = win.seen[s] + (t - start);   // stream position of frame t
      for (int idx = tid; idx < L * kDP; idx += 128) {
        const int i = idx / kDP, c = idx % kDP;
        const int64_t src = t - (L - 1) + i, q = pos - (L - 1) + i;
        float v = 0.f;
        if (c < D && src >= start) v = __ldg(logits + static_cast<int64_t>(c) * ldx + src);
        else if (c < D && q >= 0) v = __ldg(win.ring + (s * (L - 1) + q % (L - 1)) * D + c);
        Xs[idx] = v;
      }
    } else {
      for (int idx = tid; idx < L * kDP; idx += 128) {
        const int i = idx / kDP, c = idx % kDP;
        const int64_t src = t - (L - 1) + i;
        Xs[idx] = (c < D && src >= start) ? __ldg(logits + static_cast<int64_t>(c) * ldx + src) : 0.f;
      }
    }
    if (tid < kDP) qv[tid] = tid < D ? __ldg(query + t * D + tid) : 0.f;
    group_sync(grp);
    if constexpr (DK == 32) {
      // ---- (2) encoder Q, K, V: thread = one of the 128 projection columns
      {
        float wq[kDP], wk[kDP], wv[kDP];
#pragma unroll
        for (int c = 0; c < kDP; ++c) { wq[c] = EA[kAttnWQ + tid * kDP + c]; wk[c] = EA[kAttnWK + tid * kDP + c]; wv[c] = EA[kAttnWV + tid * kDP + c]; }
        const float bq = EA[kAttnBQ + tid], bk = EA[kAttnBK + tid], bv = EA[kAttnBV + tid];
        for (int i = 0; i < L; ++i) {
          float q = bq, k = bk, v = bv;
#pragma unroll
          for (int c = 0; c < kDP; ++c) { const float x = Xs[i * kDP + c]; q = fmaf(x, wq[c], q); k = fmaf(x, wk[c], k); v = fmaf(x, wv[c], v); }
          Qs[i * kLdS + tid] = q; Ks[i * kLdS + tid] = k; Vs[i * kLdS + tid] = v;
        }
      }
      group_sync(grp);
      // ---- (3) self-attention: warp = head, lane = query row
      if (lane < L) {
        float q[kDK];
#pragma unroll
        for (int d = 0; d < kDK; ++d) q[d] = Qs[lane * kLdS + warp * kDK + d];
        float s[kLMax];
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < kLMax; ++j) {
          float a = 0.f;
          if (j < L) {
#pragma unroll
            for (int d = 0; d < kDK; ++d) a = fmaf(q[d], Ks[j * kLdS + warp * kDK + d], a);
            a *= p.scale;
            m = fmaxf(m, a);
          }
          s[j] = a;
        }
        float den = 0.f;
#pragma unroll
        for (int j = 0; j < kLMax; ++j) { s[j] = (j < L) ? __expf(s[j] - m) : 0.f; den += s[j]; }
        const float inv = 1.0f / den;
        float ctx[kDK];
#pragma unroll
        for (int d = 0; d < kDK; ++d) ctx[d] = 0.f;
#pragma unroll
        for (int j = 0; j < kLMax; ++j) {
          if (j < L) {
            const float pj = s[j] * inv;
#pragma unroll
            for (int d = 0; d < kDK; ++d) ctx[d] = fmaf(pj, Vs[j * kLdS + warp * kDK + d], ctx[d]);
          }
        }
#pragma unroll
        for (int d = 0; d < kDK; ++d) Qs[lane * kLdS + warp * kDK + d] = ctx[d];   // only this lane ever read this Q row
      }
    } else {
      // ---- (2) encoder K, V: thread = projection columns tid and tid + 128
#pragma unroll 1
      for (int col = tid; col < kHD; col += 128) {
        float wk[kDP], wv[kDP];
#pragma unroll
        for (int c = 0; c < kDP; ++c) { wk[c] = EA[kAttnWK + col * kDP + c]; wv[c] = EA[kAttnWV + col * kDP + c]; }
        const float bk = EA[kAttnBK + col], bv = EA[kAttnBV + col];
        for (int i = 0; i < L; ++i) {
          float k = bk, v = bv;
#pragma unroll
          for (int c = 0; c < kDP; ++c) { const float x = Xs[i * kDP + c]; k = fmaf(x, wk[c], k); v = fmaf(x, wv[c], v); }
          Ks[i * kLdS + col] = k; Vs[i * kLdS + col] = v;
        }
      }
      group_sync(grp);
      // ---- (3) self-attention: warp = head, lane = query row (lanes past L repeat row L - 1 and store nothing)
      {
        const int r = lane < L ? lane : L - 1;
        float s[kLMax];
        float m = -INFINITY;
        {
          float x[kDP];
#pragma unroll
          for (int c = 0; c < kDP; ++c) x[c] = Xs[r * kDP + c];
          float q[kDK];   // this row's Q of head `warp`, summed in the order of the projection above
#pragma unroll
          for (int d = 0; d < kDK; ++d) {
            const int col = warp * kDK + d;
            float a = EA[kAttnBQ + col];
#pragma unroll
            for (int c = 0; c < kDP; ++c) a = fmaf(x[c], EA[kAttnWQ + col * kDP + c], a);
            q[d] = a;
          }
#pragma unroll
          for (int j = 0; j < kLMax; ++j) {
            float a = 0.f;
            if (j < L) {
#pragma unroll
              for (int d = 0; d < kDK; ++d) a = fmaf(q[d], Ks[j * kLdS + warp * kDK + d], a);
              a *= p.scale;
              m = fmaxf(m, a);
            }
            s[j] = a;
          }
        }
        float den = 0.f;
#pragma unroll
        for (int j = 0; j < kLMax; ++j) { s[j] = (j < L) ? __expf(s[j] - m) : 0.f; den += s[j]; }
        const float inv = 1.0f / den;
        float ctx[kDK];
#pragma unroll
        for (int d = 0; d < kDK; ++d) ctx[d] = 0.f;
#pragma unroll
        for (int j = 0; j < kLMax; ++j) {
          if (j < L) {
            const float pj = s[j] * inv;
#pragma unroll
            for (int d = 0; d < kDK; ++d) ctx[d] = fmaf(pj, Vs[j * kLdS + warp * kDK + d], ctx[d]);
          }
        }
        __syncwarp();   // every lane of this head is done reading its K columns
        if (lane < L) {
#pragma unroll
          for (int d = 0; d < kDK; ++d) Cs[lane * kLdS + warp * kDK + d] = ctx[d];
        }
      }
    }
    group_sync(grp);
    // ---- (4) output projection + residual: warp = group of 4 channels, lane = row
    if (lane < L) {
      float acc[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { const int c = warp * 4 + u; acc[u] = (c < D) ? EA[kAttnBO + c] + Xs[lane * kDP + c] : 0.f; }
      for (int k = 0; k < kHD; ++k) {
        const float cv = Cs[lane * kLdS + k];
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[u] = fmaf(cv, EA[kAttnWO + (warp * 4 + u) * kHD + k], acc[u]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) Ys[lane * kDP + warp * 4 + u] = acc[u];
    }
    group_sync(grp);
    // ---- LayerNorm, FFN, LayerNorm per row (warp 0, lane = row)
    if (warp == 0 && lane < L) {
      float y[kDP];
#pragma unroll
      for (int c = 0; c < kDP; ++c) y[c] = Ys[lane * kDP + c];
      layer_norm_inplace(y, D, EA + kAttnG, EA + kAttnB);
      float o[kDP];
#pragma unroll
      for (int c = 0; c < kDP; ++c) o[c] = (c < D) ? EF[kFfnB2 + c] + y[c] : 0.f;
      for (int mm = 0; mm < FF; ++mm) {
        float h = EF[kFfnB1 + mm];
#pragma unroll
        for (int c = 0; c < kDP; ++c) h = fmaf(y[c], EF[kFfnW1 + mm * kDP + c], h);
        h = fmaxf(h, 0.f);
#pragma unroll
        for (int c = 0; c < kDP; ++c) o[c] = fmaf(h, EF[kFfnW2 + c * kFFMax + mm], o[c]);
      }
      layer_norm_inplace(o, D, EF + kFfnG, EF + kFfnB);
#pragma unroll
      for (int c = 0; c < kDP; ++c) Es[lane * kDP + c] = o[c];
    }
    group_sync(grp);
    // ---- (5) decoder: K, V of the encoder output, Q of the query: thread = projection column (d_k = 64: columns tid and tid + 128)
#pragma unroll 1
    for (int col = tid; col < kHD; col += 128) {
      float wk[kDP], wv[kDP];
      float qd = DA[kAttnBQ + col];
#pragma unroll
      for (int c = 0; c < kDP; ++c) {
        wk[c] = DA[kAttnWK + col * kDP + c]; wv[c] = DA[kAttnWV + col * kDP + c];
        qd = fmaf(qv[c], DA[kAttnWQ + col * kDP + c], qd);
      }
      const float bk = DA[kAttnBK + col], bv = DA[kAttnBV + col];
      for (int i = 0; i < L; ++i) {
        float k = bk, v = bv;
#pragma unroll
        for (int c = 0; c < kDP; ++c) { const float e = Es[i * kDP + c]; k = fmaf(e, wk[c], k); v = fmaf(e, wv[c], v); }
        Ks[i * kLdS + col] = k; Vs[i * kLdS + col] = v;
      }
      Qd[col] = qd;   // row 0 of Qd
    }
    group_sync(grp);
    {  // cross-attention: warp = head, lane = key; softmax across the warp; context: lane = channel of the head (d_k = 64: two)
      float a = -INFINITY;
      if (lane < L) {
        a = 0.f;
#pragma unroll
        for (int d = 0; d < kDK; ++d) a = fmaf(Qd[warp * kDK + d], Ks[lane * kLdS + warp * kDK + d], a);
        a *= p.scale;
      }
      const float m = warp_max(a);
      const float e = (lane < L) ? __expf(a - m) : 0.f;
      const float pj = e / warp_sum(e);
#pragma unroll
      for (int d0 = 0; d0 < kDK; d0 += 32) {
        float ctx = 0.f;
        for (int j = 0; j < L; ++j) ctx = fmaf(__shfl_sync(0xffffffffu, pj, j), Vs[j * kLdS + warp * kDK + d0 + lane], ctx);
        __syncwarp();
        Qd[kLdS + warp * kDK + d0 + lane] = ctx;   // row 1 of Qd
      }
    }
    group_sync(grp);
    if (warp == 0) {  // output projection + residual + LayerNorm + FFN + LayerNorm for the single decoder row: lane = channel
      float o = 0.f;
      if (lane < D) {
        o = DA[kAttnBO + lane] + qv[lane];
        for (int k = 0; k < kHD; ++k) o = fmaf(Qd[kLdS + k], DA[kAttnWO + lane * kHD + k], o);
      }
      const float fD = static_cast<float>(D);
      float mean = warp_sum(lane < D ? o : 0.f) / fD;
      float dv = lane < D ? o - mean : 0.f;
      float rstd = rsqrtf(warp_sum(dv * dv) / fD + 1e-5f);
      const float dn = lane < D ? dv * rstd * DA[kAttnG + lane] + DA[kAttnB + lane] : 0.f;
      // FFN: lane = hidden unit (two per lane when d_ff > 32)
      float h0 = 0.f, h1 = 0.f;
      {
        float a0 = lane < FF ? DF[kFfnB1 + lane] : 0.f, a1 = lane + 32 < FF ? DF[kFfnB1 + lane + 32] : 0.f;
        for (int c = 0; c < D; ++c) {
          const float dc = __shfl_sync(0xffffffffu, dn, c);
          if (lane < FF) a0 = fmaf(dc, DF[kFfnW1 + lane * kDP + c], a0);
          if (lane + 32 < FF) a1 = fmaf(dc, DF[kFfnW1 + (lane + 32) * kDP + c], a1);
        }
        h0 = lane < FF ? fmaxf(a0, 0.f) : 0.f;
        h1 = lane + 32 < FF ? fmaxf(a1, 0.f) : 0.f;
      }
      float o2 = lane < D ? DF[kFfnB2 + lane] + dn : 0.f;
      for (int mm = 0; mm < 32; ++mm) {
        const float ha = __shfl_sync(0xffffffffu, h0, mm), hb = __shfl_sync(0xffffffffu, h1, mm);
        if (lane < D) {
          o2 = fmaf(ha, DF[kFfnW2 + lane * kFFMax + mm], o2);
          o2 = fmaf(hb, DF[kFfnW2 + lane * kFFMax + mm + 32], o2);
        }
      }
      mean = warp_sum(lane < D ? o2 : 0.f) / fD;
      dv = lane < D ? o2 - mean : 0.f;
      rstd = rsqrtf(warp_sum(dv * dv) / fD + 1e-5f);
      if (lane < D) out[t * D + lane] = dv * rstd * DF[kFfnG + lane] + DF[kFfnB + lane];
    }
    group_sync(grp);   // the tiles are rewritten by the next frame
  }
}

// After a stream step: the last min(len_q - 1, count) logits rows of every chunk go to their ring slots, then seen advances.
// One block per chunk; the block reads seen[s] before its thread 0 advances it.
__global__ void trans_stream_commit_kernel(const float* __restrict__ logits, int64_t ldx, const int64_t* __restrict__ tab, int n_ids, int D, int L,
                                           float* __restrict__ ring, int64_t* __restrict__ seen) {
  const int k = blockIdx.x;
  const int64_t s = tab[n_ids + 1 + k], r0 = tab[k], cnt = tab[k + 1] - r0, seen0 = seen[s], keep = cnt < L - 1 ? cnt : L - 1;
  for (int64_t i = threadIdx.x; i < keep * D; i += blockDim.x) {
    const int64_t j = cnt - keep + i / D;   // row in the chunk
    const int c = static_cast<int>(i % D);
    ring[(s * (L - 1) + (seen0 + j) % (L - 1)) * D + c] = __ldg(logits + static_cast<int64_t>(c) * ldx + r0 + j);
  }
  __syncthreads();
  if (threadIdx.x == 0) seen[s] = seen0 + cnt;
}

}  // namespace
}  // namespace sv

struct sv_trans {
  sv_trans_cfg cfg;
  int device = 0;
  sv::StateDict sd;
  float* d_blob = nullptr;
  int64_t* d_offsets = nullptr;
  int offsets_cap = 0;
  sv::StreamRegistry streams{"trans stream"};
};

namespace sv {
namespace {

// nn.Linear weight [rows, cols] (+ optional bias [rows]) -> blob[w_off + r * ld + c], blob[b_off + r]
int put_linear(const sv_trans* h, const std::string& p, int rows, int cols, int ld, std::vector<float>* blob, int w_off, int b_off) {
  const HostTensor* w;
  SV_TRY(h->sd.get(p + ".weight", {rows, cols}, "trans", &w));
  for (int r = 0; r < rows; ++r)
    for (int c = 0; c < cols; ++c) (*blob)[w_off + r * ld + c] = w->data[static_cast<size_t>(r) * cols + c];
  if (h->sd.tensors.count(p + ".bias")) {   // bias-free variants of the upstream code: treated as zero
    const HostTensor* b;
    SV_TRY(h->sd.get(p + ".bias", {rows}, "trans", &b));
    for (int r = 0; r < rows; ++r) (*blob)[b_off + r] = b->data[r];
  }
  return SV_OK;
}
int put_norm(const sv_trans* h, const std::string& p, int D, std::vector<float>* blob, int g_off, int b_off) {
  const HostTensor *g, *b;
  SV_TRY(h->sd.get(p + ".weight", {D}, "trans", &g));
  SV_TRY(h->sd.get(p + ".bias", {D}, "trans", &b));
  for (int c = 0; c < D; ++c) { (*blob)[g_off + c] = g->data[c]; (*blob)[b_off + c] = b->data[c]; }
  return SV_OK;
}

template <int DK>
int pack_blob(const sv_trans* h, std::vector<float>* blob) {
  using C = HeadCfg<DK>;
  const int D = h->cfg.d_model, FF = h->cfg.d_ff;
  blob->assign(C::kBlobSize, 0.f);
  const char* attn_name[2] = {"encoder.layers.0.enc_self_attn", "decoder.layers.0.dec_enc_attn"};
  const char* ffn_name[2] = {"encoder.layers.0.pos_ffn", "decoder.layers.0.pos_ffn"};
  for (int s = 0; s < 2; ++s) {
    const int a0 = s * (C::kAttnSize + kFfnSize), f0 = a0 + C::kAttnSize;
    const std::string ap = attn_name[s], fp = ffn_name[s];
    SV_TRY(put_linear(h, ap + ".W_Q", C::kHD, D, kDP, blob, a0 + C::kAttnWQ, a0 + C::kAttnBQ));
    SV_TRY(put_linear(h, ap + ".W_K", C::kHD, D, kDP, blob, a0 + C::kAttnWK, a0 + C::kAttnBK));
    SV_TRY(put_linear(h, ap + ".W_V", C::kHD, D, kDP, blob, a0 + C::kAttnWV, a0 + C::kAttnBV));
    SV_TRY(put_linear(h, ap + ".fc", D, C::kHD, C::kHD, blob, a0 + C::kAttnWO, a0 + C::kAttnBO));
    SV_TRY(put_norm(h, ap + ".layer_norm", D, blob, a0 + C::kAttnG, a0 + C::kAttnB));
    SV_TRY(put_linear(h, fp + ".fc1", FF, D, kDP, blob, f0 + kFfnW1, f0 + kFfnB1));
    SV_TRY(put_linear(h, fp + ".fc2", D, FF, kFFMax, blob, f0 + kFfnW2, f0 + kFfnB2));
    SV_TRY(put_norm(h, fp + ".layer_norm", D, blob, f0 + kFfnG, f0 + kFfnB));
  }
  return SV_OK;
}

// One launch of the head kernel over T rows: a persistent grid of at most one CTA per SM, kGroups rows in flight per CTA.
template <int DK, class Window>
int launch_head(const float* logits, int64_t ldx, const float* query, const int64_t* offsets, int64_t T, const float* blob, float* out,
                const TransParams& p, const Window& win, cudaStream_t st) {
  using C = HeadCfg<DK>;
  SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(trans_head_kernel<DK, Window>), C::kSmemBytes));
  const int grid = static_cast<int>(std::min<int64_t>((T + C::kGroups - 1) / C::kGroups, std::max(1, device_sm_count())));
  trans_head_kernel<DK, Window><<<grid, 128 * C::kGroups, C::kSmemBytes, st>>>(logits, ldx, query, offsets, T, blob, out, p, win);
  return launch_status("trans_head_kernel");
}

template <class Window>
int launch_head(int d_k, const float* logits, int64_t ldx, const float* query, const int64_t* offsets, int64_t T, const float* blob, float* out,
                const TransParams& p, const Window& win, cudaStream_t st) {
  return d_k == 64 ? launch_head<64>(logits, ldx, query, offsets, T, blob, out, p, win, st)
                   : launch_head<32>(logits, ldx, query, offsets, T, blob, out, p, win, st);
}

}  // namespace
}  // namespace sv

extern "C" {

int sv_trans_create(const sv_trans_cfg* cfg, sv_trans_handle** out) {
  using namespace sv;
  SV_CHECK(cfg && out, "null argument");
  SV_CHECK(cfg->d_model >= 1 && cfg->d_model <= kDP, "trans: 1 <= d_model <= 16");
  SV_CHECK(cfg->len_q >= 1 && cfg->len_q <= kLMax, "trans: 1 <= len_q <= 32");
  SV_CHECK(cfg->d_ff >= 1 && cfg->d_ff <= kFFMax, "trans: 1 <= d_ff <= 64");
  if (cfg->n_heads != kH || cfg->d_k != cfg->d_v || (cfg->d_k != 32 && cfg->d_k != 64))
    return fail(SV_ERR_UNSUPPORTED, "trans: n_heads = 4 and d_k = d_v = 32 or 64 are supported (the reference's mstcn_f_maps = 32 and >= 64 configurations)");
  if (cfg->n_layers != 1) return fail(SV_ERR_UNSUPPORTED, "trans: n_layers must be 1 (adapter_transformer.py:322)");
  int dev = 0;
  SV_CUDA_OK(cudaGetDevice(&dev));
  sv_trans* h = new sv_trans();
  h->cfg = *cfg;
  h->device = dev;
  *out = h;
  return SV_OK;
}

int sv_trans_destroy(sv_trans_handle* h) {
  if (!h) return SV_OK;
  if (h->d_blob) cudaFree(h->d_blob);
  if (h->d_offsets) cudaFree(h->d_offsets);
  delete h;
  return SV_OK;
}

int sv_trans_set_tensor(sv_trans_handle* h, const char* name, const float* host_data, const int64_t* shape, int32_t ndim) {
  using namespace sv;
  SV_CHECK(h && name && host_data, "null argument");
  return h->sd.set(name, host_data, shape, ndim);
}

int sv_trans_pack_weights(sv_trans_handle* h) {
  using namespace sv;
  SV_CHECK(h, "null handle");
  std::vector<float> blob;
  SV_TRY(h->cfg.d_k == 64 ? pack_blob<64>(h, &blob) : pack_blob<32>(h, &blob));
  SV_TRY(upload(h->device, &h->d_blob, blob));
  h->sd.packed = true;
  return SV_OK;
}

int sv_trans_forward(sv_trans_handle* h, const float* logits, int64_t ldx, const float* query, const int64_t* video_offsets, int32_t n_videos,
                     float* out, void* stream) {
  using namespace sv;
  SV_CHECK(h && logits && query && video_offsets && out, "null argument");
  if (!h->sd.packed) return fail(SV_ERR_STATE, "trans: pack_weights() has not been called");
  SV_CHECK(n_videos >= 1 && video_offsets[0] == 0, "trans: offsets");
  for (int i = 0; i < n_videos; ++i) SV_CHECK(video_offsets[i + 1] > video_offsets[i], "trans: empty video / non-increasing offsets");
  const int64_t T = video_offsets[n_videos];
  SV_CHECK(ldx >= T, "trans: logits row stride");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (h->offsets_cap < n_videos + 1) {
    if (h->d_offsets) cudaFree(h->d_offsets);
    h->offsets_cap = std::max(128, 2 * (n_videos + 1));
    SV_CUDA_OK(cudaMalloc(&h->d_offsets, h->offsets_cap * sizeof(int64_t)));
  }
  SV_CUDA_OK(cudaMemcpyAsync(h->d_offsets, video_offsets, (n_videos + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  TransParams p;
  p.D = h->cfg.d_model; p.L = h->cfg.len_q; p.FF = h->cfg.d_ff; p.n_videos = n_videos;
  p.scale = 1.0f / sqrtf(static_cast<float>(h->cfg.d_k));
  return launch_head(h->cfg.d_k, logits, ldx, query, h->d_offsets, T, h->d_blob, out, p, OfflineWindow{}, st);
}

size_t sv_trans_stream_state_bytes(const sv_trans_handle* h, int32_t n_streams) {
  if (!h || n_streams < 1) return 0;
  return sv::StreamRegistry::counter_bytes(n_streams) + static_cast<size_t>(n_streams) * (h->cfg.len_q - 1) * h->cfg.d_model * sizeof(float);
}

int sv_trans_stream_reset(sv_trans_handle* h, void* state, size_t state_bytes, int32_t n_streams, const int32_t* stream_ids, int32_t n_ids,
                          void* stream) {
  using namespace sv;
  SV_CHECK(h && state, "null argument");
  return h->streams.reset(state, state_bytes, sv_trans_stream_state_bytes(h, n_streams), n_streams, stream_ids, n_ids,
                          static_cast<cudaStream_t>(stream));
}

int sv_trans_stream_forward(sv_trans_handle* h, void* state, size_t state_bytes, int32_t n_streams, const float* logits, int64_t ldx,
                            const float* query, const int32_t* stream_ids, const int64_t* counts, int32_t n_ids, float* out, void* stream) {
  using namespace sv;
  SV_CHECK(h && state && logits && query && stream_ids && counts && out, "null argument");
  if (!h->sd.packed) return fail(SV_ERR_STATE, "trans: pack_weights() has not been called");
  // a misaligned state cannot have been reset: say what is wrong with it before looking it up
  SV_CHECK((reinterpret_cast<uintptr_t>(state) & 255) == 0, "trans stream: state must be 256-byte aligned");
  std::vector<int64_t> tab;
  SV_TRY(h->streams.check_step(state, state_bytes, sv_trans_stream_state_bytes(h, n_streams), n_streams, stream_ids, counts, n_ids, &tab));
  const int64_t T = tab[n_ids];
  SV_CHECK(ldx >= T, "trans: logits row stride");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (h->offsets_cap < static_cast<int>(tab.size())) {
    if (h->d_offsets) cudaFree(h->d_offsets);
    h->offsets_cap = std::max(128, 2 * static_cast<int>(tab.size()));
    SV_CUDA_OK(cudaMalloc(&h->d_offsets, h->offsets_cap * sizeof(int64_t)));
  }
  SV_CUDA_OK(cudaMemcpyAsync(h->d_offsets, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  TransParams p;
  p.D = h->cfg.d_model; p.L = h->cfg.len_q; p.FF = h->cfg.d_ff; p.n_videos = n_ids;
  p.scale = 1.0f / sqrtf(static_cast<float>(h->cfg.d_k));
  int64_t* seen = static_cast<int64_t*>(state);
  float* ring = reinterpret_cast<float*>(static_cast<char*>(state) + StreamRegistry::counter_bytes(n_streams));
  const StreamWindow win{h->d_offsets + n_ids + 1, seen, ring};
  SV_TRY(launch_head(h->cfg.d_k, logits, ldx, query, h->d_offsets, T, h->d_blob, out, p, win, st));
  trans_stream_commit_kernel<<<n_ids, 128, 0, st>>>(logits, ldx, h->d_offsets, n_ids, p.D, p.L, ring, seen);
  SV_TRY(launch_status("trans_stream_commit_kernel"));
  h->streams.advance(state, stream_ids, counts, n_ids);
  return SV_OK;
}

}  // extern "C"
