// MS-TCN MultiStageModel_S (mstcn.py:94-130, 153-178, 181-214) for sm_100a, fp32, all videos of a batch at once.
//
// Layout: activations are TIME-MAJOR [T_total, F] fp32 (the memory layout of the reference's `long_feature`,
// trans_SV_output.py:271-272), videos concatenated; a per-frame "video start row" array masks causal history at
// video boundaries, so one launch per layer covers every video.  The causal branch (mstcn_causal_conv=True) is
//   y[t] = x[t] + W1 * relu(Wd[0] x[t-2d] + Wd[1] x[t-d] + Wd[2] x[t] + bd) + b1        (mstcn.py:208-214; SURVEY a15)
// which equals conv(pad 2d) -> relu -> drop last 2d samples -> 1x1 -> add.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include <map>
#include <string>
#include <vector>

#include "kernels.cuh"

namespace sv {
namespace {

// ---- stage-1 input projection (conv_1x1, mstcn.py:174: out[t,f] = sum_d feats[t,d] W[f,d] + b[f]) on tensor cores with fp32-level
// accuracy ("3xTF32"): each fp32 operand is split into a TF32
// high part and a TF32 residual, and  x*w ~= xh*wh + xh*wl + xl*wh  (dropped term ~2^-22 relative), three mma.sync.m16n8k8.tf32
// per tile step.  The 8 KB/frame feature read is the only HBM traffic, and with the arithmetic off the FP32 pipe the kernel
// is bound by it (an fp32 SIMT GEMM needs 16 FLOP per byte from a 72 TFLOP/s pipe: measured 0.10 of the HBM peak, compute-bound).
// feats tiles arrive through a 3-stage cp.async ring; W is pre-split on the host.
__device__ __forceinline__ uint32_t to_tf32(float x) { uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return r; }
__device__ __forceinline__ void mma_tf32_1688(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  const int bytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}

// Q = 16 appends the Trans-SVNet query head to the same pass over the features: columns F..F+Q-1 of the packed weight hold
// `Transformer.fc.weight` (Linear(f_dim, out_features, bias=False), adapter_transformer.py:325) and the epilogue writes
// query[t, c] = tanh(feats[t] . fc[c]) (adapter_transformer.py:348) for c < q_out.
template <int F, int Q>
__global__ void __launch_bounds__(128) mstcn_inproj_tf32x3_kernel(const float* __restrict__ feats, const float* __restrict__ Whi,
                                                                  const float* __restrict__ Wlo, const float* __restrict__ bias, int64_t T, int D,
                                                                  float* __restrict__ out, float* __restrict__ query, int q_out) {
  constexpr int FW = F + Q;
  constexpr int BM = 128, BK = 32, ST = 3, NT = FW / 8, MT = 2;   // each warp: 2 m16 tiles (32 rows) x FW columns
  constexpr int LDA = BK + 4, LDW = FW + 8;  // conflict-free fragment loads
  extern __shared__ __align__(16) float sm[];
  float* As = sm;                       // [ST][BM][LDA]
  float* Wh = As + ST * BM * LDA;       // [ST][BK][LDW]
  float* Wl = Wh + ST * BK * LDW;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int64_t row0 = static_cast<int64_t>(blockIdx.x) * BM;
  const int nk = D / BK;

  auto issue = [&](int kt, int stg) {
    const int k0 = kt * BK;
    for (int i = tid; i < BM * (BK / 4); i += 128) {      // 128 rows x 8 chunks of 16 B
      const int r = i >> 3, c4 = i & 7;
      const bool ok = row0 + r < T;
      cp_async_16(As + (stg * BM + r) * LDA + c4 * 4, ok ? feats + (row0 + r) * D + k0 + c4 * 4 : feats, ok);
    }
    for (int i = tid; i < BK * (FW / 4); i += 128) {      // 32 k x FW/4 chunks, hi and lo
      const int kk = i / (FW / 4), f4 = i % (FW / 4);
      cp_async_16(Wh + (stg * BK + kk) * LDW + f4 * 4, Whi + static_cast<int64_t>(k0 + kk) * FW + f4 * 4, true);
      cp_async_16(Wl + (stg * BK + kk) * LDW + f4 * 4, Wlo + static_cast<int64_t>(k0 + kk) * FW + f4 * 4, true);
    }
  };
  float acc[MT][NT][4];
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int i = 0; i < NT; ++i) { acc[m][i][0] = acc[m][i][1] = acc[m][i][2] = acc[m][i][3] = 0.f; }

  for (int s = 0; s < ST - 1; ++s) {
    if (s < nk) issue(s, s);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int kt = 0; kt < nk; ++kt) {
    asm volatile("cp.async.wait_group %0;" ::"n"(ST - 2) : "memory");
    __syncthreads();                                       // stage kt%ST landed for everyone; stage (kt-1)%ST is free again
    if (kt + ST - 1 < nk) issue(kt + ST - 1, (kt + ST - 1) % ST);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const float* a_s = As + ((kt % ST) * BM + warp * 32) * LDA;
    const float* wh_s = Wh + (kt % ST) * BK * LDW;
    const float* wl_s = Wl + (kt % ST) * BK * LDW;
#pragma unroll
    for (int kk = 0; kk < BK / 8; ++kk) {
      uint32_t ah[MT][4], al[MT][4];
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        const float* am = a_s + m * 16 * LDA;
        const float a[4] = {am[g * LDA + kk * 8 + t], am[(g + 8) * LDA + kk * 8 + t], am[g * LDA + kk * 8 + t + 4], am[(g + 8) * LDA + kk * 8 + t + 4]};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ah[m][j] = to_tf32(a[j]);
          al[m][j] = to_tf32(a[j] - __uint_as_float(ah[m][j]));
        }
      }
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const uint32_t bh0 = __float_as_uint(wh_s[(kk * 8 + t) * LDW + nt * 8 + g]), bh1 = __float_as_uint(wh_s[(kk * 8 + t + 4) * LDW + nt * 8 + g]);
        const uint32_t bl0 = __float_as_uint(wl_s[(kk * 8 + t) * LDW + nt * 8 + g]), bl1 = __float_as_uint(wl_s[(kk * 8 + t + 4) * LDW + nt * 8 + g]);
#pragma unroll
        for (int m = 0; m < MT; ++m) {
          mma_tf32_1688(acc[m][nt], al[m], bh0, bh1);   // small terms first
          mma_tf32_1688(acc[m][nt], ah[m], bl0, bl1);
          mma_tf32_1688(acc[m][nt], ah[m], bh0, bh1);
        }
      }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
  for (int m = 0; m < MT; ++m) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int col = nt * 8 + t * 2;
      const int64_t r0 = row0 + warp * 32 + m * 16 + g, r1 = r0 + 8;
      if (col < F) {
        const float2 b = __ldg(reinterpret_cast<const float2*>(bias + col));
        if (r0 < T) *reinterpret_cast<float2*>(out + r0 * F + col) = make_float2(acc[m][nt][0] + b.x, acc[m][nt][1] + b.y);
        if (r1 < T) *reinterpret_cast<float2*>(out + r1 * F + col) = make_float2(acc[m][nt][2] + b.x, acc[m][nt][3] + b.y);
      } else if (query != nullptr) {
        const int c = col - F;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (c + j < q_out) {
            if (r0 < T) query[r0 * q_out + c + j] = tanhf(acc[m][nt][j]);
            if (r1 < T) query[r1 * q_out + c + j] = tanhf(acc[m][nt][2 + j]);
          }
        }
      }
    }
  }
}

// ---- where a tap row that precedes its video's (or stream chunk's) first row in x comes from.  The layer kernels take one of these
// as a template parameter; nothing else in them depends on it.
//   OfflineTaps: x holds whole videos, so such a row is the causal zero padding.
//   StreamTaps:  x holds one step of a stream (rows seen[s] .. seen[s]+count-1 of stream s); a row at stream position q >= 0 comes
//                from the layer's ring in the stream state (slot q mod 2d), a row at q < 0 is the zero padding.
struct OfflineTaps {
  static constexpr bool kStream = false;
};
struct StreamTaps {
  static constexpr bool kStream = true;
  const int2* __restrict__ rowmap;   // [T]: (stream, stream position) of every row of x
  const float* __restrict__ ring;    // this stage's / layer's ring of stream 0; ring rows = 2 * dilation (a power of two)
  int64_t stream_stride;             // floats from one stream's state to the next
  int ld;                            // floats per ring row (= F)
  // the ring row `shift` positions before row tt, or null for the zero padding
  __device__ __forceinline__ const float* row(int64_t tt, int64_t shift, int dilation) const {
    const int2 m = rowmap[tt];
    const int64_t q = static_cast<int64_t>(m.y) - shift;
    if (q < 0) return nullptr;
    return ring + m.x * stream_stride + (q & (2 * dilation - 1)) * ld;
  }
};

// ---- one DilatedResidualLayer for every frame of every video.  One thread = NS consecutive time steps, all F channels
// (NS = 2 for F = 32: every broadcast weight read from shared memory then feeds two FMAs per output channel).
// smem: Wd [3][F_in][F_out], W1 [F_in][F_out], bd[F], b1[F] (weights broadcast-read, conflict-free).
template <int F, int NS, class Taps>
__global__ void __launch_bounds__(128) mstcn_layer_kernel(const float* __restrict__ x, const int* __restrict__ frame_start,
                                                          const float* __restrict__ wpack, int dilation, int64_t T, float* __restrict__ y,
                                                          const Taps taps) {
  extern __shared__ __align__(16) float sw[];
  constexpr int NW = 3 * F * F + F * F + 2 * F;
  for (int i = threadIdx.x; i < NW / 4; i += blockDim.x) reinterpret_cast<float4*>(sw)[i] = __ldg(reinterpret_cast<const float4*>(wpack) + i);
  __syncthreads();
  const float* Wd = sw;
  const float* W1 = sw + 3 * F * F;
  const float* bd = W1 + F * F;
  const float* b1 = bd + F;
  const int64_t t0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * NS;
  if (t0 >= T) return;
  float acc[NS][F];
#pragma unroll
  for (int s = 0; s < NS; ++s)
#pragma unroll
    for (int f = 0; f < F; ++f) acc[s][f] = bd[f];
#pragma unroll
  for (int tap = 0; tap < 3; ++tap) {
    const float* xp[NS];
    bool ok[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const int64_t tt = t0 + s;
      const int64_t ts = tt - static_cast<int64_t>(2 - tap) * dilation;
      ok[s] = tt < T && ts >= static_cast<int64_t>(frame_start[tt < T ? tt : T - 1]);  // zero left padding, never across a video boundary
      xp[s] = x + (ok[s] ? ts : 0) * F;
      if constexpr (Taps::kStream) {
        const float* hp = (!ok[s] && tt < T) ? taps.row(tt, tt - ts, dilation) : nullptr;
        if (hp != nullptr) { ok[s] = true; xp[s] = hp; }
      }
    }
#pragma unroll
    for (int c4 = 0; c4 < F / 4; ++c4) {
      float xs[NS][4];
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const float4 xv = ok[s] ? __ldg(reinterpret_cast<const float4*>(xp[s]) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        xs[s][0] = xv.x; xs[s][1] = xv.y; xs[s][2] = xv.z; xs[s][3] = xv.w;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4* wr = reinterpret_cast<const float4*>(Wd + (tap * F + c4 * 4 + j) * F);
#pragma unroll
        for (int f4 = 0; f4 < F / 4; ++f4) {
          const float4 w = wr[f4];
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            acc[s][f4 * 4 + 0] = fmaf(xs[s][j], w.x, acc[s][f4 * 4 + 0]);
            acc[s][f4 * 4 + 1] = fmaf(xs[s][j], w.y, acc[s][f4 * 4 + 1]);
            acc[s][f4 * 4 + 2] = fmaf(xs[s][j], w.z, acc[s][f4 * 4 + 2]);
            acc[s][f4 * 4 + 3] = fmaf(xs[s][j], w.w, acc[s][f4 * 4 + 3]);
          }
        }
      }
    }
  }
  // out = x[t] + b1 + W1 * relu(acc)
  float out[NS][F];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const int64_t tt = t0 + s < T ? t0 + s : T - 1;
    const float4* xr = reinterpret_cast<const float4*>(x + tt * F);
#pragma unroll
    for (int f4 = 0; f4 < F / 4; ++f4) {
      const float4 v = __ldg(xr + f4);
      out[s][f4 * 4 + 0] = v.x + b1[f4 * 4 + 0]; out[s][f4 * 4 + 1] = v.y + b1[f4 * 4 + 1];
      out[s][f4 * 4 + 2] = v.z + b1[f4 * 4 + 2]; out[s][f4 * 4 + 3] = v.w + b1[f4 * 4 + 3];
    }
  }
#pragma unroll
  for (int c = 0; c < F; ++c) {
    float h[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) h[s] = fmaxf(acc[s][c], 0.f);
    const float4* wr = reinterpret_cast<const float4*>(W1 + c * F);
#pragma unroll
    for (int f4 = 0; f4 < F / 4; ++f4) {
      const float4 w = wr[f4];
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        out[s][f4 * 4 + 0] = fmaf(h[s], w.x, out[s][f4 * 4 + 0]);
        out[s][f4 * 4 + 1] = fmaf(h[s], w.y, out[s][f4 * 4 + 1]);
        out[s][f4 * 4 + 2] = fmaf(h[s], w.z, out[s][f4 * 4 + 2]);
        out[s][f4 * 4 + 3] = fmaf(h[s], w.w, out[s][f4 * 4 + 3]);
      }
    }
  }
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    if (t0 + s < T) {
      float4* yp = reinterpret_cast<float4*>(y + (t0 + s) * F);
#pragma unroll
      for (int f4 = 0; f4 < F / 4; ++f4) yp[f4] = make_float4(out[s][f4 * 4], out[s][f4 * 4 + 1], out[s][f4 * 4 + 2], out[s][f4 * 4 + 3]);
    }
  }
}

// ---- one DilatedResidualLayer on tensor cores, F = 32 (the path's f_maps): both convolutions of the layer are small GEMMs over time
// rows — the dilated conv is [rows, 3F] x [3F, F] (the three taps are three row-shifted views of the input), the 1x1 conv [rows, F] x [F, F]
// — done as 3xTF32 mma.sync (hi/lo split of both operands, fp32-level accuracy, same scheme as the stage-1 projection).  A CTA walks
// 128-row tiles; the three shifted input tiles arrive by cp.async with rows before the video start zero-filled (= the causal left
// padding, per row, so batched videos never see each other); weights (pre-split on the host) stay in shared memory for all tiles.
// The fp32 SIMT kernel below it is bound by broadcast LDS of the weights (20 TFLOP/s); this one by the L2 stream of the activations.
constexpr int kTcLdW = 40;                                                       // F + 8: conflict-free B fragments
constexpr int kTcWpack = 2 * (96 * kTcLdW) + 2 * (32 * kTcLdW) + 64;             // Wd hi | Wd lo | W1 hi | W1 lo | bd | b1
template <class Taps>
__global__ void __launch_bounds__(128) mstcn_layer_tc_kernel(const float* __restrict__ x, const int* __restrict__ frame_start, const float* __restrict__ wpack,
                                                             int dilation, int64_t T, float* __restrict__ y, int num_tiles, const Taps taps) {
  constexpr int F = 32, BM = 128, LDA = F + 4, LDW = kTcLdW;
  extern __shared__ __align__(16) float sm[];
  float* Xs = sm;                         // [3 taps][BM][LDA]
  float* Ws = Xs + 3 * BM * LDA;          // kTcWpack
  float* Hs = Ws + kTcWpack;              // [4 warps][32][LDA]: relu(conv_dilated) of the warp's rows, A operand of the 1x1 conv
  const float* Wdh = Ws;
  const float* Wdl = Wdh + 96 * LDW;
  const float* W1h = Wdl + 96 * LDW;
  const float* W1l = W1h + 32 * LDW;
  const float* bd = W1l + 32 * LDW;
  const float* b1 = bd + F;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  for (int i = tid; i < kTcWpack / 4; i += 128) reinterpret_cast<float4*>(Ws)[i] = __ldg(reinterpret_cast<const float4*>(wpack) + i);
  float* hs = Hs + warp * 32 * LDA;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int64_t row0 = static_cast<int64_t>(tile) * BM;
    __syncthreads();   // the previous tile's reads of Xs are done (and, first time round, Ws is complete)
    for (int i = tid; i < 3 * BM * (F / 4); i += 128) {
      const int tap = i / (BM * (F / 4)), rem = i - tap * (BM * (F / 4)), r = rem >> 3, c4 = rem & 7;
      const int64_t tt = row0 + r;
      const int64_t ts = tt - static_cast<int64_t>(2 - tap) * dilation;
      const bool ok = tt < T && ts >= static_cast<int64_t>(frame_start[tt < T ? tt : T - 1]);   // zero left padding, never across a video boundary
      if constexpr (Taps::kStream) {
        const float* hp = (!ok && tt < T) ? taps.row(tt, tt - ts, dilation) : nullptr;
        cp_async_16(Xs + (tap * BM + r) * LDA + c4 * 4, ok ? x + ts * F + c4 * 4 : (hp != nullptr ? hp + c4 * 4 : x), ok || hp != nullptr);
      } else {
        cp_async_16(Xs + (tap * BM + r) * LDA + c4 * 4, ok ? x + ts * F + c4 * 4 : x, ok);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    float acc[2][4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const float2 b = *reinterpret_cast<const float2*>(bd + nt * 8 + t * 2);
#pragma unroll
      for (int m = 0; m < 2; ++m) { acc[m][nt][0] = b.x; acc[m][nt][1] = b.y; acc[m][nt][2] = b.x; acc[m][nt][3] = b.y; }
    }
#pragma unroll
    for (int tap = 0; tap < 3; ++tap) {
      const float* a_s = Xs + (tap * BM + warp * 32) * LDA;
#pragma unroll
      for (int kk = 0; kk < F / 8; ++kk) {
        uint32_t ah[2][4], al[2][4];
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          const float* am = a_s + m * 16 * LDA + kk * 8;
          const float a[4] = {am[g * LDA + t], am[(g + 8) * LDA + t], am[g * LDA + t + 4], am[(g + 8) * LDA + t + 4]};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            ah[m][j] = to_tf32(a[j]);
            al[m][j] = to_tf32(a[j] - __uint_as_float(ah[m][j]));
          }
        }
        const int k0 = tap * F + kk * 8;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const uint32_t bh0 = __float_as_uint(Wdh[(k0 + t) * LDW + nt * 8 + g]), bh1 = __float_as_uint(Wdh[(k0 + t + 4) * LDW + nt * 8 + g]);
          const uint32_t bl0 = __float_as_uint(Wdl[(k0 + t) * LDW + nt * 8 + g]), bl1 = __float_as_uint(Wdl[(k0 + t + 4) * LDW + nt * 8 + g]);
#pragma unroll
          for (int m = 0; m < 2; ++m) {
            mma_tf32_1688(acc[m][nt], al[m], bh0, bh1);   // small terms first
            mma_tf32_1688(acc[m][nt], ah[m], bl0, bl1);
            mma_tf32_1688(acc[m][nt], ah[m], bh0, bh1);
          }
        }
      }
    }
    // h = relu(.) -> the warp's scratch rows (accumulator layout -> A-operand layout goes through shared memory)
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        *reinterpret_cast<float2*>(hs + (m * 16 + g) * LDA + nt * 8 + t * 2) = make_float2(fmaxf(acc[m][nt][0], 0.f), fmaxf(acc[m][nt][1], 0.f));
        *reinterpret_cast<float2*>(hs + (m * 16 + g + 8) * LDA + nt * 8 + t * 2) = make_float2(fmaxf(acc[m][nt][2], 0.f), fmaxf(acc[m][nt][3], 0.f));
      }
    __syncwarp();
    // out = x[t] + b1 + W1 h   (x[t] is the tap-2 tile)
    const float* x_s = Xs + (2 * BM + warp * 32) * LDA;
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const float2 b = *reinterpret_cast<const float2*>(b1 + nt * 8 + t * 2);
        const float2 x0 = *reinterpret_cast<const float2*>(x_s + (m * 16 + g) * LDA + nt * 8 + t * 2);
        const float2 x1 = *reinterpret_cast<const float2*>(x_s + (m * 16 + g + 8) * LDA + nt * 8 + t * 2);
        acc[m][nt][0] = x0.x + b.x; acc[m][nt][1] = x0.y + b.y; acc[m][nt][2] = x1.x + b.x; acc[m][nt][3] = x1.y + b.y;
      }
#pragma unroll
    for (int kk = 0; kk < F / 8; ++kk) {
      uint32_t ah[2][4], al[2][4];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const float* am = hs + m * 16 * LDA + kk * 8;
        const float a[4] = {am[g * LDA + t], am[(g + 8) * LDA + t], am[g * LDA + t + 4], am[(g + 8) * LDA + t + 4]};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ah[m][j] = to_tf32(a[j]);
          al[m][j] = to_tf32(a[j] - __uint_as_float(ah[m][j]));
        }
      }
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const uint32_t bh0 = __float_as_uint(W1h[(kk * 8 + t) * LDW + nt * 8 + g]), bh1 = __float_as_uint(W1h[(kk * 8 + t + 4) * LDW + nt * 8 + g]);
        const uint32_t bl0 = __float_as_uint(W1l[(kk * 8 + t) * LDW + nt * 8 + g]), bl1 = __float_as_uint(W1l[(kk * 8 + t + 4) * LDW + nt * 8 + g]);
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          mma_tf32_1688(acc[m][nt], al[m], bh0, bh1);
          mma_tf32_1688(acc[m][nt], ah[m], bl0, bl1);
          mma_tf32_1688(acc[m][nt], ah[m], bh0, bh1);
        }
      }
    }
    __syncwarp();   // every lane has read hs before the next tile overwrites it
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const int64_t r0 = row0 + warp * 32 + m * 16 + g, r1 = r0 + 8;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        if (r0 < T) *reinterpret_cast<float2*>(y + r0 * F + nt * 8 + t * 2) = make_float2(acc[m][nt][0], acc[m][nt][1]);
        if (r1 < T) *reinterpret_cast<float2*>(y + r1 * F + nt * 8 + t * 2) = make_float2(acc[m][nt][2], acc[m][nt][3]);
      }
    }
  }
}

// ---- conv_out_classes (mstcn.py:177): logits[c, t] = Wout[c,:] . h[t,:] + b[c]; channel-major output (coalesced over t).
// Optionally fused with the next stage's softmax(dim=channels) + conv_1x1 (mstcn.py:126, 174): next[t, f].
template <int F>
__global__ void __launch_bounds__(128) mstcn_out_kernel(const float* __restrict__ h, const float* __restrict__ Wout /*[C][F]*/,
                                                        const float* __restrict__ bout, int C, int64_t T, float* __restrict__ logits /*[C][T]*/,
                                                        const float* __restrict__ Wnext /*[C][F] (k-major) or null*/,
                                                        const float* __restrict__ bnext, float* __restrict__ next /*[T][F]*/) {
  constexpr int MAXC = 32;
  __shared__ float sWo[MAXC * F];
  __shared__ float sWn[MAXC * F];
  __shared__ float sbo[MAXC];
  __shared__ float sbn[F];
  for (int i = threadIdx.x; i < C * F; i += blockDim.x) { sWo[i] = Wout[i]; if (Wnext) sWn[i] = Wnext[i]; }
  for (int i = threadIdx.x; i < C; i += blockDim.x) sbo[i] = bout[i];
  if (Wnext) for (int i = threadIdx.x; i < F; i += blockDim.x) sbn[i] = bnext[i];
  __syncthreads();
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= T) return;
  float hv[F];
  const float4* hp = reinterpret_cast<const float4*>(h + t * F);
#pragma unroll
  for (int f4 = 0; f4 < F / 4; ++f4) { const float4 v = __ldg(hp + f4); hv[f4 * 4] = v.x; hv[f4 * 4 + 1] = v.y; hv[f4 * 4 + 2] = v.z; hv[f4 * 4 + 3] = v.w; }
  float lg[MAXC];
  float mx = -INFINITY;
  for (int c = 0; c < C; ++c) {
    float a = sbo[c];
#pragma unroll
    for (int f = 0; f < F; ++f) a = fmaf(hv[f], sWo[c * F + f], a);
    lg[c] = a;
    logits[static_cast<int64_t>(c) * T + t] = a;
    mx = fmaxf(mx, a);
  }
  if (Wnext == nullptr) return;
  float den = 0.f;
  for (int c = 0; c < C; ++c) { lg[c] = expf(lg[c] - mx); den += lg[c]; }
  const float inv = 1.0f / den;
  float o[F];
#pragma unroll
  for (int f = 0; f < F; ++f) o[f] = sbn[f];
  for (int c = 0; c < C; ++c) {
    const float p = lg[c] * inv;
#pragma unroll
    for (int f = 0; f < F; ++f) o[f] = fmaf(p, sWn[c * F + f], o[f]);
  }
  float4* np = reinterpret_cast<float4*>(next + t * F);
#pragma unroll
  for (int f4 = 0; f4 < F / 4; ++f4) np[f4] = make_float4(o[f4 * 4], o[f4 * 4 + 1], o[f4 * 4 + 2], o[f4 * 4 + 3]);
}

// out[t][j][c] = x[c][t - (len_q - 1) + j] (zero where the index is negative): the 30-frame causal windows of the MS-TCN logits that
// Transformer.original_forward builds with a Python loop (adapter_transformer.py:335-343), for one video.
__global__ void causal_windows_kernel(const float* __restrict__ x, int64_t ldx, int C, int64_t T, int len_q, float* __restrict__ out) {
  const int64_t total = T * len_q * C;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const int64_t r = i / C;
    const int j = static_cast<int>(r % len_q);
    const int64_t t = r / len_q;
    const int64_t src = t - (len_q - 1) + j;
    out[i] = src >= 0 ? __ldg(x + static_cast<int64_t>(c) * ldx + src) : 0.f;
  }
}

__global__ void frame_start_kernel(const int64_t* __restrict__ offsets, int n_videos, int64_t T, int* __restrict__ frame_start) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= T) return;
  int lo = 0, hi = n_videos;  // find v with offsets[v] <= t < offsets[v+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (offsets[mid] <= t) lo = mid; else hi = mid;
  }
  frame_start[t] = static_cast<int>(offsets[lo]);
}

// ---- stream steps.  `tab` = the step's host tables: row offsets of the n_ids chunks [n_ids + 1], then their stream ids [n_ids].
__device__ __forceinline__ int step_chunk(const int64_t* __restrict__ offsets, int n_ids, int64_t t) {
  int lo = 0, hi = n_ids;  // chunk k with offsets[k] <= t < offsets[k+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (offsets[mid] <= t) lo = mid; else hi = mid;
  }
  return lo;
}

// frame_start_kernel of a step: every row's chunk start (the first row the layer kernels read from x) and (stream, position).
__global__ void stream_rowmap_kernel(const int64_t* __restrict__ tab, int n_ids, int64_t T, const int64_t* __restrict__ seen,
                                     int* __restrict__ frame_start, int2* __restrict__ rowmap) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const int k = step_chunk(tab, n_ids, t);
  const int s = static_cast<int>(tab[n_ids + 1 + k]);
  frame_start[t] = static_cast<int>(tab[k]);
  rowmap[t] = make_int2(s, static_cast<int>(seen[s] + (t - tab[k])));
}

// After the step: the last min(2 * 2^l, count) input rows of every layer l of every stage go to their ring slots, then seen advances.
// act holds the layer inputs of the step, buffer g * (layers + 1) + l for stage g, layer l.  No kernel of this step reads a ring
// after this one starts, so the ring writes cannot race a reader.
template <int F>
__global__ void mstcn_stream_commit_kernel(const float* __restrict__ act, int64_t T, int stages, int layers, const int64_t* __restrict__ tab,
                                           int n_ids, const int2* __restrict__ rowmap, float* __restrict__ rings, int64_t stream_stride,
                                           int64_t* __restrict__ seen) {
  const int64_t ring_rows = 2 * ((int64_t{1} << layers) - 1);   // per stage
  const int64_t total = T * (F / 4);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / (F / 4);
    const int c4 = static_cast<int>(i % (F / 4));
    const int64_t end = tab[step_chunk(tab, n_ids, r) + 1];
    const int2 m = rowmap[r];
    float* ring_s = rings + m.x * stream_stride;
    for (int g = 0; g < stages; ++g) {
      for (int l = 0; l < layers; ++l) {
        const int64_t R = int64_t{2} << l;   // ring rows of layer l; its ring starts R - 2 rows into the stage's rings
        if (end - r > R) continue;
        const float4 v = __ldg(reinterpret_cast<const float4*>(act + ((static_cast<int64_t>(g) * (layers + 1) + l) * T + r) * F) + c4);
        reinterpret_cast<float4*>(ring_s + (g * ring_rows + R - 2 + (m.y & (R - 1))) * F)[c4] = v;
      }
    }
    if (r == end - 1 && c4 == 0) seen[m.x] = static_cast<int64_t>(m.y) + 1;
  }
}

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

}  // namespace
}  // namespace sv

struct sv_mstcn {
  sv_mstcn_cfg cfg;
  int device = 0;
  std::map<std::string, sv::HostTensor> tensors;
  bool packed = false;
  float* d_weights = nullptr;  // single device blob
  // offsets (in floats) into the blob
  struct Stage { size_t w_in, b_in, w_out, b_out, w_next, b_next, w_in_hi = 0, w_in_lo = 0; std::vector<size_t> layer, layer_tc; };
  std::vector<Stage> stages;
  int q_out = 0;  // rows of the optional query head `fc.weight` packed next to the stage-1 projection (0 = absent)
  int64_t launches = 0;
  // host copy of the frame counters of every stream state reset through this handle, keyed by the state's address: the handle is the
  // only writer of those counters, and the copy lets a step be refused before launch (unknown state, position past 2^31)
  std::map<const void*, std::vector<int64_t>> stream_seen;
};

namespace sv {
namespace {

std::string stage_prefix(int s) { return s == 0 ? std::string("stage1_phase") : "stages." + std::to_string(s - 1); }

int expect(const sv_mstcn* h, const std::string& key, std::initializer_list<int64_t> shape, const HostTensor** out) {
  auto it = h->tensors.find(key);
  if (it == h->tensors.end()) return fail(SV_ERR_STATE, "mstcn: missing state_dict key '" + key + "'");
  if (it->second.shape != std::vector<int64_t>(shape)) return fail(SV_ERR_INVALID, "mstcn: wrong shape for '" + key + "'");
  *out = &it->second;
  return SV_OK;
}

constexpr int kQCols = 16;  // query-head columns appended to the stage-1 projection (out_features <= 16)

template <int F, int Q>
int launch_inproj(sv_mstcn* h, const float* feats, int64_t T, float* out, float* query, cudaStream_t st) {
  const sv_mstcn::Stage& S = h->stages[0];
  const float* W = h->d_weights;
  constexpr size_t smem = (3 * 128 * (32 + 4) + 2 * 3 * 32 * (F + Q + 8)) * sizeof(float);
  SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mstcn_inproj_tf32x3_kernel<F, Q>), static_cast<int>(smem)));
  mstcn_inproj_tf32x3_kernel<F, Q><<<static_cast<unsigned>(ceil_div64(T, 128)), 128, smem, st>>>(feats, W + S.w_in_hi, W + S.w_in_lo, W + S.b_in, T,
                                                                                                 h->cfg.f_dim, out, query, h->q_out);
  return launch_status("mstcn_inproj_tf32x3_kernel");
}

// What a stream step adds to a forward: the state it reads history from and commits to.
struct StreamStep {
  const int64_t* tab;   // device copy of the step's tables (see stream_rowmap_kernel)
  int n_ids;
  int64_t* seen;        // state: [n_streams] frame counters
  float* rings;         // state: rings of stream 0
  int64_t stream_stride;
};

// Stream-state layout (documented in surgvid.h): int64 seen[n_streams], padded to 256 B, then per stream, per stage, per layer l a ring
// of 2 * 2^l rows x f_maps floats (ring of layer l starts 2 * (2^l - 1) rows into the stage's 2 * (2^layers - 1) rows).
size_t stream_seen_bytes(int32_t n_streams) { return (static_cast<size_t>(n_streams) * sizeof(int64_t) + 255) & ~static_cast<size_t>(255); }
int64_t stream_ring_rows(const sv_mstcn_cfg& c) { return 2 * ((int64_t{1} << c.layers) - 1); }   // per stage
int64_t stream_stride_floats(const sv_mstcn_cfg& c) { return c.stages * stream_ring_rows(c) * c.f_maps; }

template <int F, int NS, class Taps>
int launch_layer(bool tc, int tc_grid, int tc_tiles, size_t tc_smem, unsigned lb, size_t layer_smem, const float* x, const int* frame_start,
                 const float* w, const float* w_tc, int dilation, int64_t T, float* y, const Taps& taps, cudaStream_t st) {
  if (tc) {
    mstcn_layer_tc_kernel<Taps><<<tc_grid, 128, tc_smem, st>>>(x, frame_start, w_tc, dilation, T, y, tc_tiles, taps);
    return launch_status("mstcn_layer_tc_kernel");
  }
  mstcn_layer_kernel<F, NS, Taps><<<lb, 128, layer_smem, st>>>(x, frame_start, w, dilation, T, y, taps);
  return launch_status("mstcn_layer_kernel");
}

// The whole-video forward (ss == null) or one stream step (ss != null) over T rows.  Offline, the activations ping-pong between two
// buffers; a step keeps every layer's input (buffer g * (layers + 1) + l) for the commit at its end.
template <int F>
int run_forward(sv_mstcn* h, const float* feats, const int64_t* d_offsets, int n_videos, int64_t T, float* logits, float* query, void* ws,
                cudaStream_t st, const StreamStep* ss = nullptr) {
  const sv_mstcn_cfg& c = h->cfg;
  char* p = static_cast<char*>(ws);
  const int64_t n_bufs = ss ? static_cast<int64_t>(c.stages) * (c.layers + 1) : 2;
  float* act = reinterpret_cast<float*>(p);
  int* frame_start = reinterpret_cast<int*>(act + n_bufs * T * F);
  int2* rowmap = reinterpret_cast<int2*>(frame_start + ((T + 1) & ~int64_t{1}));
  auto buf = [&](int64_t i) { return act + (ss ? i : (i & 1)) * T * F; };
  const unsigned tb = static_cast<unsigned>(ceil_div64(T, 128));
  if (ss) {
    stream_rowmap_kernel<<<tb, 128, 0, st>>>(ss->tab, ss->n_ids, T, ss->seen, frame_start, rowmap);
    SV_TRY(launch_status("stream_rowmap_kernel"));
  } else {
    frame_start_kernel<<<tb, 128, 0, st>>>(d_offsets, n_videos, T, frame_start);
    SV_TRY(launch_status("frame_start_kernel"));
  }
  h->launches = 1;
  const float* W = h->d_weights;
  const size_t layer_smem = (3 * F * F + F * F + 2 * F) * sizeof(float);
  constexpr int NS = 1;  // time steps per thread in the layer kernel (NS = 2 measured slower on B200: 167 registers, 92 vs 76 us)
  const unsigned lb = static_cast<unsigned>(ceil_div64(ceil_div64(T, NS), 128));
  static const bool use_tc = [] { const char* e = getenv("SURGVID_MSTCN_TC"); return !(e && atoi(e) == 0); }();   // A/B switch
  const bool tc = F == 32 && use_tc;
  const size_t tc_smem = (3 * 128 * (32 + 4) + kTcWpack + 4 * 32 * (32 + 4)) * sizeof(float);
  const int tc_tiles = static_cast<int>(ceil_div64(T, 128));
  const int tc_grid = std::min(tc_tiles, 2 * std::max(1, device_sm_count()));
  if (ss) {
    SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mstcn_layer_kernel<F, NS, StreamTaps>), static_cast<int>(layer_smem)));
    if (tc) SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mstcn_layer_tc_kernel<StreamTaps>), static_cast<int>(tc_smem)));
  } else {
    SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mstcn_layer_kernel<F, NS, OfflineTaps>), static_cast<int>(layer_smem)));
    if (tc) SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mstcn_layer_tc_kernel<OfflineTaps>), static_cast<int>(tc_smem)));
  }
  for (int s = 0; s < c.stages; ++s) {
    const sv_mstcn::Stage& S = h->stages[s];
    const int64_t b0 = static_cast<int64_t>(s) * (c.layers + 1);   // this stage's input buffer
    if (s == 0) {
      if (h->q_out > 0) SV_TRY((launch_inproj<F, kQCols>(h, feats, T, buf(0), query, st)));
      else SV_TRY((launch_inproj<F, 0>(h, feats, T, buf(0), nullptr, st)));
      ++h->launches;
    }
    for (int l = 0; l < c.layers; ++l) {
      const float* w = W + S.layer[l];
      const float* w_tc = tc ? W + S.layer_tc[l] : nullptr;
      if (ss) {
        const StreamTaps taps{rowmap, ss->rings + (s * stream_ring_rows(c) + (int64_t{2} << l) - 2) * F, ss->stream_stride, F};
        SV_TRY((launch_layer<F, NS>(tc, tc_grid, tc_tiles, tc_smem, lb, layer_smem, buf(b0 + l), frame_start, w, w_tc, 1 << l, T, buf(b0 + l + 1), taps, st)));
      } else {
        SV_TRY((launch_layer<F, NS>(tc, tc_grid, tc_tiles, tc_smem, lb, layer_smem, buf(b0 + l), frame_start, w, w_tc, 1 << l, T, buf(b0 + l + 1),
                                    OfflineTaps{}, st)));
      }
      ++h->launches;
    }
    const bool last = s == c.stages - 1;
    // writes this stage's logits; unless last, also softmax + the next stage's conv_1x1 into the next stage's input buffer
    mstcn_out_kernel<F><<<tb, 128, 0, st>>>(buf(b0 + c.layers), W + S.w_out, W + S.b_out, c.out_features, T,
                                           logits + static_cast<int64_t>(s) * c.out_features * T, last ? nullptr : W + S.w_next,
                                           last ? nullptr : W + S.b_next, last ? nullptr : buf(b0 + c.layers + 1));
    SV_TRY(launch_status("mstcn_out_kernel"));
    ++h->launches;
  }
  if (ss) {
    const unsigned cb = static_cast<unsigned>(std::min<int64_t>(ceil_div64(T * (F / 4), 256), static_cast<int64_t>(device_sm_count()) * 8));
    mstcn_stream_commit_kernel<F><<<cb, 256, 0, st>>>(act, T, c.stages, c.layers, ss->tab, ss->n_ids, rowmap, ss->rings, ss->stream_stride, ss->seen);
    SV_TRY(launch_status("mstcn_stream_commit_kernel"));
    ++h->launches;
  }
  return SV_OK;
}

}  // namespace
}  // namespace sv

extern "C" {

int sv_mstcn_create(const sv_mstcn_cfg* cfg, sv_mstcn_handle** out) {
  using namespace sv;
  SV_CHECK(cfg && out, "null argument");
  SV_CHECK(cfg->stages >= 1 && cfg->layers >= 1 && cfg->layers <= 16, "mstcn: stages>=1, 1<=layers<=16");
  if (cfg->f_maps != 32 && cfg->f_maps != 64) return fail(SV_ERR_UNSUPPORTED, "mstcn: f_maps must be 32 or 64");
  if (!cfg->causal) return fail(SV_ERR_UNSUPPORTED, "mstcn: only the causal branch (mstcn_causal_conv=True) is implemented");
  SV_CHECK(cfg->out_features >= 1 && cfg->out_features <= 32, "mstcn: out_features in [1,32]");
  SV_CHECK(cfg->f_dim % 32 == 0, "mstcn: f_dim must be a multiple of 32");
  int dev = 0;
  SV_CUDA_OK(cudaGetDevice(&dev));
  sv_mstcn* h = new sv_mstcn();
  h->cfg = *cfg;
  h->device = dev;
  *out = h;
  return SV_OK;
}

int sv_mstcn_destroy(sv_mstcn_handle* h) {
  if (!h) return SV_OK;
  if (h->d_weights) cudaFree(h->d_weights);
  delete h;
  return SV_OK;
}

int sv_mstcn_set_tensor(sv_mstcn_handle* h, const char* name, const float* host_data, const int64_t* shape, int32_t ndim) {
  using namespace sv;
  SV_CHECK(h && name && host_data && (shape || ndim == 0), "null argument");
  HostTensor t;
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= shape[i]; }
  t.data.assign(host_data, host_data + n);
  h->tensors[name] = std::move(t);
  h->packed = false;
  return SV_OK;
}

int sv_mstcn_pack_weights(sv_mstcn_handle* h) {
  using namespace sv;
  SV_CHECK(h, "null handle");
  const sv_mstcn_cfg& c = h->cfg;
  const int64_t F = c.f_maps, C = c.out_features;
  std::vector<float> blob;
  auto reserve = [&](size_t n) { size_t off = blob.size(); blob.resize(off + ((n + 3) / 4) * 4, 0.f); return off; };
  h->stages.assign(c.stages, sv_mstcn::Stage());
  for (int s = 0; s < c.stages; ++s) {
    const std::string p = stage_prefix(s);
    const int64_t dim = s == 0 ? c.f_dim : C;
    sv_mstcn::Stage& S = h->stages[s];
    const HostTensor *w, *b;
    SV_TRY(expect(h, p + ".conv_1x1.weight", {F, dim, 1}, &w));
    SV_TRY(expect(h, p + ".conv_1x1.bias", {F}, &b));
    // k-major [dim][F] so that a K-chunk of W is contiguous over f
    S.w_in = reserve(dim * F);
    for (int64_t f = 0; f < F; ++f)
      for (int64_t d = 0; d < dim; ++d) blob[S.w_in + d * F + f] = w->data[f * dim + d];
    S.b_in = reserve(F);
    std::copy(b->data.begin(), b->data.end(), blob.begin() + S.b_in);
    if (s == 0) {  // TF32 hi/lo split of the stage-1 projection for the 3xTF32 tensor-core kernel
      auto tf32_rna = [](float x) {
        uint32_t u;
        memcpy(&u, &x, 4);
        u = (u + 0x1000u) & 0xFFFFE000u;  // round to nearest (ties away) at 10 mantissa bits, like cvt.rna.tf32.f32
        float r;
        memcpy(&r, &u, 4);
        return r;
      };
      // optional query head of the Trans-SVNet wrapper: `fc.weight` [out_q, f_dim], no bias (adapter_transformer.py:325)
      h->q_out = 0;
      const HostTensor* fc = nullptr;
      auto fit = h->tensors.find("fc.weight");
      if (fit != h->tensors.end()) {
        fc = &fit->second;
        if (fc->shape.size() != 2 || fc->shape[1] != dim || fc->shape[0] < 1 || fc->shape[0] > kQCols)
          return fail(SV_ERR_INVALID, "mstcn: 'fc.weight' must be [out_features <= 16, f_dim]");
        h->q_out = static_cast<int>(fc->shape[0]);
      }
      const int64_t FW = F + (fc ? kQCols : 0);
      S.w_in_hi = reserve(dim * FW);
      S.w_in_lo = reserve(dim * FW);
      for (int64_t d = 0; d < dim; ++d) {
        for (int64_t f = 0; f < FW; ++f) {
          float x = 0.f;
          if (f < F) x = blob[S.w_in + d * F + f];
          else if (f - F < h->q_out) x = fc->data[(f - F) * dim + d];
          const float hi = tf32_rna(x);
          blob[S.w_in_hi + d * FW + f] = hi;
          blob[S.w_in_lo + d * FW + f] = tf32_rna(x - hi);
        }
      }
    }
    for (int l = 0; l < c.layers; ++l) {
      const std::string lp = p + ".layers." + std::to_string(l);
      const HostTensor *wd, *bd, *w1, *b1;
      SV_TRY(expect(h, lp + ".conv_dilated.weight", {F, F, 3}, &wd));
      SV_TRY(expect(h, lp + ".conv_dilated.bias", {F}, &bd));
      SV_TRY(expect(h, lp + ".conv_1x1.weight", {F, F, 1}, &w1));
      SV_TRY(expect(h, lp + ".conv_1x1.bias", {F}, &b1));
      const size_t off = reserve(3 * F * F + F * F + 2 * F);
      S.layer.push_back(off);
      // Wd[tap][cin][cout] ; conv1d weight is [cout][cin][tap], tap k multiplies x[t-(2-k)d]
      for (int64_t k = 0; k < 3; ++k)
        for (int64_t ci = 0; ci < F; ++ci)
          for (int64_t co = 0; co < F; ++co) blob[off + (k * F + ci) * F + co] = wd->data[(co * F + ci) * 3 + k];
      const size_t o1 = off + 3 * F * F;
      for (int64_t ci = 0; ci < F; ++ci)
        for (int64_t co = 0; co < F; ++co) blob[o1 + ci * F + co] = w1->data[co * F + ci];
      std::copy(bd->data.begin(), bd->data.end(), blob.begin() + o1 + F * F);
      std::copy(b1->data.begin(), b1->data.end(), blob.begin() + o1 + F * F + F);
      if (F == 32) {  // tensor-core layer kernel: [k][n] rows padded to kTcLdW, TF32 hi/lo pre-split
        auto tf32_rna = [](float x) {
          uint32_t u;
          memcpy(&u, &x, 4);
          u = (u + 0x1000u) & 0xFFFFE000u;
          float r;
          memcpy(&r, &u, 4);
          return r;
        };
        const size_t ot = reserve(kTcWpack);
        S.layer_tc.push_back(ot);
        const size_t dh = ot, dl = dh + 96 * kTcLdW, oh = dl + 96 * kTcLdW, ol = oh + 32 * kTcLdW, obd = ol + 32 * kTcLdW, ob1 = obd + 32;
        for (int64_t k = 0; k < 3; ++k)
          for (int64_t ci = 0; ci < F; ++ci)
            for (int64_t co = 0; co < F; ++co) {
              const float w = wd->data[(co * F + ci) * 3 + k], hi = tf32_rna(w);
              blob[dh + (k * F + ci) * kTcLdW + co] = hi;
              blob[dl + (k * F + ci) * kTcLdW + co] = tf32_rna(w - hi);
            }
        for (int64_t ci = 0; ci < F; ++ci)
          for (int64_t co = 0; co < F; ++co) {
            const float w = w1->data[co * F + ci], hi = tf32_rna(w);
            blob[oh + ci * kTcLdW + co] = hi;
            blob[ol + ci * kTcLdW + co] = tf32_rna(w - hi);
          }
        std::copy(bd->data.begin(), bd->data.end(), blob.begin() + obd);
        std::copy(b1->data.begin(), b1->data.end(), blob.begin() + ob1);
      }
    }
    SV_TRY(expect(h, p + ".conv_out_classes.weight", {C, F, 1}, &w));
    SV_TRY(expect(h, p + ".conv_out_classes.bias", {C}, &b));
    S.w_out = reserve(C * F);
    std::copy(w->data.begin(), w->data.end(), blob.begin() + S.w_out);  // [C][F]
    S.b_out = reserve(C);
    std::copy(b->data.begin(), b->data.end(), blob.begin() + S.b_out);
  }
  // next-stage input projection in [C][F] (k-major) form next to the producing stage
  for (int s = 0; s + 1 < c.stages; ++s) {
    h->stages[s].w_next = h->stages[s + 1].w_in;
    h->stages[s].b_next = h->stages[s + 1].b_in;
  }
  if (h->d_weights) { cudaFree(h->d_weights); h->d_weights = nullptr; }
  SV_CUDA_OK(cudaSetDevice(h->device));
  SV_CUDA_OK(cudaMalloc(&h->d_weights, blob.size() * sizeof(float)));
  SV_CUDA_OK(cudaMemcpy(h->d_weights, blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice));
  h->packed = true;
  return SV_OK;
}

size_t sv_mstcn_workspace_bytes(const sv_mstcn_handle* h, int64_t total_frames) {
  if (!h || total_frames <= 0) return 0;
  const size_t T = static_cast<size_t>(total_frames);
  return 2 * T * h->cfg.f_maps * sizeof(float) + T * sizeof(int) + 4096 * sizeof(int64_t) + 256;
}

int sv_mstcn_forward(sv_mstcn_handle* h, const float* feats, const int64_t* video_offsets, int32_t n_videos, float* logits,
                     void* workspace, size_t workspace_bytes, void* stream) {
  return sv_mstcn_forward_query(h, feats, video_offsets, n_videos, logits, nullptr, workspace, workspace_bytes, stream);
}

int sv_mstcn_forward_query(sv_mstcn_handle* h, const float* feats, const int64_t* video_offsets, int32_t n_videos, float* logits, float* query,
                           void* workspace, size_t workspace_bytes, void* stream) {
  using namespace sv;
  SV_CHECK(h && feats && video_offsets && logits && workspace, "null argument");
  if (!h->packed) return fail(SV_ERR_STATE, "mstcn: pack_weights() has not been called");
  if (query != nullptr && h->q_out == 0) return fail(SV_ERR_STATE, "mstcn: a query output was requested but no 'fc.weight' tensor was set");
  SV_CHECK(n_videos >= 1 && n_videos < 4096, "mstcn: 1 <= n_videos < 4096");
  SV_CHECK(video_offsets[0] == 0, "mstcn: video_offsets[0] must be 0");
  for (int i = 0; i < n_videos; ++i) SV_CHECK(video_offsets[i + 1] > video_offsets[i], "mstcn: empty video / non-increasing offsets");
  const int64_t T = video_offsets[n_videos];
  SV_CHECK(T < (1LL << 31), "mstcn: too many frames");
  SV_CHECK(workspace_bytes >= sv_mstcn_workspace_bytes(h, T), "mstcn: workspace too small");
  SV_CHECK((reinterpret_cast<uintptr_t>(feats) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "mstcn: alignment");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // offsets live at the tail of the workspace
  char* tail = static_cast<char*>(workspace) + 2 * static_cast<size_t>(T) * h->cfg.f_maps * sizeof(float) + static_cast<size_t>(T) * sizeof(int);
  tail = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(tail) + 255) & ~static_cast<uintptr_t>(255));
  int64_t* d_offsets = reinterpret_cast<int64_t*>(tail);
  SV_CUDA_OK(cudaMemcpyAsync(d_offsets, video_offsets, (n_videos + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  if (h->cfg.f_maps == 32) return run_forward<32>(h, feats, d_offsets, n_videos, T, logits, query, workspace, st);
  return run_forward<64>(h, feats, d_offsets, n_videos, T, logits, query, workspace, st);
}

size_t sv_mstcn_stream_state_bytes(const sv_mstcn_handle* h, int32_t n_streams) {
  if (!h || n_streams < 1) return 0;
  return sv::stream_seen_bytes(n_streams) + static_cast<size_t>(n_streams) * sv::stream_stride_floats(h->cfg) * sizeof(float);
}

size_t sv_mstcn_stream_workspace_bytes(const sv_mstcn_handle* h, int64_t rows) {
  if (!h || rows <= 0) return 0;
  const size_t T = static_cast<size_t>(rows), bufs = static_cast<size_t>(h->cfg.stages) * (h->cfg.layers + 1);
  const size_t rowmap_end = bufs * T * h->cfg.f_maps * sizeof(float) + ((T + 1) & ~size_t{1}) * sizeof(int) + T * sizeof(int2);
  return rowmap_end + 256 + (2 * T + 1) * sizeof(int64_t);
}

int sv_mstcn_stream_reset(sv_mstcn_handle* h, void* state, size_t state_bytes, int32_t n_streams, const int32_t* stream_ids, int32_t n_ids,
                          void* stream) {
  using namespace sv;
  SV_CHECK(h && state, "null argument");
  SV_CHECK(n_streams >= 1, "mstcn stream: n_streams >= 1");
  SV_CHECK(state_bytes >= sv_mstcn_stream_state_bytes(h, n_streams), "mstcn stream: state too small");
  SV_CHECK((reinterpret_cast<uintptr_t>(state) & 255) == 0, "mstcn stream: state must be 256-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t* seen = static_cast<int64_t*>(state);
  if (stream_ids == nullptr) {   // every stream: the whole state, so that no stale ring row is left behind
    SV_CUDA_OK(cudaMemsetAsync(state, 0, sv_mstcn_stream_state_bytes(h, n_streams), st));
    h->stream_seen[state].assign(n_streams, 0);
    return SV_OK;
  }
  auto it = h->stream_seen.find(state);
  if (it == h->stream_seen.end()) return fail(SV_ERR_STATE, "mstcn stream: reset every stream of a new state (stream_ids = NULL) first");
  SV_CHECK(static_cast<int32_t>(it->second.size()) == n_streams, "mstcn stream: n_streams differs from the state's last full reset");
  SV_CHECK(n_ids >= 1, "mstcn stream: n_ids >= 1");
  std::vector<char> hit(n_streams, 0);
  for (int i = 0; i < n_ids; ++i) {
    SV_CHECK(stream_ids[i] >= 0 && stream_ids[i] < n_streams, "mstcn stream: stream id out of range");
    SV_CHECK(!hit[stream_ids[i]], "mstcn stream: duplicate stream id");
    hit[stream_ids[i]] = 1;
  }
  // only the counter: ring rows are read at positions [0, seen) alone, and those are rewritten before they are read again
  for (int i = 0; i < n_ids; ++i) {
    SV_CUDA_OK(cudaMemsetAsync(seen + stream_ids[i], 0, sizeof(int64_t), st));
    it->second[stream_ids[i]] = 0;
  }
  return SV_OK;
}

int sv_mstcn_stream_step(sv_mstcn_handle* h, void* state, size_t state_bytes, int32_t n_streams, const float* feats, const int32_t* stream_ids,
                         const int64_t* counts, int32_t n_ids, float* logits, float* query, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace sv;
  SV_CHECK(h && state && feats && stream_ids && counts && logits && workspace, "null argument");
  if (!h->packed) return fail(SV_ERR_STATE, "mstcn: pack_weights() has not been called");
  if (query != nullptr && h->q_out == 0) return fail(SV_ERR_STATE, "mstcn: a query output was requested but no 'fc.weight' tensor was set");
  SV_CHECK(n_streams >= 1, "mstcn stream: n_streams >= 1");
  SV_CHECK(state_bytes >= sv_mstcn_stream_state_bytes(h, n_streams), "mstcn stream: state too small");
  auto it = h->stream_seen.find(state);
  if (it == h->stream_seen.end()) return fail(SV_ERR_STATE, "mstcn stream: the state was not reset through this handle (reset every stream first)");
  SV_CHECK(static_cast<int32_t>(it->second.size()) == n_streams, "mstcn stream: n_streams differs from the state's last full reset");
  SV_CHECK(n_ids >= 1 && n_ids <= n_streams, "mstcn stream: 1 <= n_ids <= n_streams");
  std::vector<int64_t> tab(2 * static_cast<size_t>(n_ids) + 1);   // chunk row offsets [n_ids + 1], then stream ids [n_ids]
  std::vector<char> hit(n_streams, 0);
  for (int i = 0; i < n_ids; ++i) {
    const int32_t s = stream_ids[i];
    SV_CHECK(s >= 0 && s < n_streams, "mstcn stream: stream id out of range");
    SV_CHECK(!hit[s], "mstcn stream: duplicate stream id");
    hit[s] = 1;
    SV_CHECK(counts[i] >= 1, "mstcn stream: counts must be >= 1");
    SV_CHECK(counts[i] < (1LL << 31) - it->second[s], "mstcn stream: a stream position would pass 2^31");
    tab[i + 1] = tab[i] + counts[i];
    SV_CHECK(tab[i + 1] < (1LL << 31), "mstcn stream: too many rows in one step");
    tab[n_ids + 1 + i] = s;
  }
  const int64_t T = tab[n_ids];
  SV_CHECK(workspace_bytes >= sv_mstcn_stream_workspace_bytes(h, T), "mstcn stream: workspace too small");
  SV_CHECK((reinterpret_cast<uintptr_t>(feats) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0 &&
               (reinterpret_cast<uintptr_t>(state) & 255) == 0, "mstcn stream: alignment (feats 16 B, workspace and state 256 B)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bufs = static_cast<size_t>(h->cfg.stages) * (h->cfg.layers + 1);
  char* tail = static_cast<char*>(workspace) + bufs * T * h->cfg.f_maps * sizeof(float) + ((T + 1) & ~int64_t{1}) * sizeof(int) + T * sizeof(int2);
  tail = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(tail) + 255) & ~static_cast<uintptr_t>(255));
  int64_t* d_tab = reinterpret_cast<int64_t*>(tail);
  SV_CUDA_OK(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  StreamStep ss;
  ss.tab = d_tab;
  ss.n_ids = n_ids;
  ss.seen = static_cast<int64_t*>(state);
  ss.rings = reinterpret_cast<float*>(static_cast<char*>(state) + stream_seen_bytes(n_streams));
  ss.stream_stride = stream_stride_floats(h->cfg);
  const int rc = h->cfg.f_maps == 32 ? run_forward<32>(h, feats, nullptr, 0, T, logits, query, workspace, st, &ss)
                                     : run_forward<64>(h, feats, nullptr, 0, T, logits, query, workspace, st, &ss);
  if (rc != SV_OK) return rc;
  for (int i = 0; i < n_ids; ++i) it->second[stream_ids[i]] += counts[i];
  return SV_OK;
}

int sv_op_causal_windows(const float* x, int64_t ldx, int32_t C, const int64_t* video_offsets, int32_t n_videos, int32_t len_q, float* out,
                         void* stream) {
  using namespace sv;
  SV_CHECK(x && video_offsets && out, "null argument");
  SV_CHECK(C >= 1 && len_q >= 1 && n_videos >= 1, "causal_windows: C, len_q, n_videos >= 1");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int v = 0; v < n_videos; ++v) {
    const int64_t t0 = video_offsets[v], Tv = video_offsets[v + 1] - t0;
    SV_CHECK(Tv > 0, "causal_windows: empty video");
    const int64_t total = Tv * len_q * C;
    const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div64(total, 256), static_cast<int64_t>(device_sm_count()) * 16));
    causal_windows_kernel<<<blocks, 256, 0, st>>>(x + t0, ldx, C, Tv, len_q, out + t0 * len_q * C);
    SV_TRY(launch_status("causal_windows_kernel"));
  }
  return SV_OK;
}

int64_t sv_mstcn_last_launch_count(const sv_mstcn_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
