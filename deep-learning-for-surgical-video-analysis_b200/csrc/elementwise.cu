// HBM-bound kernels of the LFB path: LayerNorm, patch gather (im2col), depthwise 3x3 + GELU, Gaussian 5x5,
// bilinear token resize, token mean.  All 128-bit vectorised on channels-last (token-major == NHWC) tensors;
// the reference's NCHW<->NLC transposes (mix_transformer_evp.py:26-28, 115-116, 212, 376) never happen.
#include <algorithm>

#include "kernels.cuh"

namespace sv {

namespace {

// ------------------------------------------------------------------------------------------ LayerNorm
// LPR lanes cooperate on one row (32/LPR rows per warp); each lane holds NV float4 of the row in registers.
// Two-pass (mean, then centred variance) like ATen's LayerNorm; biased variance; eps inside the square root.
// EXACT: C == 4 * LPR * NV, every lane slot is a real element (no per-slot predicates) — true for every width of the model.
// The kernel is instruction-issue-bound before it is memory-bound, so the arithmetic is kept lean: 1/C is passed in, rstd is one
// MUFU.RSQ (2 ulp, far below the bf16 rounding of the outputs), normalisation is one FFMA per element with per-channel a = rstd*gamma,
// b = beta - mean*a.
// NCHW: the fp32 result goes channel-major instead, out_f32[frame][c][token] with pH tokens per frame (the MiT stage maps that
// forward_features returns); out_patch must be NULL.  The CTA's 8 * RPW rows are staged in shared memory, then every thread stores one
// token position for C * RPW / 32 channels, so each channel's run of consecutive tokens goes out as one contiguous store of
// 32 * RPW bytes (split where the run crosses a frame).  Arithmetic and lane mapping are those of the token-major form, so the fp32
// written is the value out_bf16 rounds.  Four CTAs per SM instead of five: at five, the staging address math spills for C = 40, 80, 512.
template <int LPR, int NV, bool EXACT, bool NCHW = false>
__global__ void __launch_bounds__(256, NCHW ? 4 : 5) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, float eps, float inv_c, int64_t rows, int C,
                                                         float* __restrict__ out_f32, bf16* __restrict__ out_bf16,
                                                         bf16* __restrict__ out_patch, int pH, int pW, int psr) {
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR;
  const int64_t warp_global = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t row = warp_global * RPW + lane / LPR;
  const bool row_ok = row < rows;
  const int nvec = C >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + (row_ok ? row : 0) * C) + sub;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if (EXACT || sub + i * LPR < nvec) {
      v[i] = xr[i * LPR];
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    } else {
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * inv_c;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if (EXACT || sub + i * LPR < nvec) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q * inv_c + eps);
  if constexpr (!NCHW) {
    if (!row_ok) return;
  }
  // optional second bf16 copy in "sr-patch" order: token (b,h,w) -> row (b, h/sr, w/sr), column ((h%sr)*sr + w%sr)*C + c,
  // i.e. the A operand of the spatial-reduction conv (k = stride = sr, no padding) as a plain GEMM.
  int64_t patch_off = -1;
  if (out_patch != nullptr) {  // 32-bit index math (rows < 2^31 checked by the launcher); sr is a power of two
    const uint32_t r32 = static_cast<uint32_t>(row);
    const uint32_t hw = static_cast<uint32_t>(pH) * static_cast<uint32_t>(pW);
    const uint32_t b = r32 / hw;
    const uint32_t rem = r32 - b * hw;
    const uint32_t h = rem / static_cast<uint32_t>(pW);
    const uint32_t w = rem - h * static_cast<uint32_t>(pW);
    const uint32_t lg = 31u - __clz(psr);
    const uint32_t Hk = static_cast<uint32_t>(pH) >> lg, Wk = static_cast<uint32_t>(pW) >> lg;
    const uint32_t hq = h >> lg, wq = w >> lg;
    if (hq < Hk && wq < Wk)
      patch_off = (static_cast<int64_t>((b * Hk + hq) * Wk + wq) << (2 * lg)) * C + (((h & (psr - 1)) << lg) + (w & (psr - 1))) * C;
  }
  const float4* g4 = reinterpret_cast<const float4*>(gamma) + sub;
  const float4* b4 = reinterpret_cast<const float4*>(beta) + sub;
  float* of = !NCHW && out_f32 ? out_f32 + row * C + sub * 4 : nullptr;
  bf16* ob = out_bf16 && (!NCHW || row_ok) ? out_bf16 + row * C + sub * 4 : nullptr;
  // NCHW staging tile [c][row of the CTA], row stride R + P: P makes the 4 scalar stores of a warp hit distinct banks where RPW >= 4
  constexpr int R = 8 * RPW, P = RPW >= 4 ? RPW / 4 : 1;
  __shared__ float tile[NCHW ? 4 * LPR * NV * (R + P) : 1];
  const int lr = (threadIdx.x >> 5) * RPW + lane / LPR;
  bf16* op = patch_off >= 0 ? out_patch + patch_off + sub * 4 : nullptr;
  const float nm = -mean * rstd;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if (EXACT || sub + i * LPR < nvec) {
      const float4 g = __ldg(g4 + i * LPR);
      const float4 b = __ldg(b4 + i * LPR);
      float4 y;   // (v - mean) * rstd * g + b  ==  v * (rstd*g) + (b - mean*rstd*g)
      y.x = fmaf(v[i].x, rstd * g.x, fmaf(nm, g.x, b.x));
      y.y = fmaf(v[i].y, rstd * g.y, fmaf(nm, g.y, b.y));
      y.z = fmaf(v[i].z, rstd * g.z, fmaf(nm, g.z, b.z));
      y.w = fmaf(v[i].w, rstd * g.w, fmaf(nm, g.w, b.w));
      if (of) *reinterpret_cast<float4*>(of + i * LPR * 4) = y;
      if constexpr (NCHW) {
        if (row_ok) {
          float* t = tile + (sub + i * LPR) * 4 * (R + P) + lr;
          t[0] = y.x;
          t[R + P] = y.y;
          t[2 * (R + P)] = y.z;
          t[3 * (R + P)] = y.w;
        }
      }
      if (ob || op) {
        uint2 o;
        o.x = pack_bf16x2(y.x, y.y);
        o.y = pack_bf16x2(y.z, y.w);
        if (ob) *reinterpret_cast<uint2*>(ob + i * LPR * 4) = o;
        if (op) *reinterpret_cast<uint2*>(op + i * LPR * 4) = o;
      }
    }
  }
  if constexpr (NCHW) {
    __syncthreads();
    // thread -> (row R-periodic, channel every 256 / R): the row, and with it the frame and token, is fixed per thread (32-bit math:
    // rows * C < 2^31 is checked by the launcher)
    const uint32_t t = threadIdx.x;
    const uint32_t r32 = blockIdx.x * static_cast<uint32_t>(R) + (t & (R - 1));
    if (r32 < static_cast<uint32_t>(rows)) {
      const uint32_t hw = static_cast<uint32_t>(pH);
      const uint32_t f = r32 / hw;
      float* dst = out_f32 + f * static_cast<uint32_t>(C) * hw + (r32 - f * hw);
      for (uint32_t c = t / R; c < static_cast<uint32_t>(C); c += 256 / R) __stcs(dst + c * hw, tile[c * (R + P) + (t & (R - 1))]);
    }
  }
}

template <int LPR, int NV, bool NCHW>
int ln_launch(const float* x, const float* g, const float* b, float eps, int64_t rows, int C, float* of, bf16* ob, bf16* op, int pH, int pW,
              int psr, cudaStream_t st) {
  constexpr int RPW = 32 / LPR;
  const int64_t warps = ceil_div64(rows, RPW);
  const int64_t blocks = ceil_div64(warps, 8);
  const float inv_c = 1.0f / static_cast<float>(C);
  if (C == 4 * LPR * NV)
    layernorm_kernel<LPR, NV, true, NCHW><<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, g, b, eps, inv_c, rows, C, of, ob, op, pH, pW, psr);
  else
    layernorm_kernel<LPR, NV, false, NCHW><<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, g, b, eps, inv_c, rows, C, of, ob, op, pH, pW, psr);
  return launch_status("layernorm_kernel");
}

// lane mapping per width: one table for both output forms, so a channel-major result is bit-identical to the token-major one
template <bool NCHW>
int ln_dispatch(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int C, float* out_f32, bf16* out_bf16,
                bf16* out_patch, int pH, int pW, int psr, cudaStream_t st) {
  const int nvec = C / 4;
#define SV_LN(L, N) return ln_launch<L, N, NCHW>(x, gamma, beta, eps, rows, C, out_f32, out_bf16, out_patch, pH, pW, psr, st)
  // exact lane mappings first (every slot a real element): the model's widths 16/32/64/128/256/512 and 40/80/160/320
  // (narrow rows: fewer lanes per row and two float4 per lane — the fixed per-thread work, shuffles and patch index math are
  //  amortised over more bytes: 64 -> 49 us for 627200 x 64, 28 -> 26 us for 156800 x 128; ten float4 per lane for C = 320 spills)
  if (nvec == 4) SV_LN(2, 2);
  if (nvec == 8) SV_LN(4, 2);
  if (nvec == 16) SV_LN(8, 2);
  if (nvec == 32) SV_LN(8, 4);
  if (nvec == 64) SV_LN(16, 4);
  if (nvec == 128) SV_LN(32, 4);
  if (nvec == 10) SV_LN(2, 5);
  if (nvec == 20) SV_LN(4, 5);
  if (nvec == 40) SV_LN(8, 5);
  if (nvec == 80) SV_LN(16, 5);
  // anything else: predicated slots
  if (nvec <= 4) SV_LN(4, 1);
  if (nvec <= 8) SV_LN(8, 1);
  if (nvec <= 16) SV_LN(16, 1);
  if (nvec <= 32) SV_LN(32, 1);
  if (nvec <= 64) SV_LN(32, 2);
  if (nvec <= 96) SV_LN(32, 3);
  SV_LN(32, 4);
#undef SV_LN
}

// ------------------------------------------------------------------------------------------ im2col
// NHWC bf16 source, Cin % 8 == 0: one thread moves one 16-byte channel chunk of one (m, kh, kw) tap.
// grid = (chunks of one output row, Ho, B): the only index arithmetic left per thread is two 32-bit divisions by k*k*cv and cv
// (the flat 64-bit version spent ~450 instructions per 16 bytes moved and was issue-bound).
__global__ void __launch_bounds__(256) im2col_nhwc_kernel(const bf16* __restrict__ src, int Cin, int H, int W, int k, int stride, int pad,
                                                          int Ho, int Wo, bf16* __restrict__ out, int64_t ldo) {
  const uint32_t cv = static_cast<uint32_t>(Cin) >> 3;
  const uint32_t kc = static_cast<uint32_t>(k * k) * cv;            // 16-byte chunks per output pixel
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= static_cast<uint32_t>(Wo) * kc) return;
  const uint32_t ow = t / kc, j = t - ow * kc;
  const uint32_t tap = j / cv, c8 = j - tap * cv;
  const uint32_t kh = tap / static_cast<uint32_t>(k), kw = tap - kh * static_cast<uint32_t>(k);
  const int oh = blockIdx.y, b = blockIdx.z;
  const int ih = oh * stride - pad + static_cast<int>(kh);
  const int iw = static_cast<int>(ow) * stride - pad + static_cast<int>(kw);
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (ih >= 0 && ih < H && iw >= 0 && iw < W)
    v = __ldg(reinterpret_cast<const uint4*>(src + ((static_cast<int64_t>(b) * H + ih) * W + iw) * Cin + c8 * 8));
  const int64_t m = (static_cast<int64_t>(b) * Ho + oh) * Wo + ow;
  *reinterpret_cast<uint4*>(out + m * ldo + j * 8) = v;   // column (kh*k + kw)*Cin + c8*8 == j*8
}

// NCHW fp32 source (network inputs: Cin = 3 or 2): one thread gathers 8 consecutive k indices (kh,kw,c order).
// The k -> (plane offset, kh, kw) decomposition is tabulated once per block in shared memory (no div/mod per element).
__global__ void __launch_bounds__(256) im2col_nchw_f32_kernel(const float* __restrict__ src, int B, int Cin, int H, int W, int k, int stride,
                                                              int pad, int Ho, int Wo, bf16* __restrict__ out, int64_t ldo) {
  __shared__ int tab_off[256];
  __shared__ int tab_hw[256];
  const int K = k * k * Cin;
  const int kpad = static_cast<int>(ldo);
  for (int kk = threadIdx.x; kk < kpad; kk += blockDim.x) {
    if (kk < K) {
      const int c = kk % Cin, kw = (kk / Cin) % k, kh = kk / (Cin * k);
      tab_off[kk] = (c * H + kh) * W + kw;
      tab_hw[kk] = (kh << 16) | kw;
    } else {
      tab_off[kk] = 0;
      tab_hw[kk] = -1;
    }
  }
  __syncthreads();
  const int kchunks = kpad >> 3;
  const int64_t total = static_cast<int64_t>(B) * Ho * Wo * kchunks;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int kc = static_cast<int>(idx % kchunks);
  const int64_t m = idx / kchunks;
  const int ow = static_cast<int>(m % Wo);
  const int oh = static_cast<int>((m / Wo) % Ho);
  const int b = static_cast<int>(m / (static_cast<int64_t>(Wo) * Ho));
  const int ih0 = oh * stride - pad, iw0 = ow * stride - pad;
  const float* sb = src + static_cast<int64_t>(b) * Cin * H * W + static_cast<int64_t>(ih0) * W + iw0;
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int kk = kc * 8 + j;
    const int hw = tab_hw[kk];
    float val = 0.f;
    if (hw >= 0) {
      const int ih = ih0 + (hw >> 16), iw = iw0 + (hw & 0xffff);
      if (ih >= 0 && ih < H && iw >= 0 && iw < W) val = __ldg(sb + tab_off[kk]);
    }
    f[j] = val;
  }
  uint4 o;
  o.x = pack_bf16x2(f[0], f[1]);
  o.y = pack_bf16x2(f[2], f[3]);
  o.z = pack_bf16x2(f[4], f[5]);
  o.w = pack_bf16x2(f[6], f[7]);
  *reinterpret_cast<uint4*>(out + m * ldo + kc * 8) = o;
}

// ------------------------------------------------------------------------------------------ DWConv3x3 + bias + GELU
// NHWC bf16.  Block = 8 adjacent pixel columns (threadIdx.y) x 32 lanes of 4 channels (128 channels, 256 B per pixel).
// A thread owns 4 channels (two packed fp32x2 lanes) of a vertical run of kDwRun output pixels and slides a 3x3 window
// down its column: each input row segment is loaded and unpacked to fp32 ONCE, the 36 weights stay in registers, the
// arithmetic is FFMA2 (two fp32 lanes per instruction) and the GELU is MUFU-free, so the kernel stays close to its HBM
// bound instead of the issue bound.  Row loop fully unrolled over a 4-slot register ring (loads run one row ahead).
constexpr int kDwRun = 7;
constexpr int kDwCols = 8;

struct DwRow { f32x2 v[3][2]; };  // 3 columns (w-1, w, w+1) x 2 channel pairs

__device__ __forceinline__ void dw_load_row(DwRow& r, const bf16* __restrict__ base, int hh, int H, int W, int C, int w, bool lok, bool rok) {
  const bool hok = hh >= 0 && hh < H;
  const bf16* p = base + (static_cast<int64_t>(hh) * W + w) * C;
  uint2 a = make_uint2(0u, 0u), b = make_uint2(0u, 0u), c = make_uint2(0u, 0u);
  if (hok && lok) a = __ldg(reinterpret_cast<const uint2*>(p - C));
  if (hok) b = __ldg(reinterpret_cast<const uint2*>(p));
  if (hok && rok) c = __ldg(reinterpret_cast<const uint2*>(p + C));
  r.v[0][0] = f2_from_bf16x2(a.x); r.v[0][1] = f2_from_bf16x2(a.y);
  r.v[1][0] = f2_from_bf16x2(b.x); r.v[1][1] = f2_from_bf16x2(b.y);
  r.v[2][0] = f2_from_bf16x2(c.x); r.v[2][1] = f2_from_bf16x2(c.y);
}

__global__ void __launch_bounds__(256, 2) dwconv3x3_gelu_kernel(const bf16* __restrict__ x, const float* __restrict__ w9c,
                                                                const float* __restrict__ bias, int B, int H, int W, int C,
                                                                bf16* __restrict__ out, int64_t ldo) {
  const int hsegs = (H + kDwRun - 1) / kDwRun;
  const int c0 = (blockIdx.z * 32 + threadIdx.x) * 4;
  const int w = blockIdx.x * kDwCols + threadIdx.y;
  const int hs = blockIdx.y % hsegs;
  const int b = blockIdx.y / hsegs;
  if (c0 >= C || w >= W) return;

  f32x2 wt[9][2];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(w9c + tap * C + c0));
    wt[tap][0] = f2_pack(t.x, t.y);
    wt[tap][1] = f2_pack(t.z, t.w);
  }
  const float4 bs = __ldg(reinterpret_cast<const float4*>(bias + c0));
  const f32x2 bias0 = f2_pack(bs.x, bs.y), bias1 = f2_pack(bs.z, bs.w);
  const bf16* base = x + static_cast<int64_t>(b) * H * W * C + c0;
  bf16* obase = out + (static_cast<int64_t>(b) * H * W + w) * ldo + c0;
  const int h0 = hs * kDwRun;
  const bool lok = w > 0, rok = w + 1 < W;
  DwRow ring[4];
  dw_load_row(ring[0], base, h0 - 1, H, W, C, w, lok, rok);
  dw_load_row(ring[1], base, h0, H, W, C, w, lok, rok);
  dw_load_row(ring[2], base, h0 + 1, H, W, C, w, lok, rok);
#pragma unroll
  for (int i = 0; i < kDwRun; ++i) {
    const int h = h0 + i;
    if (h < H) {  // uniform per thread; rows beyond the image are never stored
      if (i + 1 < kDwRun) dw_load_row(ring[(i + 3) & 3], base, h + 2, H, W, C, w, lok, rok);  // in flight during this row
      const DwRow& r0 = ring[i & 3];
      const DwRow& r1 = ring[(i + 1) & 3];
      const DwRow& r2 = ring[(i + 2) & 3];
      f32x2 a0 = bias0, a1 = bias1;
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        a0 = f2_fma(r0.v[dx][0], wt[dx][0], a0);     a1 = f2_fma(r0.v[dx][1], wt[dx][1], a1);
        a0 = f2_fma(r1.v[dx][0], wt[3 + dx][0], a0); a1 = f2_fma(r1.v[dx][1], wt[3 + dx][1], a1);
        a0 = f2_fma(r2.v[dx][0], wt[6 + dx][0], a0); a1 = f2_fma(r2.v[dx][1], wt[6 + dx][1], a1);
      }
      a0 = f2_gelu_erf_poly(a0);
      a1 = f2_gelu_erf_poly(a1);
      float y0, y1, y2, y3;
      f2_unpack(a0, y0, y1);
      f2_unpack(a1, y2, y3);
      uint2 o;
      o.x = pack_bf16x2(y0, y1);
      o.y = pack_bf16x2(y2, y3);
      *reinterpret_cast<uint2*>(obase + static_cast<int64_t>(h) * W * ldo) = o;
    }
  }
}

// ------------------------------------------------------------------------------------------ Gaussian 5x5 (reflect pad 2)
__device__ __forceinline__ int reflect_idx(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// Register-window version (round 2): a warp owns 28 output columns (32 lanes = 28 + 2 halo columns each side) of a strip of rows and
// walks down the strip: one 128-byte row load per lane and row, the horizontal 5-tap from warp shuffles, the vertical 5-tap from a
// rolling window of five horizontally filtered rows in registers.  No shared memory, no block barriers; four row loads are in flight
// per warp.  Same FMA order as the direct form (sum over dx first, then over dy), so results are bit-identical to the round-1 tiled kernel.
constexpr int kGW = 28;    // output columns per warp
constexpr int kGRS = 56;   // output rows per strip (+ 4 halo rows recomputed per strip)
__global__ void __launch_bounds__(256) gauss5x5_kernel(const float* __restrict__ x, float* __restrict__ out, int H, int W) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c0 = (static_cast<int>(blockIdx.x) * 8 + warp) * kGW;
  if (c0 >= W) return;
  const int y0 = static_cast<int>(blockIdx.y) * kGRS;
  const int64_t pl = blockIdx.z;
  const float* src = x + pl * H * W;
  float* dst = out + pl * H * W;
  const int sc = reflect_idx(min(c0 + lane - 2, W + 1), W);   // source column of this lane (lanes 0,1 / 30,31 are halo columns)
  const int oc = c0 + lane - 2;
  const bool wr = lane >= 2 && lane < 2 + kGW && oc < W;
  const int rows = min(kGRS, H - y0);
  const float k0 = 1.f / 16.f, k1 = 4.f / 16.f, k2 = 6.f / 16.f;   // outer(k,k) == [1 4 6 4 1]^2 / 256 exactly
  auto ld = [&](int y) { return __ldg(src + static_cast<int64_t>(reflect_idx(min(y, H + 1), H)) * W + sc); };
  auto hfilt = [&](float v) {
    const float xm2 = __shfl_up_sync(0xffffffffu, v, 2), xm1 = __shfl_up_sync(0xffffffffu, v, 1);
    const float xp1 = __shfl_down_sync(0xffffffffu, v, 1), xp2 = __shfl_down_sync(0xffffffffu, v, 2);
    float h = fmaf(xm2, k0, 0.f);
    h = fmaf(xm1, k1, h);
    h = fmaf(v, k2, h);
    h = fmaf(xp1, k1, h);
    return fmaf(xp2, k0, h);
  };
  float w0 = hfilt(ld(y0 - 2)), w1 = hfilt(ld(y0 - 1)), w2 = hfilt(ld(y0)), w3 = hfilt(ld(y0 + 1));
  auto emit = [&](int r, float w4) {
    float acc = fmaf(w0, k0, 0.f);
    acc = fmaf(w1, k1, acc);
    acc = fmaf(w2, k2, acc);
    acc = fmaf(w3, k1, acc);
    acc = fmaf(w4, k0, acc);
    if (wr) dst[static_cast<int64_t>(y0 + r) * W + oc] = acc;
    w0 = w1; w1 = w2; w2 = w3; w3 = w4;
  };
  int r = 0;
  for (; r + 4 <= rows; r += 4) {   // four independent row loads in flight
    const float v0 = ld(y0 + r + 2), v1 = ld(y0 + r + 3), v2 = ld(y0 + r + 4), v3 = ld(y0 + r + 5);
    emit(r, hfilt(v0));
    emit(r + 1, hfilt(v1));
    emit(r + 2, hfilt(v2));
    emit(r + 3, hfilt(v3));
  }
  for (; r < rows; ++r) emit(r, hfilt(ld(y0 + r + 2)));
}

// ------------------------------------------------------------------------------------------ bilinear resize (align_corners=False)
__device__ __forceinline__ void bilinear_src(int dst, int in, int outn, int& i0, int& i1, float& l1) {
  const float scale = static_cast<float>(in) / static_cast<float>(outn);
  float s = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  if (s < 0.f) s = 0.f;
  i0 = static_cast<int>(s);
  if (i0 > in - 1) i0 = in - 1;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  l1 = s - static_cast<float>(i0);
}

__global__ void __launch_bounds__(256) bilinear_tokens_kernel(const bf16* __restrict__ x, int B, int H, int W, int C, int Ho, int Wo,
                                                              bf16* __restrict__ out, int64_t ldo) {
  const int cv = C >> 3;
  const int64_t total = static_cast<int64_t>(B) * Ho * Wo * cv;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c8 = static_cast<int>(idx % cv);
  const int64_t m = idx / cv;
  const int ow = static_cast<int>(m % Wo);
  const int oh = static_cast<int>((m / Wo) % Ho);
  const int b = static_cast<int>(m / (static_cast<int64_t>(Wo) * Ho));
  int h0, h1, w0, w1;
  float lh, lw;
  bilinear_src(oh, H, Ho, h0, h1, lh);
  bilinear_src(ow, W, Wo, w0, w1, lw);
  const bf16* base = x + static_cast<int64_t>(b) * H * W * C + c8 * 8;
  const uint4 v00 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<int64_t>(h0) * W + w0) * C));
  const uint4 v01 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<int64_t>(h0) * W + w1) * C));
  const uint4 v10 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<int64_t>(h1) * W + w0) * C));
  const uint4 v11 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<int64_t>(h1) * W + w1) * C));
  const float w00 = (1.f - lh) * (1.f - lw), w01 = (1.f - lh) * lw, w10 = lh * (1.f - lw), w11 = lh * lw;
  const uint32_t* p00 = &v00.x; const uint32_t* p01 = &v01.x; const uint32_t* p10 = &v10.x; const uint32_t* p11 = &v11.x;
  uint32_t o[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 a = unpack_bf16x2(p00[j]), bq = unpack_bf16x2(p01[j]), c = unpack_bf16x2(p10[j]), d = unpack_bf16x2(p11[j]);
    o[j] = pack_bf16x2(w00 * a.x + w01 * bq.x + w10 * c.x + w11 * d.x, w00 * a.y + w01 * bq.y + w10 * c.y + w11 * d.y);
  }
  *reinterpret_cast<uint4*>(out + m * ldo + c8 * 8) = make_uint4(o[0], o[1], o[2], o[3]);
}

// ------------------------------------------------------------------------------------------ misc
__global__ void __launch_bounds__(256) token_mean_kernel(const float* __restrict__ x, int B, int tokens, int C, float* __restrict__ out) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<int64_t>(B) * C) return;
  const int c = static_cast<int>(idx % C);
  const int64_t b = idx / C;
  const float* p = x + b * tokens * C + c;
  float s = 0.f;
  for (int t = 0; t < tokens; ++t) s += p[static_cast<int64_t>(t) * C];
  out[idx] = s / static_cast<float>(tokens);
}

__global__ void __launch_bounds__(256) bf16_to_f32_kernel(const bf16* __restrict__ x, float* __restrict__ out, int64_t n) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx < n) out[idx] = __bfloat162float(x[idx]);
}

inline unsigned blocks_for(int64_t total) { return static_cast<unsigned>(ceil_div64(total, 256)); }

}  // namespace

int launch_layernorm_patch(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int C, float* out_f32,
                           bf16* out_bf16, bf16* out_patch, int pH, int pW, int psr, cudaStream_t st) {
  SV_CHECK(C % 4 == 0 && C >= 4 && C <= 512, "layernorm supports C%4==0, C<=512");
  SV_CHECK(rows > 0, "layernorm rows");
  if (out_patch)
    SV_CHECK(pH > 0 && pW > 0 && psr > 0 && (psr & (psr - 1)) == 0 && rows % (static_cast<int64_t>(pH) * pW) == 0 && rows < (1LL << 31),
             "layernorm patch geometry (sr must be a power of two)");
  return ln_dispatch<false>(x, gamma, beta, eps, rows, C, out_f32, out_bf16, out_patch, pH, pW, psr, st);
}

int launch_layernorm_nchw(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int C, int tokens, float* out_nchw,
                          bf16* out_bf16, cudaStream_t st) {
  SV_CHECK(x && gamma && beta && out_nchw, "layernorm_nchw: null argument");
  SV_CHECK(C % 4 == 0 && C >= 4 && C <= 512, "layernorm supports C%4==0, C<=512");
  SV_CHECK(tokens > 0 && rows > 0 && rows % tokens == 0, "layernorm_nchw: rows must be a positive multiple of the tokens per frame");
  SV_CHECK(rows * C < (1LL << 31), "layernorm_nchw: rows * C must be below 2^31");
  SV_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(gamma) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(beta) & 15) == 0 && (reinterpret_cast<uintptr_t>(out_nchw) & 3) == 0 &&
               (reinterpret_cast<uintptr_t>(out_bf16) & 7) == 0,
           "layernorm_nchw: alignment (x, gamma, beta 16 bytes, out_bf16 8, out_nchw 4)");
  return ln_dispatch<true>(x, gamma, beta, eps, rows, C, out_nchw, out_bf16, nullptr, tokens, 0, 0, st);
}

int launch_layernorm(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int C, float* out_f32,
                     bf16* out_bf16, cudaStream_t st) {
  return launch_layernorm_patch(x, gamma, beta, eps, rows, C, out_f32, out_bf16, nullptr, 0, 0, 0, st);
}

int launch_im2col(const float* src_nchw_f32, const bf16* src_nhwc_bf16, int B, int Cin, int H, int W, int k, int stride, int pad,
                  bf16* out, int64_t ldo, cudaStream_t st) {
  const int Ho = conv_out_dim(H, k, stride, pad), Wo = conv_out_dim(W, k, stride, pad);
  SV_CHECK(Ho > 0 && Wo > 0, "im2col output empty");
  const int K = k * k * Cin;
  SV_CHECK(ldo % 8 == 0 && ldo >= K, "im2col ldo must be a multiple of 8 and >= k*k*Cin");
  if (src_nchw_f32 != nullptr) {
    SV_CHECK(ldo <= 256, "im2col NCHW path supports k*k*Cin <= 256");
    const int64_t total = static_cast<int64_t>(B) * Ho * Wo * (ldo / 8);
    im2col_nchw_f32_kernel<<<blocks_for(total), 256, 0, st>>>(src_nchw_f32, B, Cin, H, W, k, stride, pad, Ho, Wo, out, ldo);
    return launch_status("im2col_nchw_f32_kernel");
  }
  SV_CHECK(src_nhwc_bf16 != nullptr, "im2col needs a source");
  SV_CHECK(Cin % 8 == 0 && ldo == K, "im2col NHWC path needs Cin%8==0 and ldo==k*k*Cin");
  SV_CHECK(Ho <= 65535 && B <= 65535, "im2col grid limits");
  const int64_t row_chunks = static_cast<int64_t>(Wo) * k * k * (Cin / 8);
  dim3 grid(static_cast<unsigned>(ceil_div64(row_chunks, 256)), static_cast<unsigned>(Ho), static_cast<unsigned>(B));
  im2col_nhwc_kernel<<<grid, 256, 0, st>>>(src_nhwc_bf16, Cin, H, W, k, stride, pad, Ho, Wo, out, ldo);
  return launch_status("im2col_nhwc_kernel");
}

int launch_dwconv3x3_gelu(const bf16* x, const float* w9c, const float* bias, int B, int H, int W, int C, bf16* out, int64_t ldo,
                          cudaStream_t st) {
  SV_CHECK(B > 0 && H > 0 && W > 0 && C > 0, "dwconv dims must be positive");
  SV_CHECK(ldo >= C && ldo % 4 == 0, "dwconv output row stride");
  if (dwconv_tma_supported(C)) {  // main path: TMA halo staging (dwconv_tma.cu); the register-window kernel below covers C % 128 != 0
    DwconvPlan plan;
    SV_TRY(dwconv_tma_plan(x, w9c, bias, B, H, W, C, out, ldo, &plan));
    return dwconv_tma_launch(plan, st);
  }
  SV_CHECK(C % 4 == 0, "dwconv needs C%4==0");
  const int hsegs = ceil_div(H, kDwRun);
  SV_CHECK(static_cast<int64_t>(B) * hsegs <= 65535 && ceil_div(C, 128) <= 65535, "dwconv grid limits");
  dim3 grid(ceil_div(W, kDwCols), B * hsegs, ceil_div(C, 128));
  dim3 block(32, kDwCols);
  dwconv3x3_gelu_kernel<<<grid, block, 0, st>>>(x, w9c, bias, B, H, W, C, out, ldo);
  return launch_status("dwconv3x3_gelu_kernel");
}

int dwconv_plan_info(int B, int H, int W, int C, int sms, int32_t* info) {
  SV_CHECK(info != nullptr, "dwconv plan info: null output");
  SV_CHECK(B > 0 && H > 0 && W > 0 && C > 0 && sms > 0, "dwconv dims and SM count must be positive");
  SV_CHECK(C % 4 == 0, "dwconv needs C%4==0");
  if (dwconv_tma_supported(C)) {
    DwconvShape s;
    SV_TRY(dwconv_tma_shape(B, H, W, C, sms, &s));
    // the tile ranges of dwconv3x3_gelu_tma_kernel: CTA i walks [i * per + min(i, extra), ... + per + (i < extra))
    const int per = s.num_tiles / s.grid, extra = s.num_tiles % s.grid;
    const int per_frame = s.tiles_y * s.tiles_x, per_cblk = B * per_frame;
    int cross_frame = 0, cross_cblk = 0;
    for (int i = 0; i < s.grid; ++i) {
      const int tb = i * per + std::min(i, extra), te = tb + per + (i < extra ? 1 : 0);
      if ((tb / per_frame + 1) * static_cast<int64_t>(per_frame) < te) cross_frame = 1;
      if ((tb / per_cblk + 1) * static_cast<int64_t>(per_cblk) < te) cross_cblk = 1;
    }
    const int32_t t[SV_DWCONV_PLAN_INFO_LEN] = {SV_DWCONV_TMA, s.cpl, s.gelu, s.stages, s.prefetch, s.tw, s.tiles_x, s.tiles_y, s.cblks,
                                               s.num_tiles, s.grid, per + (extra ? 1 : 0), cross_frame, cross_cblk};
    std::copy(t, t + SV_DWCONV_PLAN_INFO_LEN, info);
  } else {
    const int hsegs = ceil_div(H, kDwRun);
    SV_CHECK(static_cast<int64_t>(B) * hsegs <= 65535 && ceil_div(C, 128) <= 65535, "dwconv grid limits");
    const int64_t blocks = static_cast<int64_t>(ceil_div(W, kDwCols)) * B * hsegs * ceil_div(C, 128);
    SV_CHECK(blocks < (1LL << 31), "dwconv grid limits");
    const int32_t t[SV_DWCONV_PLAN_INFO_LEN] = {SV_DWCONV_SIMT, 4, 0, 0, 0, kDwCols, ceil_div(W, kDwCols), hsegs, ceil_div(C, 128),
                                               static_cast<int32_t>(blocks), static_cast<int32_t>(blocks), 1, 0, 0};
    std::copy(t, t + SV_DWCONV_PLAN_INFO_LEN, info);
  }
  return SV_OK;
}

int launch_gauss5x5(const float* x, float* out, int planes, int H, int W, cudaStream_t st) {
  SV_CHECK(H >= 3 && W >= 3, "gauss5x5 needs H,W >= 3 (reflect pad 2)");
  SV_CHECK(planes >= 1 && planes <= 65535 && ceil_div(H, kGRS) <= 65535, "gauss5x5 grid limits");
  dim3 grid(static_cast<unsigned>(ceil_div(W, 8 * kGW)), static_cast<unsigned>(ceil_div(H, kGRS)), static_cast<unsigned>(planes));
  gauss5x5_kernel<<<grid, 256, 0, st>>>(x, out, H, W);
  return launch_status("gauss5x5_kernel");
}

int launch_bilinear_tokens(const bf16* x, int B, int H, int W, int C, int Ho, int Wo, bf16* out, int64_t ldo, cudaStream_t st) {
  SV_CHECK(C % 8 == 0 && ldo % 8 == 0 && ldo >= C, "bilinear needs C%8==0, ldo%8==0");
  bilinear_tokens_kernel<<<blocks_for(static_cast<int64_t>(B) * Ho * Wo * (C / 8)), 256, 0, st>>>(x, B, H, W, C, Ho, Wo, out, ldo);
  return launch_status("bilinear_tokens_kernel");
}

int launch_token_mean(const float* x, int B, int tokens, int C, float* out, cudaStream_t st) {
  token_mean_kernel<<<blocks_for(static_cast<int64_t>(B) * C), 256, 0, st>>>(x, B, tokens, C, out);
  return launch_status("token_mean_kernel");
}

int launch_bf16_to_f32(const bf16* x, float* out, int64_t n, cudaStream_t st) {
  bf16_to_f32_kernel<<<blocks_for(n), 256, 0, st>>>(x, out, n);
  return launch_status("bf16_to_f32_kernel");
}

}  // namespace sv

extern "C" {

int sv_op_layernorm(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int32_t C, float* out_f32,
                    uint16_t* out_bf16, void* stream) {
  return sv::launch_layernorm(x, gamma, beta, eps, rows, C, out_f32, reinterpret_cast<sv::bf16*>(out_bf16), static_cast<cudaStream_t>(stream));
}
int sv_op_layernorm_nchw(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int32_t C, int32_t tokens_per_frame,
                         float* out_nchw, uint16_t* out_bf16, void* stream) {
  return sv::launch_layernorm_nchw(x, gamma, beta, eps, rows, C, tokens_per_frame, out_nchw, reinterpret_cast<sv::bf16*>(out_bf16),
                                   static_cast<cudaStream_t>(stream));
}
int sv_op_im2col(const float* src_nchw_f32, const uint16_t* src_nhwc_bf16, int32_t B, int32_t Cin, int32_t H, int32_t W, int32_t k,
                 int32_t stride, int32_t pad, uint16_t* out, int64_t ldo, void* stream) {
  return sv::launch_im2col(src_nchw_f32, reinterpret_cast<const sv::bf16*>(src_nhwc_bf16), B, Cin, H, W, k, stride, pad,
                           reinterpret_cast<sv::bf16*>(out), ldo, static_cast<cudaStream_t>(stream));
}
int sv_op_dwconv3x3_gelu(const uint16_t* x, const float* w, const float* bias, int32_t B, int32_t H, int32_t W, int32_t C, uint16_t* out,
                         void* stream) {
  return sv::launch_dwconv3x3_gelu(reinterpret_cast<const sv::bf16*>(x), w, bias, B, H, W, C, reinterpret_cast<sv::bf16*>(out), C,
                                   static_cast<cudaStream_t>(stream));
}
int sv_op_dwconv_plan_info(int32_t B, int32_t H, int32_t W, int32_t C, int32_t num_sms, int32_t* info) {
  return sv::dwconv_plan_info(B, H, W, C, num_sms, info);
}
int sv_op_gauss5x5(const float* x, float* out, int32_t planes, int32_t H, int32_t W, void* stream) {
  return sv::launch_gauss5x5(x, out, planes, H, W, static_cast<cudaStream_t>(stream));
}
int sv_op_bilinear_tokens(const uint16_t* x, int32_t B, int32_t H, int32_t W, int32_t C, int32_t Ho, int32_t Wo, uint16_t* out,
                          int64_t ldo, void* stream) {
  return sv::launch_bilinear_tokens(reinterpret_cast<const sv::bf16*>(x), B, H, W, C, Ho, Wo, reinterpret_cast<sv::bf16*>(out), ldo,
                                    static_cast<cudaStream_t>(stream));
}
int sv_op_token_mean(const float* x, int32_t B, int32_t tokens, int32_t C, float* out, void* stream) {
  return sv::launch_token_mean(x, B, tokens, C, out, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
