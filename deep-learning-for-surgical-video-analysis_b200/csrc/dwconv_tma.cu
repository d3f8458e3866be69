// Depthwise 3x3 (zero pad 1) + bias + GELU(erf) on NHWC bf16 — the middle of MixFFN (mix_transformer_evp.py:22-30, 63).
//
// HBM-bound op (read + write the 4C-wide hidden once).  Persistent, warp-specialised kernel:
//   * one producer warp streams (TH+2) x (TW+2) x 128-channel input tiles (halo included) into a shared-memory ring with
//     4-D TMA loads; TMA zero-fills coordinates outside the image, which IS the conv's zero padding and also keeps the
//     frames of a batch from bleeding into each other (the frame index is its own tensor dimension);
//   * eight consumer warps (warp = output column, lane = 4 channels) slide a 3x3 register window down their column,
//     FFMA2 arithmetic, MUFU-free GELU, 256-byte coalesced stores.
// Many tiles are in flight per SM regardless of register pressure, which the register-only version could not do.
#include <stdlib.h>

#include <type_traits>

#include "host.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sv {
namespace {

constexpr int kTW = 8;          // max output columns per tile (= consumer warps); 7 or 8 are used, whichever tiles W exactly
constexpr int kTH = 7;          // output rows per tile
constexpr int kCB = 128;        // channels per tile with 4 channels per lane (CPL = 4); CPL = 2 -> 64-channel tiles
constexpr int kMaxStages = 8;     // ring depth and prefetch distance are run-time (DwParams::stages / prefetch)
constexpr int kStages = 4;        // defaults
constexpr int kPrefetch = 2;      // tiles in flight ahead of the one being computed; < kStages - 1 so that the producer lane
                                  // re-fills a stage released a whole tile ago and never waits for the slowest warp
constexpr int kBoxW = kTW + 2, kBoxH = kTH + 2;
constexpr int kTileBytes = kBoxH * kBoxW * kCB * 2;  // 23 040 (CPL = 4); half of it for CPL = 2
constexpr int kThreads = 32 * kTW;  // 8 warps: 2 CTAs/SM -> 4 warps per scheduler -> 128 registers per thread available

struct DwParams {
  const float* w9c;
  const float* bias;
  bf16* out;
  int B, H, W, C;
  long long ldo;
  int tiles_x, tiles_y, cblks;
  int tw;  // output columns per tile actually used (<= kTW); box width = tw + 2
  int stages, prefetch;  // shared-memory ring depth (<= kMaxStages) and tiles requested ahead of the one being computed
  int num_tiles;
  int tiles_per_cblk;
  long long row_stride;  // elements between vertically adjacent output pixels (W * ldo)
};

// GELU (SURGVID_DW_GELU): 0 = MUFU-free erf polynomial (round 1), 1 = x * sigmoid(2 g(x)) on the MUFU pipe (EX2 + RCP),
// 2 = 0.5 x (1 + tanh(g(x))), one MUFU.TANH per element (default: measured 16 % faster than 0 and 9 % faster than 1 at every stage
// shape; end-to-end LFB parity vs the reference goldens is unchanged to three digits — rel-L2 2.10e-3 / 3.43e-3 (0), 2.06e-3 /
// 3.39e-3 (1), 2.11e-3 / 3.40e-3 (2) — because the bf16 rounding of the stored result is an order of magnitude coarser)
// CPL = channels per lane: 4 (128-channel tiles, 2 CTAs/SM at 128 registers) or 2 (64-channel tiles, half the registers per thread
// for window + weights -> 4 CTAs/SM = 32 warps: the kernel is latency-bound, not bandwidth-bound, at 16 warps per SM)
template <int GELU, int CPL>
__global__ void __launch_bounds__(kThreads, CPL == 4 ? 2 : 4)
dwconv3x3_gelu_tma_kernel(const __grid_constant__ CUtensorMap tmap_x, const DwParams p) {
  constexpr int CB = 32 * CPL, NP = CPL / 2;          // channels per tile, f32x2 pairs per lane
  constexpr int kTileB = kBoxH * kBoxW * CB * 2;
  typedef typename std::conditional<CPL == 4, uint2, uint32_t>::type LaneWord;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  __shared__ int4 tile_coord[kMaxStages];  // (cblk, tx, ty, b) of the tile in each stage, written by the producer
  uint8_t* smem = smem_raw + ((128u - (ptx::smem_u32(smem_raw) & 127u)) & 127u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmap_x);
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], p.tw);
    }
    ptx::fence_barrier_init();
  }
  __syncthreads();

  // Every warp is a consumer (warp -> output column, lane -> 4 channels); lane 0 of warp 0 additionally plays TMA
  // producer, issuing the load of tile k+kPrefetch at the top of iteration k.  (A dedicated producer warp would make
  // 9 warps per CTA = 5 on one scheduler at 2 CTAs/SM, capping the kernel at 96 registers; the consumer loop wants more.)
  auto issue_tile = [&](int t, int stage, uint32_t phase) {
    const int cblk = t / p.tiles_per_cblk;
    int r = t - cblk * p.tiles_per_cblk;
    const int per_b = p.tiles_y * p.tiles_x;
    const int b = r / per_b;
    r -= b * per_b;
    const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
    ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
    tile_coord[stage] = make_int4(cblk, tx, ty, b);  // visible to the consumers through the barrier's release/acquire
    ptx::mbar_arrive_expect_tx(&full_bar[stage], static_cast<uint32_t>(kBoxH * (p.tw + 2) * CB * 2));
    ptx::tma_load_4d(smem + stage * kTileB, &tmap_x, &full_bar[stage], cblk * CB, tx * p.tw - 1, ty * kTH - 1, b);
  };
  // each CTA walks one contiguous range of tiles: neighbouring tiles (shared halos) are loaded back to back and the
  // 128-channel weight block in registers changes at most a couple of times per CTA
  const int per_cta = p.num_tiles / static_cast<int>(gridDim.x), extra = p.num_tiles % static_cast<int>(gridDim.x);
  const int t_begin = static_cast<int>(blockIdx.x) * per_cta + min(static_cast<int>(blockIdx.x), extra);
  const int t_end = t_begin + per_cta + (static_cast<int>(blockIdx.x) < extra ? 1 : 0);
  // Measured and NOT adopted (round 2, profiles/r02/order_ab_negative.log): a run-time tile order with the channel block fastest and tiles
  // dealt round-robin (slower: weight reloads, lost halo reuse), and warp 0 as a converged producer with an elect.sync lane (no gain:
  // one TMA per 7 x 8 x 128 outputs is not where this arithmetic-bound kernel spends its time).
  const bool is_producer = threadIdx.x == 0;
  int pt = t_begin, pstage = 0;  // producer cursor
  uint32_t pphase = 0;
  if (is_producer) {
    for (int i = 0; i < p.prefetch && pt < t_end; ++i, ++pt) {
      issue_tile(pt, pstage, pphase);
      if (++pstage == p.stages) { pstage = 0; pphase ^= 1u; }
    }
  }
  const int col = warp;
  const bool active = col < p.tw;
  const int boxw = p.tw + 2;
  int stage = 0;
  uint32_t phase = 0;
  int cur_cblk = -1;
  f32x2 wt[9][NP];
  f32x2 biasv[NP];
#pragma unroll
  for (int q = 0; q < NP; ++q) biasv[q] = 0;
  for (int t = t_begin; t < t_end; ++t) {
    if (is_producer && pt < t_end) {
      issue_tile(pt, pstage, pphase);
      ++pt;
      if (++pstage == p.stages) { pstage = 0; pphase ^= 1u; }
    }
    __syncwarp();
    if (active) {
      ptx::mbar_wait(&full_bar[stage], phase);
      const int4 tc = tile_coord[stage];
      const int cblk = tc.x, tx = tc.y, ty = tc.z, b = tc.w;
      const int c0 = cblk * CB + lane * CPL;
      if (cblk != cur_cblk) {  // weights of this 128-channel block stay in registers across tiles
        cur_cblk = cblk;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          if constexpr (CPL == 4) {
            const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.w9c + tap * p.C + c0));
            wt[tap][0] = f2_pack(w4.x, w4.y);
            wt[tap][NP - 1] = f2_pack(w4.z, w4.w);
          } else {
            const float2 w2 = __ldg(reinterpret_cast<const float2*>(p.w9c + tap * p.C + c0));
            wt[tap][0] = f2_pack(w2.x, w2.y);
          }
        }
        if constexpr (CPL == 4) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + c0));
          biasv[0] = f2_pack(b4.x, b4.y);
          biasv[NP - 1] = f2_pack(b4.z, b4.w);
        } else {
          const float2 b2 = __ldg(reinterpret_cast<const float2*>(p.bias + c0));
          biasv[0] = f2_pack(b2.x, b2.y);
        }
      }
      const int w = tx * p.tw + col;
      const int h0 = ty * kTH;
      // smem tile: [kBoxH][boxw][CB ch] bf16; this thread reads box columns col, col+1, col+2
      const LaneWord* tile = reinterpret_cast<const LaneWord*>(smem + stage * kTileB) + col * 32 + lane;
      const int row_words = boxw * 32;
      auto load_row = [&](int br, f32x2 (&dst)[3][NP]) {
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const LaneWord v = tile[br * row_words + dx * 32];
          if constexpr (CPL == 4) {
            dst[dx][0] = f2_from_bf16x2(v.x);
            dst[dx][NP - 1] = f2_from_bf16x2(v.y);
          } else {
            dst[dx][0] = f2_from_bf16x2(v);
          }
        }
      };
      f32x2 ring[3][3][NP];
      load_row(0, ring[0]);
      load_row(1, ring[1]);
      bf16* optr = p.out + ((static_cast<long long>(b) * p.H + h0) * p.W + w) * p.ldo + c0;
      const int rows_ok = (w < p.W) ? min(kTH, p.H - h0) : 0;  // rows of this tile column that exist
#pragma unroll
      for (int i = 0; i < kTH; ++i) {
        load_row(i + 2, ring[(i + 2) % 3]);
        // three independent 3-tap chains per accumulator (one per window row) instead of one 9-deep chain
        f32x2 a[NP];
#pragma unroll
        for (int q = 0; q < NP; ++q) {
          f32x2 sacc[3];
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            const f32x2 (&rr)[3][NP] = ring[(i + dy) % 3];
            f32x2 t = dy == 0 ? f2_fma(rr[1][q], wt[1][q], biasv[q]) : f2_mul(rr[1][q], wt[dy * 3 + 1][q]);
            t = f2_fma(rr[0][q], wt[dy * 3][q], t);
            sacc[dy] = f2_fma(rr[2][q], wt[dy * 3 + 2][q], t);
          }
          a[q] = f2_add(f2_add(sacc[0], sacc[1]), sacc[2]);
        }
        if constexpr (GELU == 0) {
          if constexpr (CPL == 4) f2_gelu_erf_poly_x2(a[0], a[NP - 1]);
          else a[0] = f2_gelu_erf_poly(a[0]);
        } else {
#pragma unroll
          for (int q = 0; q < NP; ++q) a[q] = GELU == 1 ? f2_gelu_sigmoid(a[q]) : f2_gelu_tanh(a[q]);
        }
        if (i < rows_ok) {
          if constexpr (CPL == 4) {
            float y0, y1, y2, y3;
            f2_unpack(a[0], y0, y1);
            f2_unpack(a[NP - 1], y2, y3);
            uint2 o;
            o.x = pack_bf16x2(y0, y1);
            o.y = pack_bf16x2(y2, y3);
            *reinterpret_cast<uint2*>(optr) = o;
          } else {
            float y0, y1;
            f2_unpack(a[0], y0, y1);
            *reinterpret_cast<uint32_t*>(optr) = pack_bf16x2(y0, y1);
          }
        }
        optr += p.row_stride;
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&empty_bar[stage]);  // this warp is done reading the stage
    }
    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
  }
}

}  // namespace

static int dw_cpl() {
  static const int cpl = [] { const char* e = getenv("SURGVID_DW_CPL"); const int v = e ? atoi(e) : 4; return v == 2 ? 2 : 4; }();
  return cpl;
}
bool dwconv_tma_supported(int C) { return C % kCB == 0; }

int dwconv_tma_shape(int B, int H, int W, int C, int sms, DwconvShape* s) {
  SV_CHECK(B > 0 && H > 0 && W > 0 && sms > 0 && dwconv_tma_supported(C), "dwconv TMA shape");
  static const int env_stages = [] { const char* e = getenv("SURGVID_DW_STAGES"); return e ? atoi(e) : 0; }();
  static const int env_prefetch = [] { const char* e = getenv("SURGVID_DW_PREFETCH"); return e ? atoi(e) : 0; }();
  static const int gelu_mode = [] { const char* e = getenv("SURGVID_DW_GELU"); const int v = e ? atoi(e) : 2; return v == 0 || v == 1 ? v : 2; }();
  s->cpl = dw_cpl();
  s->gelu = gelu_mode;
  s->stages = std::min(kMaxStages, std::max(2, env_stages > 0 ? env_stages : kStages));
  s->prefetch = std::min(s->stages - 1, std::max(1, env_prefetch > 0 ? env_prefetch : kPrefetch));
  s->tw = (W % 8 == 0) ? 8 : ((W % 7 == 0) ? 7 : 8);
  s->tiles_x = ceil_div(W, s->tw);
  s->tiles_y = ceil_div(H, kTH);
  s->cblks = C / (32 * s->cpl);
  const long long nt = static_cast<long long>(s->cblks) * B * s->tiles_y * s->tiles_x;
  if (nt >= (1LL << 31)) return fail(SV_ERR_INVALID, "dwconv: more than 2^31 tiles");
  s->num_tiles = static_cast<int>(nt);
  s->grid = static_cast<int>(std::min<long long>(s->num_tiles, (s->cpl == 4 ? 2LL : 4LL) * sms));
  s->smem_bytes = s->stages * (kBoxH * kBoxW * 32 * s->cpl * 2) + 128;
  return SV_OK;
}

int dwconv_tma_plan(const bf16* x, const float* w9c, const float* bias, int B, int H, int W, int C, bf16* out, int64_t ldo, DwconvPlan* plan) {
  SV_CHECK(ldo >= C && ldo % 4 == 0, "dwconv output row stride");
  SV_CHECK(dwconv_tma_supported(C), "dwconv TMA path needs C % 128 == 0");
  SV_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0, "dwconv alignment");
  DwconvShape s;
  SV_TRY(dwconv_tma_shape(B, H, W, C, 1, &s));   // tw and cpl do not depend on the SM count
  cuuint64_t gdim[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(B)};
  cuuint64_t gstr[3] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(W) * C * 2, static_cast<cuuint64_t>(H) * W * C * 2};
  cuuint32_t box[4] = {static_cast<cuuint32_t>(32 * s.cpl), static_cast<cuuint32_t>(s.tw + 2), kBoxH, 1};
  SV_TRY(encode_tiled(&plan->tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, x, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "dwconv"));
  plan->w9c = w9c; plan->bias = bias; plan->out = out; plan->B = B; plan->H = H; plan->W = W; plan->C = C; plan->ldo = ldo; plan->tw = s.tw;
  plan->cpl = s.cpl;
  return SV_OK;
}

int dwconv_tma_launch(const DwconvPlan& plan, cudaStream_t st) {
  DwconvShape s;
  SV_TRY(dwconv_tma_shape(plan.B, plan.H, plan.W, plan.C, device_sm_count(), &s));
  typedef void (*KernFn)(const CUtensorMap, const DwParams);
  KernFn kern;
  if (plan.cpl == 4) kern = s.gelu == 0 ? dwconv3x3_gelu_tma_kernel<0, 4> : (s.gelu == 1 ? dwconv3x3_gelu_tma_kernel<1, 4> : dwconv3x3_gelu_tma_kernel<2, 4>);
  else kern = s.gelu == 0 ? dwconv3x3_gelu_tma_kernel<0, 2> : (s.gelu == 1 ? dwconv3x3_gelu_tma_kernel<1, 2> : dwconv3x3_gelu_tma_kernel<2, 2>);
  SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(kern), s.smem_bytes));
  DwParams p;
  p.w9c = plan.w9c; p.bias = plan.bias; p.out = plan.out; p.B = plan.B; p.H = plan.H; p.W = plan.W; p.C = plan.C; p.ldo = plan.ldo;
  p.tw = plan.tw;
  p.stages = s.stages; p.prefetch = s.prefetch;
  p.tiles_x = s.tiles_x; p.tiles_y = s.tiles_y; p.cblks = s.cblks;
  p.num_tiles = s.num_tiles;
  p.tiles_per_cblk = plan.B * p.tiles_y * p.tiles_x;
  p.row_stride = static_cast<long long>(plan.W) * plan.ldo;
  kern<<<s.grid, kThreads, s.smem_bytes, st>>>(plan.tmap, p);
  return launch_status("dwconv3x3_gelu_tma_kernel");
}

}  // namespace sv
