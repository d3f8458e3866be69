// Second half of the MixFFN as ONE kernel:   x += fc2( GELU( DWConv3x3(h1) + b_dw ) ) [+ shared_mlp(T_next)]
// (reference: Mlp.forward, mix_transformer_evp.py:60-67 — dwconv :26-29, GELU :64, fc2 :66; the bracketed term is the
// K-concatenated adapter of the next block, see evp.cu).
//
// The stand-alone path writes GELU(DWConv(h1)) (the 4C-wide hidden tensor, the largest activation of the network) to HBM
// and reads it back as the A operand of the fc2 GEMM.  Here the depthwise conv + GELU is the PRODUCER of the GEMM's A tiles:
//
//   warp 0        TMA: (R+2) x (W+2) pixel halo tile of h1, 64 channels at a time (4-D tensor map, OOB zero fill = the conv's
//                 zero padding and the isolation between frames) + the 9 taps and bias of those 64 channels
//   warp 1        TMA: the [N x 64] slice of W_fc2 for the k-block (and, for the adapter tail, the A tile itself)
//   warp 2        one thread issues tcgen05.mma (M = 128 rows = R full image rows of one frame, N = C in 1 or 2 pieces),
//                 fp32 accumulators in TMEM
//   warps 3..10   transform: 3x3 window from the halo tile -> FFMA2 -> erf-GELU -> bf16 -> the 128B-swizzled K-major A tile
//                 in shared memory (generic-proxy stores + fence.proxy.async, then an mbarrier arrive)
//   warps 11..14  epilogue: TMEM -> + bias + fp32 residual x (in place)
//
// An M tile is R consecutive full rows of one frame (R*W <= 128 tokens, contiguous in the token-major tensors), so the halo
// needs no per-tap masks.  HBM traffic per block: h1 once (halo re-reads hit L2) + x read/write; the hidden tensor after the
// GELU never exists in memory.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "gemm_epi.cuh"
#include "host.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sv {
namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kATileBytes = kBlockM * kBlockK * 2;
// Warp roles by warpgroup (setmaxnreg re-balances the register file per 4-warp group):
//   warps 0..3    TMA (h1 halo + taps), TMA (weight slices), MMA issuer, TMA (adapter tail) -> 40 registers
//   warps 4..19   16 transform warps (4 per scheduler: the transform is latency-bound)   -> 72 registers
//   warps 20..23  epilogue, one per TMEM lane quarter                                     -> 152 registers
constexpr int kNTW = 16;                      // transform warps
constexpr int kPPW = kBlockM / 2 / kNTW;      // token pairs per transform warp (4)
constexpr int kFirstTW = 4;
constexpr int kFirstEpi = kFirstTW + kNTW;    // 20
constexpr int kThreads = 32 * (kFirstEpi + 4);  // 768
constexpr int kRegsCtl = 40, kRegsTransform = 72, kRegsEpi = 152;  // 4*40 + 16*72 + 4*152 = 24 * 80 (the launch allocation)
constexpr int kDwBytes = 10 * kBlockK * 4;    // 9 taps + bias, fp32, 64 channels
constexpr int kMaxStages = 4;
constexpr int kTmemCols = 512;
constexpr int kSmemLimit = 232448 - 2048;     // 227 KB per block minus 1 KB alignment slack and 1 KB for the static barriers

struct MixParams {
  int M, N, hidden;
  int kb_h, kb_t, tail_cols;
  int n_split, bn;
  int H, W, R, frames, tiles_y, num_tiles;
  int raw_bytes, raw_stage_bytes, RS, AS, BS;   // ring depths: h1 halo, A tiles, weight slices
  const float* bias;
  float* x;
  long long ldx;
};

__global__ void __launch_bounds__(kThreads, 1)
mixffn_fc2_kernel(const __grid_constant__ CUtensorMap tmap_h1, const __grid_constant__ CUtensorMap tmap_dw,
                  const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_t, const MixParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t raw_full[kMaxStages];
  __shared__ __align__(8) uint64_t raw_empty[kMaxStages];
  __shared__ __align__(8) uint64_t a_full[kMaxStages];
  __shared__ __align__(8) uint64_t a_empty[kMaxStages];
  __shared__ __align__(8) uint64_t b_full[kMaxStages];
  __shared__ __align__(8) uint64_t b_empty[kMaxStages];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ __align__(8) uint64_t tmem_empty_bar;
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int b_stage_bytes = p.N * kBlockK * 2;
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* b_ring = smem + p.AS * kATileBytes;
  uint8_t* raw_ring = b_ring + p.BS * b_stage_bytes;
  float* staging = reinterpret_cast<float*>(raw_ring + p.RS * p.raw_stage_bytes);
  float* bias_smem = staging + 4 * 32 * kStageLd;
  const int n_pad = (p.N + 3) & ~3;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_h1);
    ptx::prefetch_tensormap(&tmap_dw);
  }
  if (warp == 1 && lane == 0) ptx::prefetch_tensormap(&tmap_w);
  if (warp == 3 && lane == 0 && p.kb_t > 0) ptx::prefetch_tensormap(&tmap_t);
  if (warp == 2) {
    if (lane == 0) {
      for (int s = 0; s < kMaxStages; ++s) {
        ptx::mbar_init(&raw_full[s], 1);
        ptx::mbar_init(&raw_empty[s], kNTW);
        ptx::mbar_init(&a_full[s], 1 + kNTW);   // every transform warp + the TMA thread (which brings the adapter-tail tiles)
        ptx::mbar_init(&a_empty[s], 1);
        ptx::mbar_init(&b_full[s], 1);
        ptx::mbar_init(&b_empty[s], 1);
      }
      ptx::mbar_init(&tmem_full_bar, 1);
      ptx::mbar_init(&tmem_empty_bar, 4);
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(&tmem_base_slot, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  const int num_kb = p.kb_h + p.kb_t;
  const int rows_tile = p.R * p.W;
  auto tile_geom = [&](int tile, int& b, int& y0, int& base_row, int& rows_valid) {
    b = tile / p.tiles_y;
    y0 = (tile - b * p.tiles_y) * p.R;
    base_row = (b * p.H + y0) * p.W;
    rows_valid = min(p.R, p.H - y0) * p.W;
  };

  if (warp < kFirstTW) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsCtl));
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA: h1 halo tiles + depthwise weights
    if (lane == 0) {
      int rs = 0;
      uint32_t rphase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        int b, y0, base_row, rows_valid;
        tile_geom(tile, b, y0, base_row, rows_valid);
        for (int kb = 0; kb < p.kb_h; ++kb) {
          ptx::mbar_wait(&raw_empty[rs], rphase ^ 1u);
          uint8_t* dst = raw_ring + rs * p.raw_stage_bytes;
          ptx::mbar_arrive_expect_tx(&raw_full[rs], static_cast<uint32_t>(p.raw_bytes + kDwBytes));
          ptx::tma_load_4d(dst, &tmap_h1, &raw_full[rs], kb * kBlockK, -1, y0 - 1, b);
          ptx::tma_load_2d(dst + p.raw_stage_bytes - kDwBytes, &tmap_dw, &raw_full[rs], kb * kBlockK, 0);
          if (++rs == p.RS) { rs = 0; rphase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ TMA: weight slices (+ adapter-tail A tiles)
    if (lane == 0) {
      int bs = 0;
      uint32_t bphase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&b_empty[bs], bphase ^ 1u);
          uint8_t* sb = b_ring + bs * b_stage_bytes;
          ptx::mbar_arrive_expect_tx(&b_full[bs], static_cast<uint32_t>(b_stage_bytes));
          for (int i = 0; i < p.n_split; ++i) ptx::tma_load_2d(sb + i * p.bn * kBlockK * 2, &tmap_w, &b_full[bs], kb * kBlockK, i * p.bn);
          if (++bs == p.BS) { bs = 0; bphase ^= 1u; }
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ A ring: one arrival per slot; brings the adapter-tail tiles by TMA
    if (lane == 0) {
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        int b, y0, base_row, rows_valid;
        tile_geom(tile, b, y0, base_row, rows_valid);
        for (int kb = 0; kb < num_kb; ++kb) {
          if (kb >= p.kb_h) {
            ptx::mbar_wait(&a_empty[as], aphase ^ 1u);
            ptx::mbar_arrive_expect_tx(&a_full[as], static_cast<uint32_t>(kATileBytes));
            ptx::tma_load_2d(smem + as * kATileBytes, &tmap_t, &a_full[as], (kb - p.kb_h) * kBlockK, base_row);
          } else {
            ptx::mbar_wait(&a_empty[as], aphase ^ 1u);
            ptx::mbar_arrive(&a_full[as]);
          }
          if (++as == p.AS) { as = 0; aphase ^= 1u; }
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = ptx::make_idesc_bf16_f32(kBlockM, p.bn);
      int as = 0, bs = 0;
      uint32_t aphase = 0, bphase = 0, tphase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        ptx::mbar_wait(&tmem_empty_bar, tphase ^ 1u);
        ptx::tc_fence_after();
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&b_full[bs], bphase);
          ptx::mbar_wait(&a_full[as], aphase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + as * kATileBytes);
          const uint32_t sb = ptx::smem_u32(b_ring + bs * b_stage_bytes);
          const uint64_t da = ptx::make_sw128_kmajor_desc(sa);
          int ksteps = kBlockK / 16;
          if (kb >= p.kb_h) ksteps = min(ksteps, (p.tail_cols - (kb - p.kb_h) * kBlockK + 15) / 16);
          for (int kk = 0; kk < ksteps; ++kk) {
            for (int i = 0; i < p.n_split; ++i) {
              const uint64_t db = ptx::make_sw128_kmajor_desc(sb + i * p.bn * kBlockK * 2);
              ptx::umma_f16(tmem_base + static_cast<uint32_t>(i * p.bn), da + static_cast<uint64_t>(kk * 2), db + static_cast<uint64_t>(kk * 2), idesc,
                            (kb | kk) != 0 ? 1u : 0u);
            }
          }
          ptx::umma_commit(&a_empty[as]);
          ptx::umma_commit(&b_empty[bs]);
          if (kb == num_kb - 1) ptx::umma_commit(&tmem_full_bar);
          if (++as == p.AS) { as = 0; aphase ^= 1u; }
          if (++bs == p.BS) { bs = 0; bphase ^= 1u; }
        }
        tphase ^= 1u;
      }
    }
  }
  } else if (warp < kFirstEpi) {
    // ------------------------------------------------------------------ transform warps: DWConv3x3 + GELU -> swizzled A tile
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsTransform));
    const int tw = warp - kFirstTW;
    const int pairs_tile = rows_tile >> 1;
    // geometry of this warp's token pairs (x, x+1) is the same for every tile: precompute byte offsets once
    int raw_off[kPPW];
#pragma unroll
    for (int j = 0; j < kPPW; ++j) {
      const int pj = tw + j * kNTW;
      const int r0 = 2 * pj;
      const int ry = r0 / p.W, x = r0 - ry * p.W;
      raw_off[j] = pj < pairs_tile ? (ry * (p.W + 2) + x) * (kBlockK * 2) + lane * 4 : -1;
    }
    // A-tile byte offset of token row r0 = 2*(tw + 8j): the swizzle term (r0 & 7) = (2*tw) & 7 does not depend on j
    const int a_off0 = 2 * tw * (kBlockK * 2) + ((((lane >> 2) ^ ((2 * tw) & 7))) << 4) + (lane & 3) * 4;
    const int row_bytes = (p.W + 2) * (kBlockK * 2);
    int rs = 0, as = 0;
    uint32_t rphase = 0, aphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < num_kb; ++kb) {
        if (kb < p.kb_h) {
          ptx::mbar_wait(&raw_full[rs], rphase);
          const uint8_t* raw = raw_ring + rs * p.raw_stage_bytes;
          const float2* dw = reinterpret_cast<const float2*>(raw + p.raw_stage_bytes - kDwBytes) + lane;
          f32x2 wt[9];
#pragma unroll
          for (int t = 0; t < 9; ++t) { const float2 w2 = dw[t * (kBlockK / 2)]; wt[t] = f2_pack(w2.x, w2.y); }
          const float2 b2 = dw[9 * (kBlockK / 2)];
          const f32x2 bias2 = f2_pack(b2.x, b2.y);
          ptx::mbar_wait(&a_empty[as], aphase ^ 1u);   // the MMAs that read this A slot have retired
          uint8_t* sa = smem + as * kATileBytes;
#pragma unroll
          for (int j = 0; j < kPPW; ++j) {
            if (raw_off[j] >= 0) {
              const uint8_t* rp = raw + raw_off[j];
              f32x2 a0 = bias2, a1 = bias2;
#pragma unroll
              for (int dy = 0; dy < 3; ++dy) {
                f32x2 v[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) v[c] = f2_from_bf16x2(*reinterpret_cast<const uint32_t*>(rp + dy * row_bytes + c * (kBlockK * 2)));
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                  a0 = f2_fma(v[dx], wt[dy * 3 + dx], a0);
                  a1 = f2_fma(v[dx + 1], wt[dy * 3 + dx], a1);
                }
              }
              f2_gelu_erf_poly_x2(a0, a1);
              float y0, y1, y2, y3;
              f2_unpack(a0, y0, y1);
              f2_unpack(a1, y2, y3);
              const int ao = a_off0 + j * (2 * kNTW * kBlockK * 2);
              *reinterpret_cast<uint32_t*>(sa + ao) = pack_bf16x2(y0, y1);
              *reinterpret_cast<uint32_t*>(sa + ((ao + kBlockK * 2) ^ 16)) = pack_bf16x2(y2, y3);   // row r0+1: swizzle bit 0 flips
            }
          }
          ptx::fence_proxy_async_smem();   // make the generic-proxy stores visible to the tensor core (async proxy)
          __syncwarp();
          if (lane == 0) {
            ptx::mbar_arrive(&a_full[as]);
            ptx::mbar_arrive(&raw_empty[rs]);
          }
          if (++rs == p.RS) { rs = 0; rphase ^= 1u; }
        } else {
          // adapter tail: the A tile arrives by TMA; this warp only keeps the barrier's arrival count uniform
          ptx::mbar_wait(&a_empty[as], aphase ^ 1u);
          if (lane == 0) ptx::mbar_arrive(&a_full[as]);
        }
        if (++as == p.AS) { as = 0; aphase ^= 1u; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (one per TMEM lane quarter)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsEpi));
    const int ew = warp - kFirstEpi;
    const int quarter = warp & 3;
    float* stg = staging + ew * (32 * kStageLd);
    float* bias_s = bias_smem + ew * n_pad;
    const int sub_row = lane >> 3;
    const int c4 = (lane & 7) * 4;
    for (int c = lane * 4; c < n_pad; c += 128) {
      float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.bias != nullptr && c < p.N) b = __ldg(reinterpret_cast<const float4*>(p.bias + c));
      *reinterpret_cast<float4*>(bias_s + c) = b;
    }
    __syncwarp();
    const int nchunks = (p.N + 31) >> 5;
    uint32_t tphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      int b, y0, base_row, rows_valid;
      tile_geom(tile, b, y0, base_row, rows_valid);
      const int row_limit = min(base_row + rows_valid, p.M);
      const int row_base = base_row + quarter * 32 + sub_row;
      {  // pull this warp's rows of x into L2 while the tile's transform/MMAs are still running
        const int prow = base_row + quarter * 32 + lane;
        if (prow < row_limit) {
          const float* rp = p.x + static_cast<long long>(prow) * p.ldx;
          for (int j = 0; j * 32 < p.N; ++j) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + j * 32));
        }
      }
      float4 res_a[8], res_b[8];
      epi_load_residual<true>(res_a, p.x, p.ldx, row_limit, row_base, c4, c4 < p.N);
      ptx::mbar_wait(&tmem_full_bar, tphase);
      ptx::tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
      uint32_t r_a[32], r_b[32];
      ptx::tmem_ld_x32(t_row, r_a);
      for (int c = 0; c < nchunks; c += 2) {
        ptx::tmem_ld_wait();
        epi_park(stg, lane, r_a);
        if (c + 1 < nchunks) {
          ptx::tmem_ld_x32(t_row + static_cast<uint32_t>((c + 1) * 32), r_b);
          epi_load_residual<true>(res_b, p.x, p.ldx, row_limit, row_base, (c + 1) * 32 + c4, (c + 1) * 32 + c4 < p.N);
        }
        __syncwarp();
        epi_store<ACT_NONE, true, true>(p.x, p.ldx, row_limit, stg, bias_s, res_a, row_base, c * 32 + c4, c * 32 + c4, c * 32 + c4 < p.N, sub_row, c4);
        __syncwarp();
        if (c + 1 >= nchunks) break;
        ptx::tmem_ld_wait();
        epi_park(stg, lane, r_b);
        if (c + 2 < nchunks) {
          ptx::tmem_ld_x32(t_row + static_cast<uint32_t>((c + 2) * 32), r_a);
          epi_load_residual<true>(res_a, p.x, p.ldx, row_limit, row_base, (c + 2) * 32 + c4, (c + 2) * 32 + c4 < p.N);
        }
        __syncwarp();
        epi_store<ACT_NONE, true, true>(p.x, p.ldx, row_limit, stg, bias_s, res_b, row_base, (c + 1) * 32 + c4, (c + 1) * 32 + c4, (c + 1) * 32 + c4 < p.N,
                                        sub_row, c4);
        __syncwarp();
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar);
      tphase ^= 1u;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// rows of a tile: the largest R with R*W <= 128, then evened out over the frame height
int pick_rows(int H, int W) {
  const int rmax = std::min(H, kBlockM / W);
  if (rmax < 1) return 0;
  const int tiles_y = ceil_div(H, rmax);
  return ceil_div(H, tiles_y);
}

}  // namespace

bool mixffn_fc2_supported(int H, int W, int hidden, int N, int tail_cols) {
  if (W < 2 || (W & 1) || W + 2 > 256 || W > kBlockM) return false;        // token pairs along x; TMA box limit
  if (hidden % kBlockK != 0 || N % 16 != 0 || N > kTmemCols || tail_cols % 8 != 0) return false;
  if (N > 256 && (N % 32 != 0 || N / 2 > 256)) return false;
  const int R = pick_rows(H, W);
  if (R < 1) return false;
  const int raw_stage = round_up((R + 2) * (W + 2) * kBlockK * 2, 128) + kDwBytes;
  const int fixed = 4 * 32 * kStageLd * 4 + 4 * round_up(N, 4) * 4;
  return 2 * kATileBytes + 2 * N * kBlockK * 2 + 2 * raw_stage + fixed <= kSmemLimit;
}

int mixffn_fc2_plan(const bf16* h1, const float* w10c, const bf16* Wcat, int64_t ldw, const float* bias, const bf16* tail, int64_t ldt,
                    int tail_cols, float* x, int64_t ldx, int frames, int H, int W, int hidden, int N, MixffnPlan* plan) {
  SV_CHECK(h1 && w10c && Wcat && x && plan, "mixffn: null argument");
  SV_CHECK(mixffn_fc2_supported(H, W, hidden, N, tail_cols), "mixffn: unsupported geometry");
  SV_CHECK(tail_cols == 0 || tail != nullptr, "mixffn: tail operand missing");
  SV_CHECK(ldw >= hidden + tail_cols && ldw % 8 == 0 && ldx >= N && ldx % 4 == 0, "mixffn: leading dimensions");
  SV_CHECK((reinterpret_cast<uintptr_t>(h1) & 15) == 0 && (reinterpret_cast<uintptr_t>(Wcat) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(w10c) & 15) == 0,
           "mixffn: operands must be 16-byte aligned");
  const long long Mll = static_cast<long long>(frames) * H * W;
  SV_CHECK(Mll < (1LL << 31), "mixffn: too many tokens");
  MixParams& p = *reinterpret_cast<MixParams*>(plan->params);
  static_assert(sizeof(MixParams) <= sizeof(plan->params), "MixffnPlan::params too small");
  p.M = static_cast<int>(Mll); p.N = N; p.hidden = hidden;
  p.kb_h = hidden / kBlockK;
  p.tail_cols = tail_cols;
  p.kb_t = ceil_div(tail_cols, kBlockK);
  p.n_split = N > 256 ? 2 : 1;
  p.bn = N / p.n_split;
  p.H = H; p.W = W; p.R = pick_rows(H, W); p.frames = frames;
  p.tiles_y = ceil_div(H, p.R);
  p.num_tiles = frames * p.tiles_y;
  p.raw_bytes = (p.R + 2) * (W + 2) * kBlockK * 2;
  p.raw_stage_bytes = round_up(p.raw_bytes, 128) + kDwBytes;
  const int b_stage = N * kBlockK * 2;
  const int fixed = 4 * 32 * kStageLd * 4 + 4 * round_up(N, 4) * 4;
  // ring depths: as deep as shared memory allows, the halo ring first (it hides the HBM latency of h1)
  p.AS = 2; p.BS = 2; p.RS = 2;
  auto total = [&](int as, int bs, int rs) { return as * kATileBytes + bs * b_stage + rs * p.raw_stage_bytes + fixed; };
  while (true) {  // round-robin: weight slices (longest latency), halo tiles, A tiles
    bool grew = false;
    if (p.BS < kMaxStages && total(p.AS, p.BS + 1, p.RS) <= kSmemLimit) { ++p.BS; grew = true; }
    if (p.RS < kMaxStages && total(p.AS, p.BS, p.RS + 1) <= kSmemLimit) { ++p.RS; grew = true; }
    if (p.AS < 3 && total(p.AS + 1, p.BS, p.RS) <= kSmemLimit) { ++p.AS; grew = true; }
    if (!grew) break;
  }
  if (const char* e = getenv("SURGVID_MIXFFN_RINGS")) {  // experiment hook: "A,B,R"
    int a_ = 0, b_ = 0, r_ = 0;
    if (sscanf(e, "%d,%d,%d", &a_, &b_, &r_) == 3 && a_ >= 1 && b_ >= 1 && r_ >= 1 && a_ <= kMaxStages && b_ <= kMaxStages && r_ <= kMaxStages &&
        total(a_, b_, r_) <= kSmemLimit) { p.AS = a_; p.BS = b_; p.RS = r_; }
  }
  p.bias = bias; p.x = x; p.ldx = ldx;
  plan->smem_bytes = static_cast<size_t>(total(p.AS, p.BS, p.RS)) + 1024;
  plan->grid = std::min(p.num_tiles, device_sm_count());
  plan->flops = 2.0 * p.M * static_cast<double>(N) * (hidden + tail_cols);
  {  // h1 as [frames, H, W, hidden] bf16; box = 64 channels x (W+2) x (R+2) x 1, no swizzle (the transform reads pixel rows of 128 B)
    cuuint64_t gdim[4] = {static_cast<cuuint64_t>(hidden), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(frames)};
    cuuint64_t gstr[3] = {static_cast<cuuint64_t>(hidden) * 2, static_cast<cuuint64_t>(W) * hidden * 2, static_cast<cuuint64_t>(H) * W * hidden * 2};
    cuuint32_t box[4] = {kBlockK, static_cast<cuuint32_t>(W + 2), static_cast<cuuint32_t>(p.R + 2), 1};
    SV_TRY(encode_tiled(&plan->tmap_h1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, h1, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "mixffn h1"));
  }
  {  // depthwise taps + bias as fp32 [10, hidden]
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(hidden), 10};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(hidden) * 4};
    cuuint32_t box[2] = {kBlockK, 10};
    SV_TRY(encode_tiled(&plan->tmap_dw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, w10c, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "mixffn dw"));
  }
  {  // [N, hidden + tail] bf16 weight, K-major, 128B swizzle
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(hidden + tail_cols), static_cast<cuuint64_t>(N)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ldw) * 2};
    cuuint32_t box[2] = {kBlockK, static_cast<cuuint32_t>(p.bn)};
    SV_TRY(encode_tiled(&plan->tmap_w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, Wcat, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "mixffn w"));
  }
  if (tail_cols > 0) {
    SV_CHECK((reinterpret_cast<uintptr_t>(tail) & 15) == 0 && ldt % 8 == 0 && ldt >= tail_cols, "mixffn: tail operand alignment");
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(tail_cols), static_cast<cuuint64_t>(p.M)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ldt) * 2};
    cuuint32_t box[2] = {kBlockK, kBlockM};
    SV_TRY(encode_tiled(&plan->tmap_t, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, tail, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "mixffn tail"));
  } else {
    plan->tmap_t = plan->tmap_w;  // never dereferenced
  }
  return SV_OK;
}

int mixffn_fc2_launch(const MixffnPlan& plan, cudaStream_t st) {
  SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mixffn_fc2_kernel), kSmemLimit + 1024));
  const MixParams& p = *reinterpret_cast<const MixParams*>(plan.params);
  mixffn_fc2_kernel<<<plan.grid, kThreads, plan.smem_bytes, st>>>(plan.tmap_h1, plan.tmap_dw, plan.tmap_w, plan.tmap_t, p);
  return launch_status("mixffn_fc2_kernel");
}

}  // namespace sv

extern "C" int sv_op_mixffn_fc2(const uint16_t* h1, const float* w10c, const uint16_t* Wcat, int64_t ldw, const float* bias, const uint16_t* tail,
                                int64_t ldt, int32_t tail_cols, float* x, int64_t ldx, int32_t frames, int32_t H, int32_t W, int32_t hidden,
                                int32_t N, void* stream) {
  sv::MixffnPlan plan;
  SV_TRY(sv::mixffn_fc2_plan(reinterpret_cast<const sv::bf16*>(h1), w10c, reinterpret_cast<const sv::bf16*>(Wcat), ldw, bias,
                             reinterpret_cast<const sv::bf16*>(tail), ldt, tail_cols, x, ldx, frames, H, W, hidden, N, &plan));
  return sv::mixffn_fc2_launch(plan, static_cast<cudaStream_t>(stream));
}
