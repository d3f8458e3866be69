// Persistent, warp-specialised bf16 GEMM for sm_100a:  out = act(A * W^T + bias) (+ residual)
//
//   * operands staged global -> shared by TMA (cp.async.bulk.tensor.2d, 128B swizzle) into an mbarrier ring,
//   * tcgen05.mma (cta_group::1, kind::f16, M=128, N=block_n) issued by ONE thread, fp32 accumulators in TMEM,
//   * two TMEM accumulator buffers so the epilogue of tile i overlaps the MMAs of tile i+1,
//   * epilogue warps read TMEM with tcgen05.ld (thread = accumulator row), transpose 32x32 fp32 blocks through a
//     per-warp shared-memory staging tile so that bias / GELU(erf) / ReLU / fp32 residual add / bf16 cast and the
//     global loads+stores run with 8 lanes on one 128-byte row segment (4 full lines per warp instruction instead of 32).
//
// Every nn.Linear, patchified nn.Conv2d and 1x1 conv of the LFB path goes through this kernel
// (reference: mix_transformer_evp.py:81-84 q/kv/proj, :37-40 fc1/fc2, :188 patch-embed conv, :89 sr conv,
// :599-642 adapter linears, :823-835 flow convs, :868 MHA projections; segformer_head.py:39,74 head).
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..9 = epilogue
// (a warp may only touch TMEM lanes 32*(warp%4) .. +31; two warps share each lane quarter and split the 32-column chunks,
// so every SM sub-partition has two epilogue warps to hide each other's latencies).
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

#include "gemm.cuh"
#include "gemm_epi.cuh"
#include "ptx.cuh"

namespace sv {

#ifdef SV_GEMM_TRACE
__device__ unsigned long long g_trace[4][4096];   // 0 producer (per k-block: slot free), 1 MMA (per k-block: operands landed), 2 MMA per tile (accumulator free), 3 epilogue warp 2 (per tile: 2t = accumulator full, 2t+1 = done)
#define SV_TRACE(role, idx) do { if (blockIdx.x == 0 && (idx) < 4096) g_trace[role][idx] = clock64(); } while (0)
#else
#define SV_TRACE(role, idx) do { } while (0)
#endif

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                       // 64 bf16 = 128 B = one swizzle row
constexpr int kMaxStages = 8;
constexpr int kEpiWarps = 8;                       // two warps per TMEM lane quarter, interleaved over 32-column chunks
constexpr int kThreads = 64 + kEpiWarps * 32;
constexpr int kTmemCols = 512;                    // 2 accumulator buffers x 256 columns
constexpr int kAccStride = 256;
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KB
constexpr int kStagingBytes = kEpiWarps * 32 * kStageLd * 4;  // transposing epilogue, per warp: 32 rows x 36 floats
constexpr int kBiasBytes = kEpiWarps * 256 * 4;   // per epilogue warp: this tile's 256 bias values
constexpr int kMaxEpiBufs = 4;                    // TMA epilogues: 2 KB staging buffers per warp
constexpr int kEpiBufBytes = 2048;
constexpr int kSmemTotal = 230400;                // dynamic shared memory per CTA: 1 KB alignment slack + operand ring + staging + bias

// PAIR = true: the kernel runs as 2-CTA clusters (tcgen05 cta_group::2).  Each CTA stages its own 128 rows of A and HALF of
// the B tile (block_n/2 rows); the leader CTA (cluster rank 0) issues one M=256 MMA per k-step that reads both CTAs' shared
// memory and writes 128 accumulator rows into each CTA's TMEM.  Shared-memory fill traffic per MAC drops by 1/4..1/3, which is
// what bounds the K >= 256 GEMMs of stages 3/4 (operands come from L2, not HBM).
// CONV = true: implicit-GEMM convolution.  tmap_a is an im2col-mode map of the NHWC input (128 pixels x 64 channels per load, same
// 128B-swizzled tile as the 2-D map), and k-block kb is tap (kh, kw), channels c0 .. c0 + 63 — the (kh, kw, cin) order of the packed
// conv weights, so the MMAs see exactly the tiles a materialised im2col buffer would give them.
template <int ACT, bool OUT_F32, bool RESID, bool PAIR, bool CONV>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a2,
                         const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_out,
                         const __grid_constant__ CUtensorMap tmap_res, const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(8) uint64_t res_full[kEpiWarps][kMaxEpiBufs];   // fp32 TMA epilogue: residual chunk landed in the warp's staging buffer

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int S = p.num_stages;
  const uint32_t cta_rank = PAIR ? ptx::cluster_ctarank() : 0u;
  const int b_rows = PAIR ? p.block_n / 2 : p.block_n;   // B-tile rows staged by THIS CTA
  const int b_tile_bytes = b_rows * kBlockK * 2;
  const int stage_bytes = kATileBytes + b_tile_bytes;
  // 128B swizzle needs 1024-byte aligned tiles
  // (offset arithmetic on the __shared__ array keeps the address space visible to the compiler: LDS/STS, not generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  float* staging = reinterpret_cast<float*>(smem + S * stage_bytes);  // epilogue transpose tiles live behind the operand ring
  float* bias_smem = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(staging) + p.staging_bytes);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_a2);
    ptx::prefetch_tensormap(&tmap_w);
    if constexpr (OUT_F32 || !RESID) ptx::prefetch_tensormap(&tmap_out);
    if constexpr (OUT_F32 && RESID) ptx::prefetch_tensormap(&tmap_res);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) {
        ptx::mbar_init(&full_bar[s], 1);
        ptx::mbar_init(&empty_bar[s], 1);
      }
      for (int w = 0; w < kEpiWarps; ++w)
        for (int b = 0; b < kMaxEpiBufs; ++b) ptx::mbar_init(&res_full[w][b], 1);
      for (int a = 0; a < 2; ++a) {
        ptx::mbar_init(&tmem_full_bar[a], 1);
        ptx::mbar_init(&tmem_empty_bar[a], PAIR ? 2 * kEpiWarps : kEpiWarps);  // one arrive per epilogue warp (of both CTAs)
      }
      ptx::fence_barrier_init();
    }
    __syncwarp();
    if (PAIR) {
      ptx::tmem_alloc_pair(&tmem_base_slot, kTmemCols);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(&tmem_base_slot, kTmemCols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if (PAIR) ptx::cluster_sync(); else __syncthreads();   // peer barriers must exist before any remote arrive / multicast commit
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  const int num_kb = (p.K + kBlockK - 1) / kBlockK;
  // persistent schedule: CTAs (or CTA pairs) stride over the tiles (256-row pair tiles when PAIR)
  const int first_tile = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // The whole warp runs the loop in lock step and polls the barriers; one elected lane issues the TMA instructions (see ptx::elect_one).
    {
      int stage = 0, tr_kb = 0;
      uint32_t phase = 0;
      // L2 prefetch cursor: runs p.prefetch k-blocks ahead of the load cursor over this CTA's (tile, k-block) sequence
      int pf_tile = first_tile, pf_kb = 0;
      auto prefetch_next = [&]() {
        if (pf_tile >= p.num_tiles) return;
        const int pm0 = (pf_tile / p.num_n_tiles) * (PAIR ? 2 * kBlockM : kBlockM) + static_cast<int>(cta_rank) * kBlockM;
        if (ptx::elect_one()) ptx::tma_prefetch_l2_2d(&tmap_a, pf_kb * kBlockK, pm0);
        if (++pf_kb == num_kb) { pf_kb = 0; pf_tile += tile_step; }
      };
      for (int i = 0; i < p.prefetch; ++i) prefetch_next();   // 2-D maps only: gemm_plan sets prefetch = 0 for convolutions
      for (int tile = first_tile; tile < p.num_tiles; tile += tile_step) {
        const int m0 = (tile / p.num_n_tiles) * (PAIR ? 2 * kBlockM : kBlockM) + static_cast<int>(cta_rank) * kBlockM;
        const int n0 = (tile % p.num_n_tiles) * p.block_n + static_cast<int>(cta_rank) * b_rows;
        // CONV: input pixel (cw, ch, cn) under output pixel m0 with the window's top-left tap, and the tap / channel cursor of k-block kb
        int cw = 0, ch = 0, cn = 0, tap_w = 0, tap_h = 0, c0 = 0;
        if constexpr (CONV) {
          const int hw = p.conv_ho * p.conv_wo;
          cn = m0 / hw;
          const int r = m0 - cn * hw;
          const int oh = r / p.conv_wo;
          ch = oh * p.conv_stride - p.conv_pad;
          cw = (r - oh * p.conv_wo) * p.conv_stride - p.conv_pad;
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          if (p.prefetch > 0) prefetch_next();
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
          SV_TRACE(0, tr_kb); ++tr_kb;
          uint8_t* sa = smem + stage * stage_bytes;
          uint8_t* sb = sa + kATileBytes;
          const bool seg2 = kb >= p.kb_split;   // second A segment (e.g. the adapter tensor next to the MixFFN hidden)
          const CUtensorMap* ma = seg2 ? &tmap_a2 : &tmap_a;
          const int ka = (seg2 ? kb - p.kb_split : kb) * kBlockK;
          if (ptx::elect_one()) {
            if (PAIR) {
              // the leader's barrier collects the bytes of both CTAs; only the leader posts the expectation
              if (cta_rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], static_cast<uint32_t>(2 * stage_bytes));
              if constexpr (CONV) ptx::tma_load_im2col_4d_pair(sa, &tmap_a, &full_bar[stage], c0, cw, ch, cn, static_cast<uint16_t>(tap_w), static_cast<uint16_t>(tap_h));
              else ptx::tma_load_2d_pair(sa, ma, &full_bar[stage], ka, m0);
              ptx::tma_load_2d_pair(sb, &tmap_w, &full_bar[stage], kb * kBlockK, n0);
            } else {
              ptx::mbar_arrive_expect_tx(&full_bar[stage], static_cast<uint32_t>(stage_bytes));
              if constexpr (CONV) ptx::tma_load_im2col_4d(sa, &tmap_a, &full_bar[stage], c0, cw, ch, cn, static_cast<uint16_t>(tap_w), static_cast<uint16_t>(tap_h));
              else ptx::tma_load_2d(sa, ma, &full_bar[stage], ka, m0);
              ptx::tma_load_2d(sb, &tmap_w, &full_bar[stage], kb * kBlockK, n0);
            }
          }
          __syncwarp();
          if constexpr (CONV) {
            c0 += kBlockK;
            if (c0 == p.conv_c) {
              c0 = 0;
              if (++tap_w == p.conv_k) { tap_w = 0; ++tap_h; }
            }
          }
          if (++stage == S) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // Converged warp, one elected lane issues: four tcgen05.mma per 64-deep k-block, fully unrolled, then the commits.  (Measured,
    // scripts/ubench/umma_rate.cu: a single divergent thread with a run-time k-step loop needs ~195 cycles per N = 256 MMA against
    // the pipe's 128; this form reaches 128.)
    if (cta_rank == 0) {
      const uint32_t idesc = ptx::make_idesc_bf16_f32(PAIR ? 2 * kBlockM : kBlockM, p.block_n);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0, tr_kb = 0, tr_tile = 0;
      uint32_t acc_phase = 0;
      for (int tile = first_tile; tile < p.num_tiles; tile += tile_step) {
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1u);  // epilogue has drained this accumulator
        SV_TRACE(2, tr_tile); ++tr_tile;
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * kAccStride);
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          SV_TRACE(1, tr_kb); ++tr_kb;
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * stage_bytes);
          const uint64_t da = ptx::make_sw128_kmajor_desc(sa);
          const uint64_t db = ptx::make_sw128_kmajor_desc(sa + kATileBytes);
          const int k_left = p.K - kb * kBlockK;
          const bool last = kb == num_kb - 1;
          // advance 16 bf16 = 32 B along K inside the swizzle row: +2 in the (addr>>4) start-address field
          if (k_left >= kBlockK) {
            if (ptx::elect_one()) {
#pragma unroll
              for (int kk = 0; kk < kBlockK / 16; ++kk) {
                const uint32_t accum = (kk != 0 || kb != 0) ? 1u : 0u;
                if (PAIR) ptx::umma_f16_pair(d_tmem, da + static_cast<uint64_t>(kk * 2), db + static_cast<uint64_t>(kk * 2), idesc, accum);
                else ptx::umma_f16(d_tmem, da + static_cast<uint64_t>(kk * 2), db + static_cast<uint64_t>(kk * 2), idesc, accum);
              }
              if (PAIR) {
                ptx::umma_commit_pair(&empty_bar[stage], 0x3);                 // both CTAs' smem slots
                if (last) ptx::umma_commit_pair(&tmem_full_bar[acc], 0x3);     // both CTAs' epilogues
              } else {
                ptx::umma_commit(&empty_bar[stage]);                           // smem slot reusable once these MMAs retire
                if (last) ptx::umma_commit(&tmem_full_bar[acc]);               // accumulator ready for the epilogue
              }
            }
          } else {
            const int ksteps = (k_left + 15) / 16;   // ragged K tail (TMA zero-fills the rest of the row)
            if (ptx::elect_one()) {
              for (int kk = 0; kk < ksteps; ++kk) {
                const uint32_t accum = (kk != 0 || kb != 0) ? 1u : 0u;
                if (PAIR) ptx::umma_f16_pair(d_tmem, da + static_cast<uint64_t>(kk * 2), db + static_cast<uint64_t>(kk * 2), idesc, accum);
                else ptx::umma_f16(d_tmem, da + static_cast<uint64_t>(kk * 2), db + static_cast<uint64_t>(kk * 2), idesc, accum);
              }
              if (PAIR) {
                ptx::umma_commit_pair(&empty_bar[stage], 0x3);
                if (last) ptx::umma_commit_pair(&tmem_full_bar[acc], 0x3);
              } else {
                ptx::umma_commit(&empty_bar[stage]);
                if (last) ptx::umma_commit(&tmem_full_bar[acc]);
              }
            }
          }
          __syncwarp();
          if (++stage == S) { stage = 0; phase ^= 1u; }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    const int quarter = warp & 3;        // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;    // 0: even 32-column chunks, 1: odd chunks
    bool done = false;
    if constexpr (!OUT_F32 && !RESID) {
      if (p.tma_out) {
      done = true;
      // bf16 result, no residual (fc1, q, kv, sr, adapter, flow and head projections): thread = accumulator row all the way.
      // bias / activation / bf16 pack in registers, 64 bytes per row into a per-warp staging tile in the 64B-swizzled layout of a
      // 2-D TMA store (box 32 columns x 32 rows; ragged M / N edges are clipped by the tensor map) — no transposition through
      // shared memory and no per-thread global stores.  (ncu, round 2: the transposing epilogue ran the L1TEX LSU data pipe at
      // 72-75 % on these GEMMs — 81 shared/global wavefronts per 32x32 block against 24 here.)
      const uint32_t nb = static_cast<uint32_t>(p.epi_bufs);
      uint8_t* sbase = reinterpret_cast<uint8_t*>(staging) + (warp - 2) * p.epi_bufs * kEpiBufBytes;   // nb 2 KB buffers, 1 KB aligned
      float* bias_s = bias_smem + (warp - 2) * 256;
      int acc = 0;
      uint32_t acc_phase = 0;
      uint32_t n_store = 0;   // stores issued by this warp so far (lane 0's bulk groups)
      int tr_tile = 0;
      for (int tile = first_tile; tile < p.num_tiles; tile += tile_step) {
        const int m0 = (tile / p.num_n_tiles) * (PAIR ? 2 * kBlockM : kBlockM) + static_cast<int>(cta_rank) * kBlockM;
        const int n0 = (tile % p.num_n_tiles) * p.block_n;
        const int n_valid = min(p.block_n, p.N - n0);
        const int nchunks = (n_valid + 31) >> 5;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c = i * 128 + lane * 4;
          float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias != nullptr && c < n_valid) b = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c));
          *reinterpret_cast<float4*>(bias_s + c) = b;
        }
        __syncwarp();
        ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
        if (warp == 2) SV_TRACE(3, 16 * tr_tile);
        ptx::tc_fence_after();
        const uint32_t t_row = tmem_base + static_cast<uint32_t>(acc * kAccStride) + (static_cast<uint32_t>(quarter * 32) << 16);
        uint32_t r_a[32], r_b[32];
        if (half < nchunks) ptx::tmem_ld_x32(t_row + static_cast<uint32_t>(half * 32), r_a);
        auto emit = [&](const uint32_t (&r)[32], int c) {
          uint8_t* sb = sbase + (n_store % nb) * kEpiBufBytes;
          if (warp == 2) SV_TRACE(3, 16 * tr_tile + 1 + 3 * (c >> 1));
          if (n_store >= nb) {   // the store issued from this buffer nb chunks ago has finished reading it
            if (ptx::elect_one()) ptx::bulk_wait_group_read(static_cast<int>(nb) - 1);
            __syncwarp();
          }
          if (warp == 2) SV_TRACE(3, 16 * tr_tile + 2 + 3 * (c >> 1));
          uint32_t w[16];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bias_s + c * 32 + i);
            // packed adds (one FADD2 per two columns: the epilogue shares four issue ports with seven other warps)
            f32x2 lo = f2_add(f2_pack(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), f2_pack(b4.x, b4.y));
            f32x2 hi = f2_add(f2_pack(__uint_as_float(r[i + 2]), __uint_as_float(r[i + 3])), f2_pack(b4.z, b4.w));
            if constexpr (ACT == ACT_GELU) f2_gelu_erf_poly_x2(lo, hi);
            float v0, v1, v2, v3;
            f2_unpack(lo, v0, v1);
            f2_unpack(hi, v2, v3);
            if constexpr (ACT == ACT_RELU) {
              v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f);
            }
            w[i >> 1] = pack_bf16x2(v0, v1);
            w[(i >> 1) + 1] = pack_bf16x2(v2, v3);
          }
          const int x = (lane >> 1) & 3;   // 64B swizzle: 16-byte chunk j of row r lives at r*64 + ((j ^ ((r >> 1) & 3)) << 4)
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<uint4*>(sb + lane * 64 + ((j ^ x) << 4)) = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (ptx::elect_one()) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmap_out)),
                         "r"(ptx::smem_u32(sb)), "r"(n0 + c * 32), "r"(m0 + quarter * 32)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          if (warp == 2) SV_TRACE(3, 16 * tr_tile + 3 + 3 * (c >> 1));
          ++n_store;
        };
        for (int c = half; c < nchunks; c += 4) {
          ptx::tmem_ld_wait();
          if (c + 2 < nchunks) ptx::tmem_ld_x32(t_row + static_cast<uint32_t>((c + 2) * 32), r_b);
          emit(r_a, c);
          if (c + 2 >= nchunks) break;
          ptx::tmem_ld_wait();
          if (c + 4 < nchunks) ptx::tmem_ld_x32(t_row + static_cast<uint32_t>((c + 4) * 32), r_a);
          emit(r_b, c + 2);
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) ptx::mbar_arrive_cluster(ptx::map_to_cta(ptx::smem_u32(&tmem_empty_bar[acc]), 0u));   // the leader's MMA warp owns both TMEMs
          else ptx::mbar_arrive(&tmem_empty_bar[acc]);
        }
        if (warp == 2) SV_TRACE(3, 16 * tr_tile + 15);
        ++tr_tile;
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      if (ptx::elect_one()) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory stays valid until the last store has read it
      }
    }
    if constexpr (OUT_F32) {
      if (p.tma_out) {
      done = true;
      // fp32 result, optionally read-modify-write of an fp32 residual (proj / fc2 / shared: x += ...): thread = accumulator row; the
      // residual arrives by 2-D TMA loads (box 16 columns x 32 rows, 64-byte swizzle) into a per-warp ring of nb 2 KB buffers, the
      // row is updated in place in shared memory and leaves through a TMA store of the same box.  The ring runs CONTINUOUSLY over
      // the warp's chunks of all its tiles: after the store of chunk i the warp waits only until the store of chunk i - lag has
      // finished reading its buffer and hands that buffer to the load of chunk i - lag + nb, so nb - lag residual loads and lag
      // result stores are in flight per warp, across tile boundaries (the residual of the next tile streams in while this tile's
      // MMAs and epilogue are still running).  No transposition, no per-thread global loads/stores.
      // (Round 2 measurement that led here, profiles/r02/gemm_operand_stream_experiment.log: with NO operand loads at all the
      // K = 1360 residual GEMM took 177 of 202 us — the kernel was bound by this epilogue: a 2-deep ring and a blocking wait for
      // every store kept only ~3 KB per warp in flight.)
      const uint32_t nb = static_cast<uint32_t>(p.epi_bufs), lag = static_cast<uint32_t>(p.epi_lag);
      uint8_t* sbase = reinterpret_cast<uint8_t*>(staging) + (warp - 2) * p.epi_bufs * kEpiBufBytes;   // nb 2 KB buffers, 1 KB aligned
      float* bias_s = bias_smem + (warp - 2) * 256;
      uint64_t* rbar = res_full[warp - 2];
      int acc = 0;
      uint32_t acc_phase = 0;
      uint32_t n_chunk = 0;    // chunks this warp has processed so far: buffer = n_chunk % nb, barrier parity = (n_chunk / nb) & 1
      uint32_t n_loaded = 0;   // residual loads issued so far (same numbering)
      int tr_tile = 0;
      const int x = (lane >> 1) & 3;   // 64B swizzle: 16-byte piece j of row r lives at r*64 + ((j ^ ((r >> 1) & 3)) << 4)
      const int m_step = PAIR ? 2 * kBlockM : kBlockM;
      auto chunks_of = [&](int n0) {   // this warp takes the 16-column chunks half, half + 2, ... of a tile
        const int nch16 = (min(p.block_n, p.N - n0) + 15) >> 4;
        return (nch16 - half + 1) >> 1;
      };
      int ld_tile = first_tile, ld_k = 0;   // residual load cursor
      auto issue_load = [&]() {
        while (ld_tile < p.num_tiles) {
          const int ln0 = (ld_tile % p.num_n_tiles) * p.block_n;
          if (ld_k < chunks_of(ln0)) {
            if (ptx::elect_one()) {
              const uint32_t slot = n_loaded % nb;
              const int lm0 = (ld_tile / p.num_n_tiles) * m_step + static_cast<int>(cta_rank) * kBlockM;
              ptx::mbar_arrive_expect_tx(&rbar[slot], static_cast<uint32_t>(kEpiBufBytes));
              ptx::tma_load_2d(sbase + slot * kEpiBufBytes, &tmap_res, &rbar[slot], ln0 + (half + 2 * ld_k) * 16, lm0 + quarter * 32);
            }
            ++n_loaded;
            ++ld_k;
            return;
          }
          ld_k = 0;
          ld_tile += tile_step;
        }
      };
      if constexpr (RESID) {
        for (uint32_t i = 0; i < nb - lag; ++i) issue_load();
      }
      for (int tile = first_tile; tile < p.num_tiles; tile += tile_step) {
        const int m0 = (tile / p.num_n_tiles) * m_step + static_cast<int>(cta_rank) * kBlockM;
        const int n0 = (tile % p.num_n_tiles) * p.block_n;
        const int n_valid = min(p.block_n, p.N - n0);
        const int my_chunks = chunks_of(n0);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c = i * 128 + lane * 4;
          float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias != nullptr && c < n_valid) b = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c));
          *reinterpret_cast<float4*>(bias_s + c) = b;
        }
        __syncwarp();
        ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
        if (warp == 2) SV_TRACE(3, 16 * tr_tile);
        ptx::tc_fence_after();
        const uint32_t t_row = tmem_base + static_cast<uint32_t>(acc * kAccStride) + (static_cast<uint32_t>(quarter * 32) << 16);
        uint32_t r_a[16], r_b[16];
        if (my_chunks > 0) ptx::tmem_ld_x16(t_row + static_cast<uint32_t>(half * 16), r_a);
        auto emit = [&](const uint32_t (&r)[16], int k) {
          const int c16 = half + 2 * k;
          const uint32_t slot = n_chunk % nb;
          uint8_t* sb = sbase + slot * kEpiBufBytes;
          float* rowp = reinterpret_cast<float*>(sb + lane * 64);
          if constexpr (RESID) {
            ptx::mbar_wait(&rbar[slot], (n_chunk / nb) & 1u);
          } else {
            if (n_chunk >= nb) {   // the store issued from this buffer nb chunks ago has finished reading it
              if (ptx::elect_one()) ptx::bulk_wait_group_read(static_cast<int>(nb) - 1);
              __syncwarp();
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float4* pp = reinterpret_cast<float4*>(rowp + ((j ^ x) << 2));
            const float4 b4 = *reinterpret_cast<const float4*>(bias_s + c16 * 16 + j * 4);
            f32x2 lo = f2_add(f2_pack(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1])), f2_pack(b4.x, b4.y));       // packed adds: half
            f32x2 hi = f2_add(f2_pack(__uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3])), f2_pack(b4.z, b4.w));   // the issue slots
            if constexpr (ACT != ACT_NONE) {
              float4 a;
              f2_unpack(lo, a.x, a.y);
              f2_unpack(hi, a.z, a.w);
              if constexpr (ACT == ACT_GELU) {
                a.x = gelu_erf(a.x); a.y = gelu_erf(a.y); a.z = gelu_erf(a.z); a.w = gelu_erf(a.w);
              } else {
                a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f);
              }
              lo = f2_pack(a.x, a.y);
              hi = f2_pack(a.z, a.w);
            }
            if constexpr (RESID) {
              const float4 q = *pp;
              lo = f2_add(lo, f2_pack(q.x, q.y));
              hi = f2_add(hi, f2_pack(q.z, q.w));
            }
            float4 v;
            f2_unpack(lo, v.x, v.y);
            f2_unpack(hi, v.z, v.w);
            *pp = v;
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (ptx::elect_one()) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmap_out)),
                         "r"(ptx::smem_u32(sb)), "r"(n0 + c16 * 16), "r"(m0 + quarter * 32)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            // the buffer of chunk n_chunk - lag is free once its store has read it: at most lag younger stores may still be pending
            if constexpr (RESID) ptx::bulk_wait_group_read(static_cast<int>(lag));
          }
          ++n_chunk;
          if constexpr (RESID) issue_load();   // chunk n_chunk - 1 - lag + nb, into the buffer just freed
        };
        for (int k = 0; k < my_chunks; k += 2) {
          ptx::tmem_ld_wait();
          if (k + 1 < my_chunks) ptx::tmem_ld_x16(t_row + static_cast<uint32_t>((half + 2 * (k + 1)) * 16), r_b);
          emit(r_a, k);
          if (k + 1 >= my_chunks) break;
          ptx::tmem_ld_wait();
          if (k + 2 < my_chunks) ptx::tmem_ld_x16(t_row + static_cast<uint32_t>((half + 2 * (k + 2)) * 16), r_a);
          emit(r_b, k + 1);
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) ptx::mbar_arrive_cluster(ptx::map_to_cta(ptx::smem_u32(&tmem_empty_bar[acc]), 0u));
          else ptx::mbar_arrive(&tmem_empty_bar[acc]);
        }
        if (warp == 2) SV_TRACE(3, 16 * tr_tile + 15);
        ++tr_tile;
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      if (ptx::elect_one()) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory stays valid until the last store has read it
      }
    }
    if (!done) {
    float* stg = staging + (warp - 2) * (32 * kStageLd);
    float* bias_s = bias_smem + (warp - 2) * 256;
    const int sub_row = lane >> 3;  // 4 rows per warp instruction
    const int c4 = (lane & 7) * 4;  // 8 lanes x 4 columns = one 32-column row segment
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t leader_tmem_empty0 = PAIR ? ptx::map_to_cta(ptx::smem_u32(&tmem_empty_bar[0]), 0u) : 0u;
    for (int tile = first_tile; tile < p.num_tiles; tile += tile_step) {
      const int m0 = (tile / p.num_n_tiles) * (PAIR ? 2 * kBlockM : kBlockM) + static_cast<int>(cta_rank) * kBlockM;
      const int n0 = (tile % p.num_n_tiles) * p.block_n;
      const int n_valid = min(p.block_n, p.N - n0);
      const int nchunks = (n_valid + 31) >> 5;
      const int row_base = m0 + quarter * 32 + sub_row;
      // while the MMAs of this tile are still running: bias slice -> smem, first residual rows -> registers
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = i * 128 + lane * 4;
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias != nullptr && c < n_valid) b = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c));
        *reinterpret_cast<float4*>(bias_s + c) = b;
      }
      if constexpr (RESID) {
        // pull this warp's share of the residual tile into L2 now, while the MMAs of the tile are still running: the residual
        // stream comes from HBM and one chunk of register prefetch cannot cover that latency
        const int prow = m0 + quarter * 32 + lane;
        if (prow < p.M) {
          const float* rp = p.residual + static_cast<long long>(prow) * p.ldr + n0;
          for (int j = half; j * 32 < n_valid; j += 2) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + j * 32));
        }
      }
      float4 res_a[8], res_b[8];
      epi_load_residual<RESID>(res_a, p.residual, p.ldr, p.M, row_base, n0 + half * 32 + c4, half * 32 + c4 < n_valid);
      __syncwarp();
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t t_row = tmem_base + static_cast<uint32_t>(acc * kAccStride) + (static_cast<uint32_t>(quarter * 32) << 16);
      uint32_t r_a[32], r_b[32];
      if (half < nchunks) ptx::tmem_ld_x32(t_row + static_cast<uint32_t>(half * 32), r_a);
      // two-deep software pipeline over this warp's chunks (c, c+2, ...): the TMEM load and residual load of the next chunk
      // overlap the stores of the current one
      for (int c = half; c < nchunks; c += 4) {
        ptx::tmem_ld_wait();
        epi_park(stg, lane, r_a);
        if (c + 2 < nchunks) {
          ptx::tmem_ld_x32(t_row + static_cast<uint32_t>((c + 2) * 32), r_b);
          epi_load_residual<RESID>(res_b, p.residual, p.ldr, p.M, row_base, n0 + (c + 2) * 32 + c4, (c + 2) * 32 + c4 < n_valid);
        }
        __syncwarp();
        epi_store<ACT, OUT_F32, RESID>(p.out, p.ldc, p.M, stg, bias_s, res_a, row_base, n0 + c * 32 + c4, c * 32 + c4, c * 32 + c4 < n_valid, sub_row, c4);
        __syncwarp();
        if (c + 2 >= nchunks) break;
        ptx::tmem_ld_wait();
        epi_park(stg, lane, r_b);
        if (c + 4 < nchunks) {
          ptx::tmem_ld_x32(t_row + static_cast<uint32_t>((c + 4) * 32), r_a);
          epi_load_residual<RESID>(res_a, p.residual, p.ldr, p.M, row_base, n0 + (c + 4) * 32 + c4, (c + 4) * 32 + c4 < n_valid);
        }
        __syncwarp();
        epi_store<ACT, OUT_F32, RESID>(p.out, p.ldc, p.M, stg, bias_s, res_b, row_base, n0 + (c + 2) * 32 + c4, (c + 2) * 32 + c4, (c + 2) * 32 + c4 < n_valid,
                                       sub_row, c4);
        __syncwarp();
      }
      // every TMEM read of this warp has completed (the last tcgen05.wait::ld is behind us): release the accumulator
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) ptx::mbar_arrive_cluster(leader_tmem_empty0 + static_cast<uint32_t>(acc) * 8u);  // the leader's MMA warp owns both TMEMs
        else ptx::mbar_arrive(&tmem_empty_bar[acc]);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
    }
  }

  ptx::tc_fence_before();
  if (PAIR) ptx::cluster_sync(); else __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if (PAIR) ptx::tmem_dealloc_pair(tmem_base, kTmemCols);
    else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 2-D bf16 row-major [rows, cols] tensor, row stride ld elements; box = [box_rows, 64 cols], 128B swizzle, zero OOB fill.
int encode_operand_map(CUtensorMap* map, const bf16* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) return fail(SV_ERR_CUDA, "cuTensorMapEncodeTiled driver entry point unavailable (no CUDA driver?)");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(SV_ERR_INVALID, "GEMM operand base must be 16-byte aligned");
  if ((ld * 2) % 16 != 0) return fail(SV_ERR_INVALID, "GEMM operand row stride must be a multiple of 8 elements");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kBlockK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed (CUresult %d) rows=%lld cols=%lld ld=%lld box_rows=%d", static_cast<int>(r),
             static_cast<long long>(rows), static_cast<long long>(cols), static_cast<long long>(ld), box_rows);
    return fail(SV_ERR_CUDA, buf);
  }
  return SV_OK;
}

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const int*,
                                  const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeIm2colFn get_encode_im2col_fn() {
  static EncodeIm2colFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeIm2colFn>(p);
  });
  return fn;
}

// im2col-mode map of an NHWC bf16 conv input: each load is one 128-pixel column of one tap, 64 channels (128 B) per pixel, 128B swizzle —
// the tile a 2-D map with box [128 rows, 64 cols] writes.  The bounding box [-pad, W - 1 + pad - (k - 1)] (and the same along H), walked
// with the conv stride, holds exactly the Ho x Wo window origins; zero OOB fill is the conv's padding and the rows past M.
int encode_im2col_map(CUtensorMap* map, const bf16* base, const ConvGeom& g) {
  EncodeIm2colFn fn = get_encode_im2col_fn();
  if (fn == nullptr) return fail(SV_ERR_CUDA, "cuTensorMapEncodeIm2col driver entry point unavailable (no CUDA driver?)");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(SV_ERR_INVALID, "conv GEMM input must be 16-byte aligned");
  const cuuint64_t es = 2;
  cuuint64_t gdim[4] = {static_cast<cuuint64_t>(g.C), static_cast<cuuint64_t>(g.W), static_cast<cuuint64_t>(g.H), static_cast<cuuint64_t>(g.B)};
  cuuint64_t gstride[3] = {gdim[0] * es, gdim[0] * gdim[1] * es, gdim[0] * gdim[1] * gdim[2] * es};
  const int lower[2] = {-g.pad, -g.pad};
  const int upper[2] = {g.pad - (g.k - 1), g.pad - (g.k - 1)};
  cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(g.stride), static_cast<cuuint32_t>(g.stride), 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<bf16*>(base), gdim, gstride, lower, upper, kBlockK, kBlockM, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof(buf), "cuTensorMapEncodeIm2col failed (CUresult %d) B=%d H=%d W=%d C=%d k=%d stride=%d pad=%d", static_cast<int>(r), g.B, g.H,
             g.W, g.C, g.k, g.stride, g.pad);
    return fail(SV_ERR_CUDA, buf);
  }
  return SV_OK;
}

// Host-side checks of a convolution's geometry; no device access.
int check_conv_args(const ConvGeom& g) {
  SV_CHECK(g.B > 0 && g.H > 0 && g.W > 0 && g.C > 0 && g.k > 0 && g.stride > 0 && g.pad >= 0, "conv GEMM: B, H, W, C, k, stride must be positive, pad >= 0");
  SV_CHECK(g.Ho() > 0 && g.Wo() > 0 && g.H + 2 * g.pad >= g.k && g.W + 2 * g.pad >= g.k, "conv GEMM: the kernel window does not fit the padded input");
  SV_CHECK(static_cast<int64_t>(g.B) * g.Ho() * g.Wo() < (1LL << 31) && static_cast<int64_t>(g.k) * g.k * g.C < (1LL << 31), "conv GEMM: M or K too large");
  return SV_OK;
}
// argument errors -> SV_ERR_INVALID, geometry the im2col map cannot express -> SV_ERR_UNSUPPORTED
int check_conv(const ConvGeom& g) {
  SV_TRY(check_conv_args(g));
  if (!conv_gemm_im2col_ok(g))
    return fail(SV_ERR_UNSUPPORTED, "conv GEMM: needs C % 64 == 0, stride <= 8 and padding corners -pad, pad - (k - 1) within [-128, 127] (got C=" +
                                        std::to_string(g.C) + " k=" + std::to_string(g.k) + " stride=" + std::to_string(g.stride) + " pad=" +
                                        std::to_string(g.pad) + "); gather with sv_op_im2col and use sv_op_gemm_bf16");
  return SV_OK;
}

}  // namespace

bool conv_gemm_im2col_ok(const ConvGeom& g) {
  const int upper = g.pad - (g.k - 1);
  return g.k > 0 && g.C % kBlockK == 0 && g.stride >= 1 && g.stride <= 8 && g.pad >= 0 && g.pad <= 128 && upper >= -128 && upper <= 127;
}

int gemm_pick_block_n(int M, int N, int K, int num_sms, int step) {
  // Candidates are legal UMMA N for M=128 (multiples of 16, <= 256).  Model: time ~ waves * (per-tile cost),
  // per-tile cost ~ fixed epilogue/pipeline overhead + N_tile * (k-blocks + epilogue share).
  // Per-tile cycle model (per SM): the slowest of
  //   MMA issue        2*c cycles per 64-deep k-block (tcgen05 floor 128*c/256 per K=16 instruction),
  //   operand staging  (128 + c) * 128 bytes per k-block over ~48 B/cycle/SM of L2->SM bandwidth (A is re-read once per n-tile),
  //   epilogue         ~6 cycles per accumulator column for the warp's 32-row slab + fixed latency,
  // times the number of waves of the persistent grid.
  // step = 32 when the result leaves through 32-column TMA store boxes: a tile's column range must then end on a multiple of 32 or
  // at the edge of the tensor (where the box is clipped), never in the middle of a neighbouring tile
  const int n_pad = round_up(N, step);
  const int m_tiles = ceil_div(M, kBlockM);
  const int kb = ceil_div(K, kBlockK);
  double best_cost = 1e30;
  int best = step;
  for (int c = 256; c >= step; c -= step) {
    if (c > n_pad) continue;
    const int n_tiles = ceil_div(N, c);
    const long long tiles = static_cast<long long>(m_tiles) * n_tiles;
    const long long waves = (tiles + num_sms - 1) / num_sms;
    const double mma = 2.0 * c * kb;
    const double load = (128.0 + c) * 128.0 * kb / 48.0;
    const double epi = 6.0 * round_up(c, 32) + 400.0;
    const double per_tile = std::max(mma, std::max(load, epi)) + 150.0;
    const double cost = waves * per_tile;
    if (cost < best_cost - 1e-9) { best_cost = cost; best = c; }
  }
  return best;
}

// Every decision of the plan that depends only on the problem's shape, the SM count and the A/B switches: tile width, pair mode,
// epilogue form, ring depth, epilogue buffers, tiles and grid.  Host only (no device, no driver); gemm_plan launches by it and
// sv_op_gemm_plan_info reports it.
int gemm_plan_shape(int M, int N, int K, int K2, int out_fp32, bool has_residual, int pair_request, int sms, GemmPlan* plan) {
  GemmParams& p = plan->p;
  p.M = M; p.N = N; p.K = K;
  static const int tma_out_env = getenv("SURGVID_GEMM_TMA_OUT") ? atoi(getenv("SURGVID_GEMM_TMA_OUT")) : 1;   // A/B switch
  // bf16 result without residual, or fp32 result with / without an fp32 residual (the bf16 + residual combination keeps the transposing
  // epilogue).  The fp32 TMA maps need 16-byte row strides, which the argument checks (ldc, ldr % 4 == 0) already guarantee.
  p.tma_out = ((out_fp32 || !has_residual) && tma_out_env) ? 1 : 0;
  p.block_n = gemm_pick_block_n(M, N, K, sms, (p.tma_out && !out_fp32) ? 32 : 16);
  // CTA-pair mode (cta_group::2): each CTA stages half of the B tile, so the ring holds more k-blocks per byte of shared memory
  // and the L2 -> shared-memory traffic of the weights halves.  Measured on B200 (profiles/r02/gemm_pair_relaxed_arrive.log, after
  // (1) the MMA issue moved to a converged warp + elect.sync and (2) the accumulator hand-back stopped using a .release.cluster
  // arrive, which had cost every epilogue warp ~1 800 cycles per tile): 143.7 -> 129.1 us (156 800 x 1280 x 320), 185 -> 173 us
  // (x 320 x 1360 + residual), 1 025 -> 912 us (39 200 x 2048 x 8192 = 1.44 PFLOP/s), 228 -> 197 us (112 700 x 2048 x 512); a tie
  // (+-2 %) on the fp32 read-modify-write GEMMs with K <= 320, whose time is the residual stream's.  'auto' (-1) enables it when
  // there are enough 256-row tiles to fill the machine and either K >= 512 or the result is bf16 with N >= 320;
  // GemmDesc::pair / SURGVID_GEMM_PAIR force it on (1) or off (0).  Results are bit-identical to single-CTA tiles.
  {
    static const int pair_env = getenv("SURGVID_GEMM_PAIR") ? atoi(getenv("SURGVID_GEMM_PAIR")) : -1;
    const int want = pair_request >= 0 ? pair_request : pair_env;
    const long long pair_tiles = static_cast<long long>(ceil_div(M, 2 * kBlockM)) * ceil_div(N, p.block_n);
    const bool pays = K >= 512 || (!out_fp32 && N >= 320);
    p.pair = want >= 0 ? (want > 0 ? 1 : 0) : ((pays && pair_tiles >= sms / 2) ? 1 : 0);
  }
  if (p.pair && (p.block_n % 32 != 0)) p.block_n = round_up(p.block_n, 32);  // each CTA stages block_n/2 rows of B (multiple of 16)
  if (p.block_n > 256) { p.block_n = 256; }
  const int b_rows = p.pair ? p.block_n / 2 : p.block_n;
  const int stage_bytes_eff = kATileBytes + b_rows * kBlockK * 2;
  // shared-memory split: [1 KB alignment slack | operand ring | epilogue staging | bias slices] = kSmemTotal.  The TMA epilogues keep
  // epi_bufs 2 KB buffers per warp in flight (stores, and residual loads for the read-modify-write form); measured (round 2) they,
  // not the operand ring, bound the K <= 1360 GEMMs, so they get 4 buffers and the ring what is left (>= 3 stages at every block_n)
  {
    static const int bufs_env = getenv("SURGVID_GEMM_EPI_BUFS") ? atoi(getenv("SURGVID_GEMM_EPI_BUFS")) : kMaxEpiBufs;
    static const int lag_env = getenv("SURGVID_GEMM_EPI_LAG") ? atoi(getenv("SURGVID_GEMM_EPI_LAG")) : 1;
    p.epi_bufs = std::min(kMaxEpiBufs, std::max(2, bufs_env));
    p.epi_lag = std::min(p.epi_bufs - 1, std::max(1, lag_env));
    p.staging_bytes = p.tma_out ? kEpiWarps * p.epi_bufs * kEpiBufBytes : kStagingBytes;
  }
  const int ring_budget = kSmemTotal - 1024 - kBiasBytes - p.staging_bytes;
  p.num_stages = std::min(kMaxStages, ring_budget / stage_bytes_eff);
  SV_CHECK(p.num_stages >= 2, "GEMM shared-memory plan");
  p.num_n_tiles = ceil_div(N, p.block_n);
  p.num_tiles = ceil_div(M, p.pair ? 2 * kBlockM : kBlockM) * p.num_n_tiles;
  {
    static const int pf_env = getenv("SURGVID_GEMM_PREFETCH") ? atoi(getenv("SURGVID_GEMM_PREFETCH")) : 0;  // measured: no gain (0 = off)
    p.prefetch = pf_env;
  }
  p.out_fp32 = out_fp32;
  p.kb_split = ceil_div(K - K2, kBlockK);
  plan->grid = p.pair ? 2 * std::min(p.num_tiles, sms / 2) : std::min(p.num_tiles, sms);
  plan->smem_bytes = static_cast<size_t>(p.num_stages) * stage_bytes_eff + p.staging_bytes + kBiasBytes + 1024;
  plan->flops = 2.0 * M * static_cast<double>(N) * K;
  return SV_OK;
}

int gemm_plan(const GemmDesc& d, GemmPlan* plan) {
  SV_CHECK(d.M > 0 && d.N > 0 && d.K > 0, "GEMM dims must be positive");
  SV_CHECK(d.K % 8 == 0 && d.N % 8 == 0, "GEMM needs K%8==0 and N%8==0");
  SV_CHECK(d.K2 >= 0 && d.K2 < d.K && (d.K2 == 0 || (d.A2 != nullptr && (d.K - d.K2) % kBlockK == 0 && d.K2 % 8 == 0 && d.lda2 >= d.K2)),
           "GEMM second A segment: K-K2 must be a multiple of 64, K2 % 8 == 0");
  const bool conv = d.conv.k > 0;
  if (conv) {
    SV_TRY(check_conv(d.conv));
    SV_CHECK(d.K2 == 0 && d.M == d.conv.B * d.conv.Ho() * d.conv.Wo() && d.K == d.conv.k * d.conv.k * d.conv.C,
             "conv GEMM: M must be B*Ho*Wo and K k*k*C, no second A segment");
  }
  SV_CHECK((conv || d.lda >= d.K - d.K2) && d.ldw >= d.K && d.ldc >= d.N, "GEMM leading dimensions too small");
  SV_CHECK(d.A && d.W && d.out, "GEMM null operand");
  SV_CHECK((reinterpret_cast<uintptr_t>(d.out) & 15) == 0 && d.ldc % (d.out_fp32 ? 4 : 8) == 0, "GEMM output must be 16B-aligned rows");
  if (d.residual) SV_CHECK((reinterpret_cast<uintptr_t>(d.residual) & 15) == 0 && d.ldr % 4 == 0 && d.ldr >= d.N, "GEMM residual alignment");
  if (d.bias) SV_CHECK((reinterpret_cast<uintptr_t>(d.bias) & 15) == 0, "GEMM bias alignment");
  const int sms = device_sm_count();
  SV_CHECK(sms > 0, "no CUDA device");
  SV_TRY(gemm_plan_shape(d.M, d.N, d.K, d.K2, d.out_fp32, d.residual != nullptr, d.pair, sms, plan));
  GemmParams& p = plan->p;
  const int b_rows = p.pair ? p.block_n / 2 : p.block_n;
  p.act = d.act;
  p.bias = d.bias; p.residual = d.residual; p.ldr = d.ldr; p.out = d.out; p.ldc = d.ldc;
  p.conv = conv ? 1 : 0;
  p.conv_k = d.conv.k; p.conv_c = d.conv.C; p.conv_stride = d.conv.stride; p.conv_pad = d.conv.pad;
  p.conv_ho = conv ? d.conv.Ho() : 0; p.conv_wo = conv ? d.conv.Wo() : 0;
  if (conv) {
    p.prefetch = 0;
    SV_TRY(encode_im2col_map(&plan->tmap_a, d.A, d.conv));
  } else {
    SV_TRY(encode_operand_map(&plan->tmap_a, d.A, d.M, d.K - d.K2, d.lda, kBlockM));
  }
  if (d.K2 > 0) SV_TRY(encode_operand_map(&plan->tmap_a2, d.A2, d.M, d.K2, d.lda2, kBlockM));
  else plan->tmap_a2 = plan->tmap_a;
  SV_TRY(encode_operand_map(&plan->tmap_w, d.W, d.N, d.K, d.ldw, b_rows));
  plan->tmap_out = plan->tmap_a;
  plan->tmap_res = plan->tmap_a;
  if (p.tma_out) {
    // bf16: box = 32 columns x 32 rows; fp32: box = 16 columns x 32 rows; 64 bytes per box row, 64-byte swizzle
    EncodeTiledFn fn = get_encode_fn();
    if (fn == nullptr) return fail(SV_ERR_CUDA, "cuTensorMapEncodeTiled driver entry point unavailable (no CUDA driver?)");
    auto enc = [&](CUtensorMap* m, const void* base, int64_t ld) -> int {
      const int es = d.out_fp32 ? 4 : 2;
      cuuint64_t gdim[2] = {static_cast<cuuint64_t>(d.N), static_cast<cuuint64_t>(d.M)};
      cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * es};
      cuuint32_t box[2] = {static_cast<cuuint32_t>(64 / es), 32};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = fn(m, d.out_fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(SV_ERR_CUDA, "cuTensorMapEncodeTiled(gemm out) failed, CUresult " + std::to_string(static_cast<int>(r)));
      return SV_OK;
    };
    SV_TRY(enc(&plan->tmap_out, d.out, d.ldc));
    if (d.residual) SV_TRY(enc(&plan->tmap_res, d.residual, d.ldr));
  }
  return SV_OK;
}

namespace {

typedef void (*GemmKernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const GemmParams);

template <int ACT, bool PAIR, bool CONV>
GemmKernelFn pick_kernel(int out_fp32, bool resid) {
  if (out_fp32) return resid ? gemm_bf16_tcgen05_kernel<ACT, true, true, PAIR, CONV> : gemm_bf16_tcgen05_kernel<ACT, true, false, PAIR, CONV>;
  return resid ? gemm_bf16_tcgen05_kernel<ACT, false, true, PAIR, CONV> : gemm_bf16_tcgen05_kernel<ACT, false, false, PAIR, CONV>;
}

template <bool CONV>
GemmKernelFn kernel_for_a(const GemmParams& p) {
  const bool resid = p.residual != nullptr;
  if (p.pair) {
    switch (p.act) {
      case ACT_GELU: return pick_kernel<ACT_GELU, true, CONV>(p.out_fp32, resid);
      case ACT_RELU: return pick_kernel<ACT_RELU, true, CONV>(p.out_fp32, resid);
      default: return pick_kernel<ACT_NONE, true, CONV>(p.out_fp32, resid);
    }
  }
  switch (p.act) {
    case ACT_GELU: return pick_kernel<ACT_GELU, false, CONV>(p.out_fp32, resid);
    case ACT_RELU: return pick_kernel<ACT_RELU, false, CONV>(p.out_fp32, resid);
    default: return pick_kernel<ACT_NONE, false, CONV>(p.out_fp32, resid);
  }
}

GemmKernelFn kernel_for(const GemmParams& p) { return p.conv ? kernel_for_a<true>(p) : kernel_for_a<false>(p); }

}  // namespace

int gemm_launch(const GemmPlan& plan, cudaStream_t stream) {
  GemmKernelFn fn = kernel_for(plan.p);
  SV_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(fn), kSmemTotal));
  if (plan.p.pair) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(plan.grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = plan.smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, fn, plan.tmap_a, plan.tmap_a2, plan.tmap_w, plan.tmap_out, plan.tmap_res, plan.p);
    if (e != cudaSuccess) return fail(SV_ERR_CUDA, std::string("cudaLaunchKernelEx(gemm pair): ") + cudaGetErrorString(e));
    return SV_OK;
  }
  fn<<<plan.grid, kThreads, plan.smem_bytes, stream>>>(plan.tmap_a, plan.tmap_a2, plan.tmap_w, plan.tmap_out, plan.tmap_res, plan.p);
  return launch_status("gemm_bf16_tcgen05_kernel");
}

}  // namespace sv

#ifdef SV_GEMM_TRACE
extern "C" int sv_debug_gemm_trace(void* host_out) { return cudaMemcpyFromSymbol(host_out, sv::g_trace, sizeof(sv::g_trace)) == cudaSuccess ? 0 : 1; }
#endif

extern "C" int sv_op_gemm_bf16(const uint16_t* A, int64_t lda, const uint16_t* W, int64_t ldw, int32_t M, int32_t N, int32_t K,
                               const float* bias, int32_t act, const float* residual, int64_t ldr, void* out, int64_t ldc,
                               int32_t out_fp32, void* stream) {
  sv::GemmDesc d;
  d.A = reinterpret_cast<const sv::bf16*>(A); d.lda = lda;
  d.W = reinterpret_cast<const sv::bf16*>(W); d.ldw = ldw;
  d.M = M; d.N = N; d.K = K; d.bias = bias; d.act = act; d.residual = residual; d.ldr = ldr;
  d.out = out; d.ldc = ldc; d.out_fp32 = out_fp32;
  if (const char* e = getenv("SURGVID_GEMM_PAIR")) d.pair = atoi(e);  // test hook: force CTA-pair mode on (1) / off (0)
  sv::GemmPlan plan;
  SV_TRY(sv::gemm_plan(d, &plan));
  return sv::gemm_launch(plan, static_cast<cudaStream_t>(stream));
}

extern "C" int sv_op_gemm_plan_info(int32_t M, int32_t N, int32_t K, int32_t K2, int32_t out_fp32, int32_t has_residual, int32_t pair_request,
                                    int32_t num_sms, int32_t* info) {
  SV_CHECK(info != nullptr, "GEMM plan info: null output");
  SV_CHECK(M > 0 && N > 0 && K > 0 && num_sms > 0, "GEMM plan info: dims and SM count must be positive");
  SV_CHECK(K % 8 == 0 && N % 8 == 0, "GEMM needs K%8==0 and N%8==0");
  SV_CHECK(K2 >= 0 && K2 < K && (K2 == 0 || ((K - K2) % 64 == 0 && K2 % 8 == 0)), "GEMM second A segment: K-K2 must be a multiple of 64, K2 % 8 == 0");
  sv::GemmPlan plan;
  SV_TRY(sv::gemm_plan_shape(M, N, K, K2, out_fp32 ? 1 : 0, has_residual != 0, pair_request, num_sms, &plan));
  const sv::GemmParams& p = plan.p;
  const int epi = !p.tma_out ? SV_GEMM_EPI_TRANSPOSE : (!out_fp32 ? SV_GEMM_EPI_BF16_TMA : (has_residual ? SV_GEMM_EPI_F32_TMA_RESID : SV_GEMM_EPI_F32_TMA));
  const int32_t v[SV_GEMM_PLAN_INFO_LEN] = {p.block_n, p.pair, p.tma_out, p.num_stages, p.epi_bufs, p.epi_lag, p.prefetch, p.num_tiles, plan.grid,
                                            epi, (out_fp32 ? 1 : 0) | (has_residual ? 2 : 0) | (p.pair ? 4 : 0), p.num_n_tiles,
                                            static_cast<int32_t>(plan.smem_bytes)};
  std::copy(v, v + SV_GEMM_PLAN_INFO_LEN, info);
  return SV_OK;
}

extern "C" int sv_op_conv_gemm_bf16(const uint16_t* x, int32_t B, int32_t H, int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad,
                                    const uint16_t* Wt, int64_t ldw, int32_t N, const float* bias, int32_t act, const float* residual, int64_t ldr,
                                    void* out, int64_t ldc, int32_t out_fp32, void* stream) {
  sv::GemmDesc d;
  d.conv.B = B; d.conv.H = H; d.conv.W = W; d.conv.C = C; d.conv.k = k; d.conv.stride = stride; d.conv.pad = pad;
  SV_CHECK(x && Wt && out, "conv GEMM: null input, weight or output");
  SV_TRY(sv::check_conv(d.conv));
  SV_CHECK(N > 0 && N % 8 == 0 && ldw >= static_cast<int64_t>(k) * k * C && ldc >= N, "conv GEMM: N % 8 == 0, ldw >= k*k*C and ldc >= N");
  SV_CHECK(act == sv::ACT_NONE || act == sv::ACT_GELU || act == sv::ACT_RELU, "conv GEMM: act must be 0 (none), 1 (GELU) or 2 (ReLU)");
  d.A = reinterpret_cast<const sv::bf16*>(x);
  d.W = reinterpret_cast<const sv::bf16*>(Wt); d.ldw = ldw;
  d.M = B * d.conv.Ho() * d.conv.Wo(); d.N = N; d.K = k * k * C; d.bias = bias; d.act = act; d.residual = residual; d.ldr = ldr;
  d.out = out; d.ldc = ldc; d.out_fp32 = out_fp32;
  if (const char* e = getenv("SURGVID_GEMM_PAIR")) d.pair = atoi(e);  // test hook, as in sv_op_gemm_bf16
  sv::GemmPlan plan;
  SV_TRY(sv::gemm_plan(d, &plan));
  return sv::gemm_launch(plan, static_cast<cudaStream_t>(stream));
}

extern "C" int sv_op_conv_gemm_plan_info(int32_t B, int32_t H, int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad, int32_t N, int32_t out_fp32,
                                         int32_t has_residual, int32_t pair_request, int32_t num_sms, int32_t* conv_info, int32_t* gemm_info) {
  SV_CHECK(conv_info != nullptr, "conv GEMM plan info: null output");
  sv::ConvGeom g;
  g.B = B; g.H = H; g.W = W; g.C = C; g.k = k; g.stride = stride; g.pad = pad;
  SV_TRY(sv::check_conv_args(g));
  const int32_t K = k * k * C, M = B * g.Ho() * g.Wo();
  const int32_t v[SV_CONV_PLAN_INFO_LEN] = {sv::conv_gemm_im2col_ok(g) ? SV_GEMM_A_IM2COL : SV_GEMM_A_TILED, g.Ho(), g.Wo(), M, K};
  std::copy(v, v + SV_CONV_PLAN_INFO_LEN, conv_info);
  if (gemm_info == nullptr) return SV_OK;
  return sv_op_gemm_plan_info(M, N, (K + 7) / 8 * 8, 0, out_fp32, has_residual, pair_request, num_sms, gemm_info);
}

extern "C" int sv_op_gemm_bf16_cat(const uint16_t* A, int64_t lda, const uint16_t* A2, int64_t lda2, int32_t K2, const uint16_t* W, int64_t ldw,
                                   int32_t M, int32_t N, int32_t K, const float* bias, int32_t act, const float* residual, int64_t ldr, void* out,
                                   int64_t ldc, int32_t out_fp32, void* stream) {
  sv::GemmDesc d;
  d.A = reinterpret_cast<const sv::bf16*>(A); d.lda = lda;
  d.A2 = reinterpret_cast<const sv::bf16*>(A2); d.lda2 = lda2; d.K2 = K2;
  d.W = reinterpret_cast<const sv::bf16*>(W); d.ldw = ldw;
  d.M = M; d.N = N; d.K = K; d.bias = bias; d.act = act; d.residual = residual; d.ldr = ldr;
  d.out = out; d.ldc = ldc; d.out_fp32 = out_fp32;
  if (const char* e = getenv("SURGVID_GEMM_PAIR")) d.pair = atoi(e);  // test hook, as in sv_op_gemm_bf16
  sv::GemmPlan plan;
  SV_TRY(sv::gemm_plan(d, &plan));
  return sv::gemm_launch(plan, static_cast<cudaStream_t>(stream));
}
