// Host-side interface of the tcgen05 GEMM (gemm_tcgen05.cu).
#pragma once
#include "common.cuh"

namespace sv {

// out[M,N] = act(A[M,K] * W[N,K]^T + bias[N]) (+ residual[M,N])
struct GemmDesc {
  const bf16* A = nullptr;   // [M, K] row-major, row stride lda (elements)
  int64_t lda = 0;
  const bf16* W = nullptr;   // [N, K] row-major (nn.Linear weight layout), row stride ldw
  int64_t ldw = 0;
  int M = 0, N = 0, K = 0;
  // optional second A segment: the last K2 columns of the K dimension are read from A2[:, 0:K2] (row stride lda2) instead of
  // A[:, K-K2:K]; K - K2 must be a multiple of 64.  Lets a GEMM consume [A | A2] without materialising the concatenation.
  const bf16* A2 = nullptr;
  int64_t lda2 = 0;
  int K2 = 0;
  const float* bias = nullptr;      // [N] or null
  int act = ACT_NONE;
  const float* residual = nullptr;  // [M, N] fp32, row stride ldr, or null (may alias out if out_fp32)
  int64_t ldr = 0;
  void* out = nullptr;              // bf16 or fp32, row stride ldc
  int64_t ldc = 0;
  int out_fp32 = 0;
  int pair = -1;  // CTA-pair mode (tcgen05 cta_group::2, 256-row tiles, B split across the pair): -1 auto, 0 off, 1 on
};

struct GemmParams {
  int M, N, K;
  int block_n;      // UMMA N (multiple of 16, <= 256)
  int num_stages;   // smem ring depth
  int num_n_tiles;
  int num_tiles;
  int pair;         // 1: 2-CTA clusters; num_tiles counts 256-row pair tiles
  int prefetch;     // k-blocks of the A operand requested into L2 ahead of the shared-memory ring (0 = off)
  int kb_split;     // k-blocks served by the first A segment (all of them without a second segment)
  int epi_bufs;     // TMA epilogues: 2 KB staging buffers per epilogue warp (2..4) = result stores / residual loads in flight per warp
  int epi_lag;      // fp32 + residual: result stores allowed to be pending when a buffer is handed back to the residual loads (1..epi_bufs-1)
  int staging_bytes;  // shared memory between the operand ring and the bias slices
  int tma_out;      // 1: bf16 result without residual is written with 2-D TMA stores from a swizzled staging tile
  int act;
  int out_fp32;
  const float* bias;
  const float* residual;
  long long ldr;
  void* out;
  long long ldc;
};

struct GemmPlan {
  CUtensorMap tmap_a;
  CUtensorMap tmap_a2;   // second A segment (copy of tmap_a when unused)
  CUtensorMap tmap_w;
  CUtensorMap tmap_out;  // TMA epilogue: 2-D store map of the result (copy of tmap_a when unused)
  CUtensorMap tmap_res;  // TMA epilogue: 2-D load map of the fp32 residual (copy of tmap_a when unused)
  GemmParams p;
  int grid = 0;
  size_t smem_bytes = 0;
  double flops = 0.0;
};

int gemm_plan(const GemmDesc& d, GemmPlan* plan);
// the shape-only part of gemm_plan (no device, no driver): fills plan->p except the pointers and act, plan->grid, plan->smem_bytes
int gemm_plan_shape(int M, int N, int K, int K2, int out_fp32, bool has_residual, int pair_request, int sms, GemmPlan* plan);
int gemm_launch(const GemmPlan& plan, cudaStream_t stream);
// pick the UMMA N for a problem (exposed for tests)
int gemm_pick_block_n(int M, int N, int K, int num_sms, int step = 16);

}  // namespace sv
