// Launchers of the HBM-bound (non-GEMM) kernels; defined in elementwise.cu / attention.cu.
#pragma once
#include "common.cuh"

namespace sv {

int launch_layernorm(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int C, float* out_f32,
                     bf16* out_bf16, cudaStream_t st);
int launch_layernorm_patch(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int C, float* out_f32,
                           bf16* out_bf16, bf16* out_patch, int pH, int pW, int psr, cudaStream_t st);
int launch_im2col(const float* src_nchw_f32, const bf16* src_nhwc_bf16, int B, int Cin, int H, int W, int k, int stride, int pad,
                  bf16* out, int64_t ldo, cudaStream_t st);
int launch_dwconv3x3_gelu(const bf16* x, const float* w9c, const float* bias, int B, int H, int W, int C, bf16* out, int64_t ldo,
                          cudaStream_t st);
int launch_gauss5x5(const float* x, float* out, int planes, int H, int W, cudaStream_t st);
int launch_bilinear_tokens(const bf16* x, int B, int H, int W, int C, int Ho, int Wo, bf16* out, int64_t ldo, cudaStream_t st);
int launch_token_mean(const float* x, int B, int tokens, int C, float* out, cudaStream_t st);
int launch_bf16_to_f32(const bf16* x, float* out, int64_t n, cudaStream_t st);
int launch_attention(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, const bf16* v, int64_t ldv, bf16* o, int64_t ldo, int B,
                     int heads, int Nq, int Nkv, int hd, float scale, cudaStream_t st);
// P = softmax(Q K^T * scale) -> fp32 [B, heads, Nq, Nkv] (attention_probs.cu); hd 32 or 64
int launch_attention_probs(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, int B, int heads, int Nq, int Nkv, int hd, float scale,
                           float* p, cudaStream_t st);

// tcgen05/TMEM attention for head_dim 64, N_kv <= 448 (attention_tc.cu); the plan owns the four 3-D tensor maps
struct AttnTcPlan {
  CUtensorMap tmap_q, tmap_k, tmap_v, tmap_o;
  int B = 0, heads = 0, Nq = 0, Nkv = 0, kt = 0, qtiles = 0, tpc = 1, tmem_cols = 0;
  float scale_log2 = 0.f;
  size_t smem_bytes = 0;
};
bool attention_tc_enabled();   // SURGVID_ATTN_TC=0 selects the mma.sync kernels everywhere (A/B switch)
bool attention_tc_supported(int hd, int Nkv, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, const void* q, const void* k, const void* v, const void* o);
int attention_tc_plan(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, const bf16* v, int64_t ldv, bf16* o, int64_t ldo, int B, int heads,
                      int Nq, int Nkv, float scale, AttnTcPlan* plan);
int attention_tc_launch(const AttnTcPlan& plan, cudaStream_t st);

// TMA-staged persistent depthwise conv (dwconv_tma.cu); the plan owns the tensor map of the input
struct DwconvPlan {
  CUtensorMap tmap;
  const float* w9c = nullptr;
  const float* bias = nullptr;
  bf16* out = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  int64_t ldo = 0;  // output row (pixel) stride in elements, >= C
  int tw = 8;       // output columns per tile (box width - 2)
  int cpl = 4;      // channels per lane: 4 (128-channel tiles) or 2 (64-channel tiles)
};
bool dwconv_tma_supported(int C);
int dwconv_tma_plan(const bf16* x, const float* w9c, const float* bias, int B, int H, int W, int C, bf16* out, int64_t ldo, DwconvPlan* plan);
int dwconv_tma_launch(const DwconvPlan& plan, cudaStream_t st);

// fused first-layer conv (k7 s4 p3 on fp32 NCHW, <= 3 channels) + LayerNorm (mode 0) or ReLU (mode 1)  (stem.cu)
bool stem_conv_supported(int Cin, int Cout, int ldw);
int launch_stem_conv(const float* src, const bf16* w, int ldw, const float* bias, const float* gamma, const float* beta, float eps, int mode,
                     int B, int Cin, int H, int W, int Cout, float* out_f32, bf16* out_bf16, cudaStream_t st);

// DWConv3x3 + GELU fused into the fc2 GEMM as the producer of its A tiles (mixffn.cu):
//   x[M, N] += bias + GELU(dwconv3x3(h1) + b_dw) @ Wcat[:, :hidden]^T (+ tail[M, tail_cols] @ Wcat[:, hidden:]^T)
// h1: [frames, H, W, hidden] bf16; w10c: fp32 [10, hidden] = 9 taps (kh*3+kw) then the depthwise bias; x fp32 in place.
struct MixffnPlan {
  CUtensorMap tmap_h1, tmap_dw, tmap_w, tmap_t;
  alignas(8) unsigned char params[128];
  int grid = 0;
  size_t smem_bytes = 0;
  double flops = 0.0;
};
bool mixffn_fc2_supported(int H, int W, int hidden, int N, int tail_cols);
int mixffn_fc2_plan(const bf16* h1, const float* w10c, const bf16* Wcat, int64_t ldw, const float* bias, const bf16* tail, int64_t ldt,
                    int tail_cols, float* x, int64_t ldx, int frames, int H, int W, int hidden, int N, MixffnPlan* plan);
int mixffn_fc2_launch(const MixffnPlan& plan, cudaStream_t st);

inline int conv_out_dim(int in, int k, int stride, int pad) { return (in + 2 * pad - k) / stride + 1; }

}  // namespace sv
