/*
 * surgvid.h — C ABI of libsurgvid.so: the B200-native (sm_100a) LFB-extraction hot path of
 * THao712/Deep-Learning-for-Surgical-Video-Analysis.
 *
 * The reference is pure Python/PyTorch and has no FFI of its own; the "interface each entry point
 * replaces" is therefore the nn.Module call the reference drivers make (file:line under
 * /root/reference).  The Python drop-in modules (same ctor / state_dict keys) bind these symbols with
 * ctypes and expose them as PyTorch custom ops (`surgvid::evp_lfb_forward`, `surgvid::mstcn_forward`);
 * see INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every function returns an int status (SV_OK == 0); the message of the last failure on the calling
 *     thread is available from sv_last_error(); nothing throws across the ABI;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all launches are
 *     asynchronous on it;
 *   - the CALLER owns every buffer including the workspace (allocate it with the framework's caching
 *     allocator and pass it in); a handle owns only its packed weights;
 *   - a handle is bound to the CUDA device current at creation, is not thread-safe, and has no global
 *     state; use one handle per (device, stream);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with SV_ERR_CUDA.
 */
#ifndef SURGVID_H_
#define SURGVID_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SV_OK 0
#define SV_ERR_INVALID 1     /* bad argument / shape */
#define SV_ERR_CUDA 2        /* CUDA runtime / driver failure (message has the CUDA error string) */
#define SV_ERR_STATE 3       /* call order violated (e.g. forward before pack_weights) */
#define SV_ERR_UNSUPPORTED 4 /* configuration outside what the kernels implement */

#define SV_ABI_VERSION 2
#define SV_PROFILE_CLASSES 9

const char* sv_last_error(void);
int sv_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * MiT-EVP encoder + SegFormer embedding head
 * replaces: mit_bX_evp(...) construction (mix_transformer_evp.py:894-943, 219-298) and
 *           MixVisionTransformerEVP.forward(x, y, flow, return_features) (mix_transformer_evp.py:418-449)
 *           as called by the LFB driver (generate_evp_LFB.py:412-414, 454).
 * ---------------------------------------------------------------------------------------------- */
typedef struct sv_evp_cfg {
  int32_t embed_dims[4]; /* mit_b3_evp: 64,128,320,512  (mix_transformer_evp.py:924) */
  int32_t num_heads[4];  /* 1,2,5,8 */
  int32_t depths[4];     /* 3,4,18,3 */
  int32_t sr_ratios[4];  /* 8,4,2,1 */
  int32_t mlp_ratio;     /* 4 */
  int32_t embedding_dim; /* SegFormerHead.embedding_dim = 2048 (segformer_head.py:53) */
  int32_t fold_head;     /* 0: linear_c{i} then linear_fuse as two GEMM levels (default, parity reference);
                            1: pre-multiplied W_fuse*W_c weights, one GEMM (exact in real arithmetic,
                               SURVEY.md §7 "head algebra"); both pool to c4's grid before the projection. */
} sv_evp_cfg;

typedef struct sv_evp sv_evp_handle;

int sv_evp_create(const sv_evp_cfg* cfg, sv_evp_handle** out);
int sv_evp_destroy(sv_evp_handle* h);

/* Hand one state_dict entry (fp32, HOST memory, contiguous) to the handle.  `name` is the reference's
 * state_dict key (SURVEY.md §8b), e.g. "block3.7.attn.kv.weight".  replaces: load_state_dict
 * (generate_evp_LFB.py:414).  host_data == NULL stores zeros; ndim <= 4.  Tensors are stored by name and checked at
 * sv_evp_pack_weights; shape == NULL with ndim > 0, or a negative dimension -> SV_ERR_INVALID. */
int sv_evp_set_tensor(sv_evp_handle* h, const char* name, const float* host_data, const int64_t* shape, int32_t ndim);

/* Fold BatchNorm (eval) into the preceding conv, reorder conv weights to (kh,kw,cin)-major implicit-GEMM
 * form, convert to bf16 and upload.  Fails with SV_ERR_STATE naming the first missing or wrongly shaped key. */
int sv_evp_pack_weights(sv_evp_handle* h);

/* Bytes of scratch the forward needs for `micro_batch` frames of HxW (frames are processed in
 * micro-batches so that the activation working set stays L2-resident). */
size_t sv_evp_workspace_bytes(const sv_evp_handle* h, int32_t micro_batch, int32_t H, int32_t W);

/* x, seg: [B,3,H,W] fp32 NCHW device; flow: [B,2,H,W] fp32 device or NULL (flow branch skipped, as
 * `flow=None` in mix_transformer_evp.py:423); out_features: [B, embedding_dim] fp32 device.
 * replaces: model_LFB.forward(inputs, segmaps, flow, return_features=True) (generate_evp_LFB.py:454). */
int sv_evp_forward(sv_evp_handle* h, const float* x, const float* seg, const float* flow, float* out_features,
                   int32_t B, int32_t H, int32_t W, int32_t micro_batch, void* workspace, size_t workspace_bytes,
                   void* stream);

/* Attention maps of the encoder blocks: the post-softmax P = softmax(Q K^T * head_dim^-0.5) of every block's spatial-reduction
 * attention (mix_transformer_evp.py:123-125; what the reference's `get_local('attn')` records from Attention.forward), fp32.
 *   sv_evp_attention_maps_layout: host only (needs no device and no handle, only the config).  *n_blocks = sum(depths).
 *     block_offsets[n_blocks + 1]: element offsets of block k's [B, heads, N, N_kv] array in one buffer, in call order (stage 1's
 *     blocks, then stage 2's, ...), the last entry is the total; block_dims[3 * n_blocks]: (heads, N, N_kv) per block.  With both
 *     arrays NULL only *n_blocks is set; otherwise max_blocks must be >= n_blocks.  Bad config, B, H or W -> SV_ERR_INVALID.
 *   sv_evp_forward_attention: sv_evp_forward (same arguments, same features bit for bit, same workspace size) that also writes every
 *     block's maps to `maps` (device, 16-byte aligned, >= block_offsets[n_blocks] fp32 elements, else SV_ERR_INVALID).  It runs its
 *     own launch plans (one attention_probs_kernel launch after each block's attention); the plans of sv_evp_forward are unchanged.
 *     Flow cross-attention maps are not captured.  Cost: 6.76 MB per frame for mit_b3_evp at 224x224, 452 MB at 480x854. */
int sv_evp_attention_maps_layout(const sv_evp_cfg* cfg, int32_t B, int32_t H, int32_t W, int64_t* block_offsets, int32_t* block_dims,
                                 int32_t max_blocks, int32_t* n_blocks);
int sv_evp_forward_attention(sv_evp_handle* h, const float* x, const float* seg, const float* flow, float* out_features, float* maps,
                             int64_t maps_elems, int32_t B, int32_t H, int32_t W, int32_t micro_batch, void* workspace,
                             size_t workspace_bytes, void* stream);

/* Encoder feature pyramid: MixVisionTransformerEVP.forward_features(x, y) (mix_transformer_evp.py:352-416), the four stage outputs
 * norm_s(x) as fp32 NCHW maps [B, C_s, H_s, W_s] (mit_b3_evp at 224x224: [B,64,56,56] [B,128,28,28] [B,320,14,14] [B,512,7,7]).
 *   sv_evp_stage_shapes: host only (needs no device and no handle, only the config).  dims[3 * s .. 3 * s + 2] = (C_s, H_s, W_s) of
 *     stage s for an HxW input: H_1 = (H + 2*3 - 7) / 4 + 1, then H_{s+1} = (H_s + 2 - 3) / 2 + 1 (W likewise).  Bad config, H or W,
 *     or an input too small for the pyramid (a stage map smaller than its sr x sr spatial-reduction window, which the reference's
 *     Conv2d rejects; 29 x 29 is the smallest input at sr 8 / 4 / 2 / 1) -> SV_ERR_INVALID; sv_evp_forward_features applies the same
 *     checks.
 *   sv_evp_forward_features: x, seg as sv_evp_forward; stage_out[s]: device, 4-byte aligned, >= B * C_s * H_s * W_s fp32 elements
 *     (stage_elems[s] gives the size).  maps: NULL, or the attention maps of every encoder block in the layout of
 *     sv_evp_attention_maps_layout (as sv_evp_forward_attention).  It runs encoder-only launch plans of its own: the encoder of
 *     sv_evp_forward without the flow branch and the SegFormer head, whose stage norms write the NCHW maps; the plans of sv_evp_forward
 *     and sv_evp_forward_attention are unchanged.  Workspace: sv_evp_workspace_bytes.  Every argument is checked before the device is
 *     touched (SV_ERR_INVALID with the message in sv_last_error()).  Afterwards the "stage{1..4}_tokens" taps hold the last
 *     micro-batch's stage outputs, as after sv_evp_forward. */
int sv_evp_stage_shapes(const sv_evp_cfg* cfg, int32_t H, int32_t W, int32_t dims[12]);
int sv_evp_forward_features(sv_evp_handle* h, const float* x, const float* seg, float* const stage_out[4], const int64_t stage_elems[4],
                            float* maps, int64_t maps_elems, int32_t B, int32_t H, int32_t W, int32_t micro_batch, void* workspace,
                            size_t workspace_bytes, void* stream);

/* head.fc / head.fc_ant on extracted features (segformer_head.py:101-106,176-179):
 * feats [B,2048] fp32 device -> y [B,7], y_ant [B,7] fp32 device. */
int sv_evp_classify(sv_evp_handle* h, const float* feats, float* y, float* y_ant, int32_t B, void* stream);

/* Debug/parity taps of the LAST micro-batch processed: "stage{1..4}_tokens" ([n,N_s,C_s], after norm_s),
 * "fused{3,4}_tokens" (after cross attention).  Converts to fp32 into dst (device); *n_elems receives the count. */
int sv_evp_read_tap(sv_evp_handle* h, const char* name, float* dst, int64_t max_elems, int64_t* n_elems, void* stream);

/* number of kernels the last sv_evp_forward call launched (for bench.py's gpu_launches) */
int64_t sv_evp_last_launch_count(const sv_evp_handle* h);

/* Per-kernel-class device timing for roofline reports: when enabled, every launch of sv_evp_forward is bracketed by
 * CUDA events on `stream` and the forward synchronises at the end of each micro-batch (never enable in a timed run).
 * Classes (index): 0 tcgen05 GEMM, 1 LayerNorm, 2 im2col, 3 DWConv+GELU, 4 attention, 5 Gaussian, 6 bilinear, 7 token mean,
 * 8 fused first-layer conv (stem).  Arrays passed to sv_evp_get_profile must hold SV_PROFILE_CLASSES entries.
 * sv_evp_set_profile resets the accumulators; sv_evp_get_profile fills ms_by_kind[], launches_by_kind[], the algorithmic
 * GEMM FLOPs (2*M*N*K summed over the GEMM launches) and, if bytes_by_kind != NULL, the algorithmic HBM bytes per class
 * (operands + results of every launch counted once) since the last reset. */
int sv_evp_set_profile(sv_evp_handle* h, int32_t enable);
int sv_evp_get_profile(const sv_evp_handle* h, double* ms_by_kind, int64_t* launches_by_kind, double* gemm_flops,
                       double* bytes_by_kind);
/* CSV with one line per launch of the schedule (shape, tile configuration, accumulated device ms) since the last reset. */
int sv_evp_dump_profile(const sv_evp_handle* h, const char* path);

/* ------------------------------------------------------------------------------------------------
 * MS-TCN MultiStageModel_S
 * replaces: mstcn.MultiStageModel_S(stages, layers, f_maps, f_dim, out_features, causal_conv)
 *           (mstcn.py:94-130) as called at trans_SV_output.py:197, 279 and tecno_trans.py:267.
 * ---------------------------------------------------------------------------------------------- */
typedef struct sv_mstcn_cfg {
  int32_t stages;       /* 2 */
  int32_t layers;       /* 8 (dilation 2^i) */
  int32_t f_maps;       /* 32 (64 in tecno.py) */
  int32_t f_dim;        /* 2048 */
  int32_t out_features; /* 14 = 7 phase logits + 7 anticipation regressors */
  int32_t causal;       /* must be 1 (mstcn_causal_conv=True, trans_SV_output.py:197) */
} sv_mstcn_cfg;

typedef struct sv_mstcn sv_mstcn_handle;

int sv_mstcn_create(const sv_mstcn_cfg* cfg, sv_mstcn_handle** out);
int sv_mstcn_destroy(sv_mstcn_handle* h);
/* Tensors are stored by name and checked at sv_mstcn_pack_weights (missing key -> SV_ERR_STATE, wrong shape -> SV_ERR_INVALID);
 * shape == NULL with ndim > 0, or a negative dimension -> SV_ERR_INVALID. */
int sv_mstcn_set_tensor(sv_mstcn_handle* h, const char* name, const float* host_data, const int64_t* shape, int32_t ndim);
int sv_mstcn_pack_weights(sv_mstcn_handle* h);
size_t sv_mstcn_workspace_bytes(const sv_mstcn_handle* h, int64_t total_frames);

/* feats: [T_total, f_dim] fp32 device, TIME-MAJOR (the memory layout of `long_feature`,
 * trans_SV_output.py:271-272), videos concatenated; video_offsets: HOST int64 [n_videos+1] row offsets
 * (videos are independent: causal history never crosses an offset); logits: [stages, out_features, T_total]
 * fp32 device — for one video this is exactly the reference's [stages,1,out_features,T] (mstcn.py:124-130). */
int sv_mstcn_forward(sv_mstcn_handle* h, const float* feats, const int64_t* video_offsets, int32_t n_videos,
                     float* logits, void* workspace, size_t workspace_bytes, void* stream);
int64_t sv_mstcn_last_launch_count(const sv_mstcn_handle* h);

/* Inputs of the Trans-SVNet head (SURVEY.md 8f-1; `Transformer.original_forward`, adapter_transformer.py:329-349), i.e. everything
 * of that function that the reference itself defines (its inner `Transformer2_3_1` module is not part of the reference):
 *   sv_mstcn_forward_query = sv_mstcn_forward plus, from the SAME pass over the features, the decoder query
 *       query[T_total, q] = tanh(feats . fc.weight^T)            (adapter_transformer.py:325,348; q = rows of `fc.weight`)
 *     `fc.weight` ([q <= 16, f_dim], no bias) is handed over with sv_mstcn_set_tensor(h, "fc.weight", ...) before pack_weights;
 *     query may be NULL (then this is sv_mstcn_forward).
 *   sv_op_causal_windows: x is [C, T_total] with row stride ldx (e.g. the last stage of `logits`); per video v,
 *       out[t, j, c] = x[c, t - (len_q - 1) + j], zero where that index precedes the video's first frame
 *     -> out [T_total, len_q, C] (the `inputs` tensor built by the loop at adapter_transformer.py:335-344). */
int sv_mstcn_forward_query(sv_mstcn_handle* h, const float* feats, const int64_t* video_offsets, int32_t n_videos, float* logits,
                           float* query, void* workspace, size_t workspace_bytes, void* stream);
int sv_op_causal_windows(const float* x, int64_t ldx, int32_t C, const int64_t* video_offsets, int32_t n_videos, int32_t len_q,
                         float* out, void* stream);

/* Online use: n_streams independent videos fed a few frames at a time, with what the causal layers need of each video's past kept in a
 * caller-owned device STATE.  Streamed logits (and query) are bit-identical to sv_mstcn_forward_query over the same video's frames.
 *   State layout (size it with sv_mstcn_stream_state_bytes, zero it with sv_mstcn_stream_reset, 256-byte aligned; nothing else writes it):
 *     int64 seen[n_streams] (frames each stream has consumed), padded to 256 bytes; then per stream, per stage, per layer l a ring of
 *     2 * 2^l rows x f_maps fp32 holding that layer's last inputs (position q in slot q mod 2 * 2^l); the ring of layer l starts
 *     2 * (2^l - 1) rows into the stage's 2 * (2^layers - 1) rows (510 rows, 65 280 B per stage at layers 8, f_maps 32).
 *   sv_mstcn_stream_reset: stream_ids NULL resets every stream (required once for a new state: the handle keeps a host copy of the
 *     counters of the states it has reset, which is how a step is checked before launch); otherwise the n_ids listed streams, whose
 *     next frame then behaves as frame 0 of a new video.
 *   sv_mstcn_stream_step: feats [sum(counts), f_dim] fp32 device (16-byte aligned), the rows of stream stream_ids[k] (counts[k] >= 1,
 *     no id twice) grouped in that order; logits [stages, out_features, sum(counts)], query [sum(counts), q] or NULL, as
 *     sv_mstcn_forward_query.  Then each listed stream's seen advances by its count.  Launches 21 kernels at stages 2, layers 8.
 *     Workspace: sv_mstcn_stream_workspace_bytes(h, sum(counts)), 256-byte aligned (it keeps every layer's inputs of the step). */
size_t sv_mstcn_stream_state_bytes(const sv_mstcn_handle* h, int32_t n_streams);
size_t sv_mstcn_stream_workspace_bytes(const sv_mstcn_handle* h, int64_t rows);
int sv_mstcn_stream_reset(sv_mstcn_handle* h, void* state, size_t state_bytes, int32_t n_streams, const int32_t* stream_ids,
                          int32_t n_ids, void* stream);
int sv_mstcn_stream_step(sv_mstcn_handle* h, void* state, size_t state_bytes, int32_t n_streams, const float* feats,
                         const int32_t* stream_ids, const int64_t* counts, int32_t n_ids, float* logits, float* query, void* workspace,
                         size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Single kernels (unit-test surface; the two forwards above are built from exactly these).
 * bf16 tensors are passed as uint16_t*. All pointers are device pointers.
 * ---------------------------------------------------------------------------------------------- */

/* out[M,N] = act(A[M,K] * W[N,K]^T + bias) (+ residual).  tcgen05/TMEM/TMA GEMM, bf16 in, fp32 accumulate.
 * replaces nn.Linear / 1x1 & patchified nn.Conv2d (mix_transformer_evp.py:81-84,37-40,188; segformer_head.py:39).
 * lda/ldw/ldc/ldr in elements; K,lda,ldw %8==0; N%8==0; act: 0 none, 1 GELU(erf), 2 ReLU;
 * out_fp32: 1 -> out is float*, 0 -> out is bf16; residual (fp32, may alias out when out_fp32) or NULL. */
int sv_op_gemm_bf16(const uint16_t* A, int64_t lda, const uint16_t* W, int64_t ldw, int32_t M, int32_t N, int32_t K,
                    const float* bias, int32_t act, const float* residual, int64_t ldr, void* out, int64_t ldc,
                    int32_t out_fp32, void* stream);

/* The launch plan sv_op_gemm_bf16 / sv_op_gemm_bf16_cat choose for a problem on a device with num_sms SMs (the same function decides
 * both).  Host only: touches neither device nor driver.  It depends on M, N, K, K2 (0 without a second A segment), the output type,
 * whether there is a residual, pair_request (-1 auto, 0 off, 1 on; the ops take it from SURGVID_GEMM_PAIR when set) and the
 * switches SURGVID_GEMM_TMA_OUT / _EPI_BUFS / _EPI_LAG / _PREFETCH / _PAIR, read once per process.  info[SV_GEMM_PLAN_INFO_LEN]:
 *   0 block_n (UMMA N), 1 pair (2-CTA clusters), 2 tma_out, 3 num_stages (operand ring depth), 4 epi_bufs, 5 epi_lag, 6 prefetch,
 *   7 num_tiles, 8 grid (CTAs), 9 epilogue form (SV_GEMM_EPI_*), 10 kernel instantiation gemm_bf16_tcgen05_kernel<act, OUT_F32, RESID,
 *   PAIR> as OUT_F32 | RESID << 1 | PAIR << 2, 11 num_n_tiles, 12 dynamic shared memory bytes.
 * Shape errors (as sv_op_gemm_bf16 reports them) -> SV_ERR_INVALID. */
#define SV_GEMM_EPI_BF16_TMA 0       /* bf16 result, no residual: 2-D TMA stores of 32x32 boxes */
#define SV_GEMM_EPI_F32_TMA 1        /* fp32 result, no residual: 2-D TMA stores of 16x32 boxes */
#define SV_GEMM_EPI_F32_TMA_RESID 2  /* fp32 result + fp32 residual: TMA residual loads into a per-warp ring, TMA stores */
#define SV_GEMM_EPI_TRANSPOSE 3      /* bf16 result + residual, or SURGVID_GEMM_TMA_OUT=0: transposed through shared memory, plain stores */
#define SV_GEMM_PLAN_INFO_LEN 13
int sv_op_gemm_plan_info(int32_t M, int32_t N, int32_t K, int32_t K2, int32_t out_fp32, int32_t has_residual, int32_t pair_request,
                         int32_t num_sms, int32_t* info);

/* Convolution as an implicit GEMM: out[M,N] = act(im2col(x) * W[N,K]^T + bias) (+ residual) with no im2col buffer.  x is the NHWC bf16
 * input [B, H, W, C] (16-byte aligned, rows of C contiguous), k x k taps, stride, symmetric zero padding pad; M = B * Ho * Wo with
 * Ho = (H + 2 pad - k) / stride + 1 (Wo likewise), output row m = (b, oh, ow); K = k * k * C in (kh, kw, cin) order, the layout
 * sv_op_im2col gathers and packed conv weights use.  The GEMM reads its A tiles through an im2col-mode TMA map (one tap and 64 channels
 * per k-block); the result is bit-identical to sv_op_im2col + sv_op_gemm_bf16.  Epilogue options (bias, act, residual, out_fp32, ldc,
 * ldr) as sv_op_gemm_bf16; ldw >= K.  Needs C % 64 == 0, stride <= 8 and -pad, pad - (k - 1) within [-128, 127]: other geometries ->
 * SV_ERR_UNSUPPORTED (gather with sv_op_im2col instead).  Bad arguments -> SV_ERR_INVALID, checked before the device is touched. */
int sv_op_conv_gemm_bf16(const uint16_t* x, int32_t B, int32_t H, int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad,
                         const uint16_t* Wt, int64_t ldw, int32_t N, const float* bias, int32_t act, const float* residual, int64_t ldr,
                         void* out, int64_t ldc, int32_t out_fp32, void* stream);

/* Host-only plan query for a convolution (touches neither device nor driver).  conv_info[SV_CONV_PLAN_INFO_LEN]: 0 A operand form
 * (SV_GEMM_A_IM2COL: sv_op_conv_gemm_bf16 runs it; SV_GEMM_A_TILED: not eligible, the im2col buffer + 2-D tiled A map path), 1 Ho,
 * 2 Wo, 3 M = B * Ho * Wo, 4 K = k * k * C.  gemm_info (may be NULL): sv_op_gemm_plan_info of that GEMM (K rounded up to a multiple
 * of 8 on the tiled path).  Bad arguments -> SV_ERR_INVALID. */
#define SV_GEMM_A_TILED 0
#define SV_GEMM_A_IM2COL 1
#define SV_CONV_PLAN_INFO_LEN 5
int sv_op_conv_gemm_plan_info(int32_t B, int32_t H, int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad, int32_t N, int32_t out_fp32,
                              int32_t has_residual, int32_t pair_request, int32_t num_sms, int32_t* conv_info, int32_t* gemm_info);

/* LayerNorm over the last dim of fp32 [rows, C] -> optional fp32 and/or bf16 outputs (either may be NULL). */
int sv_op_layernorm(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int32_t C,
                    float* out_f32, uint16_t* out_bf16, void* stream);

/* The same LayerNorm with its fp32 result channel-major: rows = frames * tokens_per_frame token-major rows in, out_nchw[frame][c][token]
 * out (the NCHW map of each frame), bit-identical to sv_op_layernorm's out_f32 permuted; out_bf16 (may be NULL) is token-major as in
 * sv_op_layernorm.  rows must be a multiple of tokens_per_frame and rows * C < 2^31; x, gamma, beta 16-byte aligned, out_bf16 8-byte,
 * out_nchw 4-byte.  Argument errors -> SV_ERR_INVALID before anything is launched. */
int sv_op_layernorm_nchw(const float* x, const float* gamma, const float* beta, float eps, int64_t rows, int32_t C, int32_t tokens_per_frame,
                         float* out_nchw, uint16_t* out_bf16, void* stream);

/* Patch gather (im2col) with k index ordered (kh, kw, cin), row stride ldo (zero padded to ldo).
 * src_nchw_f32 != NULL: source is [B,Cin,H,W] fp32; else src_nhwc_bf16 is [B,H,W,Cin] bf16 (Cin%8==0). */
int sv_op_im2col(const float* src_nchw_f32, const uint16_t* src_nhwc_bf16, int32_t B, int32_t Cin, int32_t H, int32_t W,
                 int32_t k, int32_t stride, int32_t pad, uint16_t* out, int64_t ldo, void* stream);

/* depthwise 3x3 (zero pad 1, per-frame) + bias + GELU(erf) on NHWC bf16 (mix_transformer_evp.py:22-30,63).
 * w: [9, C] fp32 (tap-major), bias [C] fp32. */
int sv_op_dwconv3x3_gelu(const uint16_t* x, const float* w, const float* bias, int32_t B, int32_t H, int32_t W,
                         int32_t C, uint16_t* out, void* stream);

/* How sv_op_dwconv3x3_gelu runs a problem on a device with num_sms SMs.  Host only: touches neither device nor driver; the launch
 * takes its geometry from the same function.  It depends on B, H, W, C and the switches SURGVID_DW_CPL / _GELU / _STAGES /
 * _PREFETCH, read once per process.  info[SV_DWCONV_PLAN_INFO_LEN]:
 *   0 kernel (SV_DWCONV_*), 1 channels per lane (cpl), 2 GELU form (0 erf polynomial, 1 sigmoid on ex2/rcp, 2 tanh.approx),
 *   3 shared-memory ring stages, 4 prefetch distance (both 0 for the SIMT kernel), 5 output columns per tile (tw), 6 tiles_x,
 *   7 tiles_y (7-row tiles), 8 channel blocks (32 * cpl channels), 9 num_tiles, 10 grid (CTAs), 11 most tiles one CTA walks,
 *   12 some CTA's tile range crosses a frame boundary, 13 some CTA's range crosses a channel-block boundary.
 * The TMA kernel takes C % 128 == 0; the SIMT kernel (one 7 x 8 x 128 tile per CTA, polynomial GELU) every other C % 4 == 0 and
 * B * ceil(H / 7) <= 65535.  Shape errors (as sv_op_dwconv3x3_gelu reports them) -> SV_ERR_INVALID. */
#define SV_DWCONV_SIMT 0
#define SV_DWCONV_TMA 1
#define SV_DWCONV_PLAN_INFO_LEN 14
int sv_op_dwconv_plan_info(int32_t B, int32_t H, int32_t W, int32_t C, int32_t num_sms, int32_t* info);

/* softmax(Q K^T * scale) V per (frame, head). Q rows = B*Nq, K/V rows = B*Nkv; head h occupies columns
 * [h*hd, (h+1)*hd) of each; hd in {20, 32, 40, 64} (mix_transformer_evp.py:123-127, 868-883).  ldq, ldk, ldv % 8 == 0 and
 * q, k, v 16-byte aligned; ldo even and o 4-byte aligned; only the [B*Nq, heads*hd] block of o is written. */
int sv_op_attention(const uint16_t* q, int64_t ldq, const uint16_t* k, int64_t ldk, const uint16_t* v, int64_t ldv,
                    uint16_t* o, int64_t ldo, int32_t B, int32_t heads, int32_t Nq, int32_t Nkv, int32_t hd, float scale,
                    void* stream);

/* Which kernel sv_op_attention runs for these operands (it depends on pointer alignment, leading dims, N_kv, hd and the
 * SURGVID_ATTN_TC switch, not on B, heads or Nq): one of SV_ATTN_*.  Host only; nothing is read through the pointers. */
#define SV_ATTN_TC_SINGLE 0      /* attention_tc_single_kernel: tcgen05, hd 64, N_kv <= 64 */
#define SV_ATTN_TC_MULTI 1       /* attention_tc_kernel<true>: tcgen05, hd 64, 64 < N_kv <= 448 */
#define SV_ATTN_RESIDENT 2       /* attention_resident_kv_kernel: mma.sync, N_kv <= 64 */
#define SV_ATTN_RESIDENT_MULTI 3 /* attention_resident_multi_kernel: mma.sync, N_kv <= 256 */
#define SV_ATTN_STREAM 4         /* attention_kernel: mma.sync, streamed key tiles, online softmax */
int sv_op_attention_kernel(const uint16_t* q, int64_t ldq, const uint16_t* k, int64_t ldk, const uint16_t* v, int64_t ldv,
                           const uint16_t* o, int64_t ldo, int32_t Nkv, int32_t hd);

/* Attention probabilities p[b, h, i, j] = softmax_j(q_i . k_j * scale), fp32, written to a contiguous [B, heads, Nq, Nkv] array
 * (64-bit offsets).  q, k as for sv_op_attention (head h = columns [h*hd, (h+1)*hd); ldq, ldk % 8 == 0; q, k 16-byte aligned);
 * p 4-byte aligned.  hd 32 or 64 (else SV_ERR_UNSUPPORTED); any Nq, Nkv >= 1.  Every row sums to 1 within fp32 rounding. */
int sv_op_attention_probs(const uint16_t* q, int64_t ldq, const uint16_t* k, int64_t ldk, int32_t B, int32_t heads, int32_t Nq,
                          int32_t Nkv, int32_t hd, float scale, float* p, void* stream);

/* reflect-pad-2 + 5x5 binomial/256 depthwise filter on fp32 NCHW (mix_transformer_evp.py:500-514). */
int sv_op_gauss5x5(const float* x, float* out, int32_t planes, int32_t H, int32_t W, void* stream);

/* bilinear (align_corners=False) resize of NHWC bf16 tokens [B,H,W,C] -> [B,Ho,Wo,C] written with row
 * stride ldo (segformer_head.py:149-156 semantics, applied before the per-pixel projection). */
int sv_op_bilinear_tokens(const uint16_t* x, int32_t B, int32_t H, int32_t W, int32_t C, int32_t Ho, int32_t Wo,
                          uint16_t* out, int64_t ldo, void* stream);

/* Fused first-layer conv: Conv2d(Cin<=3 -> Cout in {16,32,64}, k7, s4, p3) on fp32 NCHW + bias, then LayerNorm(eps) over Cout
 * (relu == 0; gamma/beta required) or ReLU (relu != 0).  w: [Cout, ldw] bf16 with k = (kh, kw, cin), zero padded, ldw % 8 == 0.
 * Outputs are token-major [B*Ho*Wo, Cout]; either may be NULL.  replaces OverlapPatchEmbed(patch_size=7, stride=4)
 * (mix_transformer_evp.py:209-215) and flow_encoder.conv1+bn1+act (:846). */
int sv_op_stem_conv(const float* src, const uint16_t* w, int32_t ldw, const float* bias, const float* gamma, const float* beta,
                    float eps, int32_t relu, int32_t B, int32_t Cin, int32_t H, int32_t W, int32_t Cout, float* out_f32,
                    uint16_t* out_bf16, void* stream);

/* sv_op_gemm_bf16 with the A operand given as two K segments: out = act([A | A2] . W^T + bias) (+ residual), where the last K2 of
 * the K columns come from A2[:, 0:K2] (row stride lda2) and the first K - K2 (a multiple of 64) from A.  This is how block i's fc2
 * consumes [GELU(DWConv(h)) | T_{i+1}] against [W_fc2 | W_shared] (Mlp.forward + PromptGenerator.get_prompt,
 * mix_transformer_evp.py:60-67, 776-815) without materialising the concatenation. */
int sv_op_gemm_bf16_cat(const uint16_t* A, int64_t lda, const uint16_t* A2, int64_t lda2, int32_t K2, const uint16_t* W, int64_t ldw,
                        int32_t M, int32_t N, int32_t K, const float* bias, int32_t act, const float* residual, int64_t ldr, void* out,
                        int64_t ldc, int32_t out_fp32, void* stream);

/* Second half of the MixFFN in one kernel (Mlp.forward, mix_transformer_evp.py:63-66): the depthwise 3x3 conv + GELU is the producer
 * of the fc2 GEMM's A tiles, so GELU(DWConv(h1)) never goes to memory.
 *   x[M, N] (fp32, in place) += bias[N] + GELU(dwconv3x3(h1) + b_dw) . Wcat[:, :hidden]^T  (+ tail[M, tail_cols] . Wcat[:, hidden:]^T)
 * h1: bf16 [frames, H, W, hidden] (M = frames*H*W); w10c: fp32 [10, hidden] = 9 taps (kh*3+kw) then the depthwise bias;
 * Wcat: bf16 [N, ldw]; tail: bf16 [M, ldt] or NULL with tail_cols == 0.  W must be even and <= 128; returns SV_ERR_INVALID otherwise. */
int sv_op_mixffn_fc2(const uint16_t* h1, const float* w10c, const uint16_t* Wcat, int64_t ldw, const float* bias, const uint16_t* tail,
                     int64_t ldt, int32_t tail_cols, float* x, int64_t ldx, int32_t frames, int32_t H, int32_t W, int32_t hidden, int32_t N,
                     void* stream);

/* mean over `tokens` consecutive rows of fp32 [B*tokens, C] -> [B, C] (AdaptiveAvgPool2d(1), segformer_head.py:167). */
int sv_op_token_mean(const float* x, int32_t B, int32_t tokens, int32_t C, float* out, void* stream);

/* ---- Trans-SVNet head (SURVEY.md 8f-1): the inner module of adapter_transformer.Transformer —
 * `self.transformer = Transformer2_3_1(d_model=out_features, d_ff=mstcn_f_maps, d_k=d_v=min(64, mstcn_f_maps), n_layers=1, n_heads=4,
 * len_q=sequence_length)` (adapter_transformer.py:317-325) called as `self.transformer(inputs, feas)` (:348) — fused with the window
 * construction of Transformer.original_forward (:335-344): the kernel reads the MS-TCN logits and the decoder query directly.
 * The source of Transformer2_3_1 is absent from the reference tree; the arithmetic is the published upstream architecture restated in
 * oracle/trans_head_oracle.py (PARITY UNPINNED).  state_dict keys expected by sv_trans_set_tensor:
 *   {encoder.layers.0.enc_self_attn, decoder.layers.0.dec_enc_attn}.{W_Q,W_K,W_V,fc}.{weight[,bias]}, .layer_norm.{weight,bias},
 *   {encoder,decoder}.layers.0.pos_ffn.{fc1,fc2}.{weight[,bias]}, .layer_norm.{weight,bias}   (missing biases = 0). */
typedef struct sv_trans_cfg {
  int32_t d_model;   /* out_features (14) */
  int32_t d_ff;      /* mstcn_f_maps (32 or 64), <= 64 */
  int32_t d_k, d_v;  /* min(64, mstcn_f_maps); d_k = d_v = 32 or 64 supported, anything else is SV_ERR_UNSUPPORTED */
  int32_t n_layers;  /* 1 */
  int32_t n_heads;   /* 4 */
  int32_t len_q;     /* sequence_length (30), <= 32 */
} sv_trans_cfg;
typedef struct sv_trans sv_trans_handle;
int sv_trans_create(const sv_trans_cfg* cfg, sv_trans_handle** out);
int sv_trans_destroy(sv_trans_handle* h);
/* Tensors are stored by name and checked at sv_trans_pack_weights (missing key -> SV_ERR_STATE, wrong shape -> SV_ERR_INVALID);
 * shape == NULL with ndim > 0, or a negative dimension -> SV_ERR_INVALID. */
int sv_trans_set_tensor(sv_trans_handle* h, const char* name, const float* host_data, const int64_t* shape, int32_t ndim);
int sv_trans_pack_weights(sv_trans_handle* h);
/* logits: fp32 channel-major [d_model][ldx] = the LAST stage of sv_mstcn_forward's output for the concatenated videos
 * (x of Transformer.original_forward, adapter_transformer.py:329-330); query: fp32 [T, d_model] = tanh(fc(LFB)) (sv_mstcn_forward_query);
 * video_offsets: host int64 [n_videos + 1]; out: fp32 [T, d_model] = transformer(inputs, feas).squeeze(1).  Windows are zero-padded on
 * the left and never cross a video boundary. */
int sv_trans_forward(sv_trans_handle* h, const float* logits, int64_t ldx, const float* query, const int64_t* video_offsets,
                     int32_t n_videos, float* out, void* stream);
/* Online use, the counterpart of sv_mstcn_stream_step: the head of the frames of one step, bit-identical to sv_trans_forward over the
 * same video's frames.  State (sv_trans_stream_state_bytes, zeroed by sv_trans_stream_reset, 256-byte aligned): int64 seen[n_streams]
 * padded to 256 bytes, then per stream a ring of len_q - 1 rows x d_model fp32 of the last logits rows (position q in slot
 * q mod (len_q - 1)).  Reset works as sv_mstcn_stream_reset.  logits [d_model][ldx] = the last stage of the step's logits, query
 * [sum(counts), d_model], out [sum(counts), d_model]; stream_ids / counts as in sv_mstcn_stream_step.  Only the step's frames are
 * computed; two launches (head, ring commit). */
size_t sv_trans_stream_state_bytes(const sv_trans_handle* h, int32_t n_streams);
int sv_trans_stream_reset(sv_trans_handle* h, void* state, size_t state_bytes, int32_t n_streams, const int32_t* stream_ids,
                          int32_t n_ids, void* stream);
int sv_trans_stream_forward(sv_trans_handle* h, void* state, size_t state_bytes, int32_t n_streams, const float* logits, int64_t ldx,
                            const float* query, const int32_t* stream_ids, const int64_t* counts, int32_t n_ids, float* out, void* stream);

/* ---- on-GPU input transforms (SURVEY.md 8f-2): the reference's per-frame dataset transforms, applied to device copies of
 * the raw uint8 frames / float32 RAFT flow instead of on the CPU inside CholecFlowDataset.__getitem__ (data_process.py:409-483).
 * A handle fixes the geometry and owns the coefficient tables; buffers and the workspace belong to the caller. */
typedef struct sv_prep sv_prep;

/* in_h x in_w: size of the uint8 RGB frames / segmentation maps; flow_h x flow_w: size of the raw flow field (0, 0 = no flow);
 * resize, crop: transforms.Resize((resize, resize)) then CenterCrop(crop) (generate_evp_LFB.py:243-245; 250 and 224);
 * mean3/std3: transforms.Normalize constants (generate_evp_LFB.py:247). */
int sv_prep_create(int32_t in_h, int32_t in_w, int32_t flow_h, int32_t flow_w, int32_t resize, int32_t crop, const float* mean3,
                   const float* std3, sv_prep** out);
int sv_prep_destroy(sv_prep* h);
/* bytes of device scratch sv_prep_images needs for B frames (uint8 intermediate between Pillow's two resampling passes) */
size_t sv_prep_workspace_bytes(const sv_prep* h, int32_t B);
/* src: uint8 [B, in_h, in_w, 3] (HWC, RGB) -> out: float32 [B, 3, crop, crop]:
 * Resize (Pillow antialiased bilinear, bit-exact) -> CenterCrop -> ToTensor -> Normalize (generate_evp_LFB.py:242-248). */
int sv_prep_images(sv_prep* h, const uint8_t* src, int32_t B, float* out, void* workspace, size_t workspace_bytes, void* stream);
/* flow: float32 [B, flow_h, flow_w, 2] -> out: float32 [B, 2, crop, crop]: cv2.resize(INTER_LINEAR) to (resize, resize),
 * u *= resize/flow_w, v *= resize/flow_h, CenterCrop (data_process.py:432-447, 461-480). */
int sv_prep_flow(sv_prep* h, const float* flow, int32_t B, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SURGVID_H_ */
