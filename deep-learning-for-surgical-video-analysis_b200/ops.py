"""PyTorch custom ops (`torch.ops.surgvid.*`) over the C ABI, plus thin tensor wrappers of the single kernels.

PyTorch is plumbing here: it owns device memory (inputs, outputs, workspace through the caching allocator)
and the stream; all arithmetic happens inside libsurgvid.so.  CUDA only — there is no CPU implementation.
"""
from __future__ import annotations

import ctypes
import itertools
from typing import Dict, List, Optional

import torch

from . import _native

_HANDLES: Dict[int, "object"] = {}  # op-visible integer id -> owner object (keeps native handles alive)


def _stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("surgvid ops run on CUDA tensors only (no CPU fallback); got a tensor on " + str(t.device))


# ----------------------------------------------------------------------------------------------- custom ops
@torch.library.custom_op("surgvid::evp_lfb_forward", mutates_args=())
def evp_lfb_forward(x: torch.Tensor, seg: torch.Tensor, flow: Optional[torch.Tensor], handle: int, micro_batch: int) -> torch.Tensor:
    """[B,3,H,W] frames + segmaps (+ [B,2,H,W] flow) -> [B, 2048] LFB features.
    Replaces model_LFB.forward(inputs, segmaps, flow, return_features=True) (generate_evp_LFB.py:454)."""
    owner = _HANDLES[handle]
    return owner._native_forward(x, seg, flow, micro_batch)


@evp_lfb_forward.register_fake
def _(x, seg, flow, handle, micro_batch):
    return x.new_empty((x.shape[0], _HANDLES[handle].embedding_dim), dtype=torch.float32)


@torch.library.custom_op("surgvid::evp_forward_features", mutates_args=())
def evp_forward_features(x: torch.Tensor, seg: torch.Tensor, handle: int, micro_batch: int) -> List[torch.Tensor]:
    """[B,3,H,W] frames + segmaps -> the encoder's four stage maps, fp32 NCHW [B, C_s, H_s, W_s] (encoder only: no flow, no head).
    Replaces MixVisionTransformerEVP.forward_features(x, y) (mix_transformer_evp.py:352-416)."""
    return _HANDLES[handle]._native_forward_features(x, seg, micro_batch)


@evp_forward_features.register_fake
def _(x, seg, handle, micro_batch):
    B, _, H, W = x.shape
    return [x.new_empty((B, c, h, w), dtype=torch.float32) for c, h, w in _HANDLES[handle].stage_shapes(H, W)]


@torch.library.custom_op("surgvid::mstcn_forward", mutates_args=())
def mstcn_forward(feats: torch.Tensor, offsets: torch.Tensor, handle: int) -> torch.Tensor:
    """feats [T_total, f_dim] fp32 time-major, offsets int64 CPU [n_videos+1] -> logits [stages, out_features, T_total].
    Replaces MultiStageModel_S.forward (mstcn.py:122-130; call site trans_SV_output.py:279)."""
    owner = _HANDLES[handle]
    return owner._native_forward(feats, offsets)


@mstcn_forward.register_fake
def _(feats, offsets, handle):
    o = _HANDLES[handle]
    return feats.new_empty((o.num_stages, o.num_classes, feats.shape[0]), dtype=torch.float32)


@torch.library.custom_op("surgvid::mstcn_forward_query", mutates_args=())
def mstcn_forward_query(feats: torch.Tensor, offsets: torch.Tensor, handle: int) -> tuple[torch.Tensor, torch.Tensor]:
    """`mstcn_forward` plus query[T_total, q] = tanh(feats @ fc.weight.T) from the same pass over the features
    (Transformer.original_forward, adapter_transformer.py:348)."""
    owner = _HANDLES[handle]
    return owner._native_forward(feats, offsets, True)


@mstcn_forward_query.register_fake
def _(feats, offsets, handle):
    o = _HANDLES[handle]
    return (feats.new_empty((o.num_stages, o.num_classes, feats.shape[0]), dtype=torch.float32),
            feats.new_empty((feats.shape[0], o.query_dim), dtype=torch.float32))


def causal_windows(x: torch.Tensor, lengths, len_q: int) -> torch.Tensor:
    """x [C, T_total] fp32 (row stride may exceed T_total) -> [T_total, len_q, C]: per video, window t holds frames t-len_q+1..t with
    zeros before the video's first frame (the `inputs` tensor of adapter_transformer.py:335-344)."""
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    C, T = x.shape
    import numpy as np
    off = np.zeros(len(lengths) + 1, dtype=np.int64)
    off[1:] = np.cumsum(np.asarray(list(lengths), dtype=np.int64))
    if int(off[-1]) != T:
        raise ValueError("sum(lengths) must equal x.shape[1]")
    out = torch.empty((T, len_q, C), dtype=torch.float32, device=x.device)
    rc = _native.lib().sv_op_causal_windows(_ptr(x), x.stride(0), C, off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(lengths), len_q, _ptr(out),
                                            _stream_ptr(x.device))
    _native.check(rc, "sv_op_causal_windows")
    return out


_NEXT_HANDLE = itertools.count(1)


def register_handle(owner) -> int:
    """A fresh integer id per registration (never reused, unlike id(owner) after garbage collection)."""
    hid = next(_NEXT_HANDLE)
    _HANDLES[hid] = owner
    return hid


def unregister_handle(hid: int):
    _HANDLES.pop(hid, None)


# ----------------------------------------------------------------------------------------------- single kernels
def gemm_bf16(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = 0,
              residual: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.bfloat16, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = act(a @ w.T + bias) (+ residual); a [M,K] bf16, w [N,K] bf16 (row strides may exceed K)."""
    _require_cuda(a, w, bias, residual, out)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    assert out.stride(1) == 1 and out.dtype in (torch.bfloat16, torch.float32)
    lib = _native.lib()
    rc = lib.sv_op_gemm_bf16(_ptr(a), a.stride(0), _ptr(w), w.stride(0), M, N, K, _ptr(bias), act, _ptr(residual),
                             0 if residual is None else residual.stride(0), _ptr(out), out.stride(0), int(out.dtype == torch.float32),
                             _stream_ptr(a.device))
    _native.check(rc, "sv_op_gemm_bf16")
    return out


GEMM_PLAN_FIELDS = ("block_n", "pair", "tma_out", "num_stages", "epi_bufs", "epi_lag", "prefetch", "num_tiles", "grid", "epilogue", "kernel",
                    "num_n_tiles", "smem_bytes")
GEMM_EPILOGUES = ("bf16_tma", "f32_tma", "f32_tma_resid", "transpose")   # SV_GEMM_EPI_* in include/surgvid.h


def gemm_plan_info(M: int, N: int, K: int, K2: int = 0, out_fp32: bool = False, residual: bool = False, pair: int = -1,
                   num_sms: Optional[int] = None) -> dict:
    """The launch plan gemm_bf16 / gemm_bf16_cat choose for this problem (sv_op_gemm_plan_info; host only).  `num_sms` defaults to
    the current device's SM count; `epilogue` is named by GEMM_EPILOGUES."""
    if num_sms is None:
        num_sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    info = (ctypes.c_int32 * len(GEMM_PLAN_FIELDS))()
    _native.check(_native.lib().sv_op_gemm_plan_info(M, N, K, K2, int(out_fp32), int(residual), pair, num_sms, info), "sv_op_gemm_plan_info")
    d = dict(zip(GEMM_PLAN_FIELDS, info))
    d["epilogue"] = GEMM_EPILOGUES[d["epilogue"]]
    return d


def conv_gemm(x: torch.Tensor, w: torch.Tensor, k: int, stride: int, pad: int, bias: Optional[torch.Tensor] = None, act: int = 0,
              residual: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.bfloat16, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Convolution as an implicit GEMM (sv_op_conv_gemm_bf16): x [B,H,W,C] bf16 NHWC (C % 64 == 0), w [N, k*k*C] bf16 in (kh, kw, cin)
    order (row stride may exceed k*k*C) -> out [B*Ho*Wo, N] = act(im2col(x) @ w.T + bias) (+ residual), rows in (b, oh, ow) order.
    Bit-identical to gemm_bf16(im2col(x, k, stride, pad), w, ...) without the im2col buffer."""
    _require_cuda(x, w, bias, residual, out)
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and x.is_contiguous() and w.stride(1) == 1
    B, H, W, C = x.shape
    M = B * ((H + 2 * pad - k) // stride + 1) * ((W + 2 * pad - k) // stride + 1)
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x.device)
    assert out.stride(1) == 1 and out.dtype in (torch.bfloat16, torch.float32)
    rc = _native.lib().sv_op_conv_gemm_bf16(_ptr(x), B, H, W, C, k, stride, pad, _ptr(w), w.stride(0), N, _ptr(bias), act, _ptr(residual),
                                            0 if residual is None else residual.stride(0), _ptr(out), out.stride(0), int(out.dtype == torch.float32),
                                            _stream_ptr(x.device))
    _native.check(rc, "sv_op_conv_gemm_bf16")
    return out


CONV_A_FORMS = ("tiled", "im2col")   # SV_GEMM_A_* in include/surgvid.h


def conv_gemm_plan_info(B: int, H: int, W: int, C: int, k: int, stride: int, pad: int, N: int, out_fp32: bool = False, residual: bool = False,
                        pair: int = -1, num_sms: int = 148) -> dict:
    """How a convolution runs (sv_op_conv_gemm_plan_info; host only): `a_form` "im2col" (conv_gemm reads the NHWC input through an
    im2col-mode TMA map) or "tiled" (not eligible: im2col buffer + gemm_bf16), Ho, Wo, M, K, and under "gemm" the GEMM's plan
    (gemm_plan_info's fields)."""
    ci = (ctypes.c_int32 * 5)()
    gi = (ctypes.c_int32 * len(GEMM_PLAN_FIELDS))()
    _native.check(_native.lib().sv_op_conv_gemm_plan_info(B, H, W, C, k, stride, pad, N, int(out_fp32), int(residual), pair, num_sms, ci, gi),
                  "sv_op_conv_gemm_plan_info")
    d = dict(zip(("a_form", "Ho", "Wo", "M", "K"), ci))
    d["a_form"] = CONV_A_FORMS[d["a_form"]]
    d["gemm"] = dict(zip(GEMM_PLAN_FIELDS, gi))
    d["gemm"]["epilogue"] = GEMM_EPILOGUES[d["gemm"]["epilogue"]]
    return d


def gemm_bf16_cat(a: torch.Tensor, a2: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = 0,
                  residual: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.bfloat16, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = act(cat([a, a2], 1) @ w.T + bias) (+ residual) without building the concatenation; a [M,K1] (K1 % 64 == 0), a2 [M,K2] bf16
    (row strides may exceed the widths), w [N, K1+K2] bf16."""
    _require_cuda(a, a2, w, bias, residual, out)
    M, K1 = a.shape
    K2 = a2.shape[1]
    N = w.shape[0]
    assert w.shape[1] == K1 + K2 and a2.shape[0] == M and a.stride(1) == 1 and a2.stride(1) == 1 and w.stride(1) == 1
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    rc = _native.lib().sv_op_gemm_bf16_cat(_ptr(a), a.stride(0), _ptr(a2), a2.stride(0), K2, _ptr(w), w.stride(0), M, N, K1 + K2, _ptr(bias), act,
                                           _ptr(residual), 0 if residual is None else residual.stride(0), _ptr(out), out.stride(0),
                                           int(out.dtype == torch.float32), _stream_ptr(a.device))
    _native.check(rc, "sv_op_gemm_bf16_cat")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, want_f32=False, want_bf16=True):
    _require_cuda(x, gamma, beta)
    rows, C = x.shape
    of = torch.empty_like(x) if want_f32 else None
    ob = torch.empty((rows, C), dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    rc = _native.lib().sv_op_layernorm(_ptr(x), _ptr(gamma), _ptr(beta), eps, rows, C, _ptr(of), _ptr(ob), _stream_ptr(x.device))
    _native.check(rc, "sv_op_layernorm")
    return of, ob


def layernorm_nchw(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, tokens_per_frame: int, want_bf16=False):
    """LayerNorm of token-major fp32 x [frames * tokens_per_frame, C] -> (fp32 [frames, C, tokens_per_frame] channel-major, the
    token-major bf16 [rows, C] or None); bit-identical to `layernorm(..., want_f32=True)[0]` permuted (sv_op_layernorm_nchw)."""
    _require_cuda(x, gamma, beta)
    rows, C = x.shape
    out = torch.empty((rows // tokens_per_frame, C, tokens_per_frame), dtype=torch.float32, device=x.device)
    ob = torch.empty((rows, C), dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    rc = _native.lib().sv_op_layernorm_nchw(_ptr(x), _ptr(gamma), _ptr(beta), eps, rows, C, tokens_per_frame, _ptr(out), _ptr(ob),
                                            _stream_ptr(x.device))
    _native.check(rc, "sv_op_layernorm_nchw")
    return out, ob


def im2col(src: torch.Tensor, k: int, stride: int, pad: int, ldo: Optional[int] = None) -> torch.Tensor:
    """src: [B,Cin,H,W] fp32 (NCHW) or [B,H,W,Cin] bf16 (NHWC) -> [B*Ho*Wo, ldo] bf16, k index (kh,kw,cin)."""
    _require_cuda(src)
    if src.dtype == torch.float32:
        B, Cin, H, W = src.shape
    else:
        B, H, W, Cin = src.shape
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    K = k * k * Cin
    ldo = ldo or (K + 7) // 8 * 8
    out = torch.empty((B * Ho * Wo, ldo), dtype=torch.bfloat16, device=src.device)
    nchw, nhwc = (src, None) if src.dtype == torch.float32 else (None, src)
    rc = _native.lib().sv_op_im2col(_ptr(nchw), _ptr(nhwc), B, Cin, H, W, k, stride, pad, _ptr(out), ldo, _stream_ptr(src.device))
    _native.check(rc, "sv_op_im2col")
    return out


def dwconv3x3_gelu(x: torch.Tensor, w9c: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """x [B,H,W,C] bf16 NHWC, w9c [9,C] fp32, bias [C] fp32 -> GELU(dwconv3x3(x)+bias) bf16."""
    _require_cuda(x, w9c, bias)
    B, H, W, C = x.shape
    out = torch.empty_like(x)
    rc = _native.lib().sv_op_dwconv3x3_gelu(_ptr(x), _ptr(w9c), _ptr(bias), B, H, W, C, _ptr(out), _stream_ptr(x.device))
    _native.check(rc, "sv_op_dwconv3x3_gelu")
    return out


DWCONV_PLAN_FIELDS = ("kernel", "cpl", "gelu", "stages", "prefetch", "tw", "tiles_x", "tiles_y", "cblks", "num_tiles", "grid",
                      "max_tiles_per_cta", "crosses_frame", "crosses_cblk")
DWCONV_KERNELS = ("simt", "tma")   # SV_DWCONV_* in include/surgvid.h


def dwconv_plan_info(B: int, H: int, W: int, C: int, num_sms: Optional[int] = None) -> dict:
    """How dwconv3x3_gelu runs this problem (sv_op_dwconv_plan_info; host only).  `num_sms` defaults to the current device's SM count;
    `kernel` is named by DWCONV_KERNELS."""
    if num_sms is None:
        num_sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    info = (ctypes.c_int32 * len(DWCONV_PLAN_FIELDS))()
    _native.check(_native.lib().sv_op_dwconv_plan_info(B, H, W, C, num_sms, info), "sv_op_dwconv_plan_info")
    d = dict(zip(DWCONV_PLAN_FIELDS, info))
    d["kernel"] = DWCONV_KERNELS[d["kernel"]]
    return d


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, heads: int, hd: int, scale: float,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q [B*Nq, >=heads*hd] bf16, k/v [B*Nkv, ...] bf16 (row-strided views allowed) -> o [B*Nq, heads*hd] bf16, written into `out`
    when given (its row stride may exceed heads*hd)."""
    _require_cuda(q, k, v, out)
    Nq, Nkv = q.shape[0] // B, k.shape[0] // B
    if out is None:
        out = torch.empty((q.shape[0], heads * hd), dtype=torch.bfloat16, device=q.device)
    assert out.dtype == torch.bfloat16 and tuple(out.shape) == (q.shape[0], heads * hd) and out.stride(1) == 1
    rc = _native.lib().sv_op_attention(_ptr(q), q.stride(0), _ptr(k), k.stride(0), _ptr(v), v.stride(0), _ptr(out), out.stride(0), B, heads, Nq,
                                       Nkv, hd, scale, _stream_ptr(q.device))
    _native.check(rc, "sv_op_attention")
    return out


def attention_probs(q: torch.Tensor, k: torch.Tensor, B: int, heads: int, Nq: int, Nkv: int, hd: int, scale: float,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(Q K^T * scale) as fp32 [B, heads, Nq, Nkv]: q [B*Nq, >=heads*hd] bf16, k [B*Nkv, >=heads*hd] bf16 (row-strided views
    allowed, as for `attention`); written into `out` (contiguous fp32) when given."""
    _require_cuda(q, k, out)
    assert q.dtype == torch.bfloat16 and k.dtype == torch.bfloat16 and q.stride(1) == 1 and k.stride(1) == 1
    assert q.shape[0] == B * Nq and k.shape[0] == B * Nkv
    if out is None:
        out = torch.empty((B, heads, Nq, Nkv), dtype=torch.float32, device=q.device)
    assert out.dtype == torch.float32 and tuple(out.shape) == (B, heads, Nq, Nkv) and out.is_contiguous()
    rc = _native.lib().sv_op_attention_probs(_ptr(q), q.stride(0), _ptr(k), k.stride(0), B, heads, Nq, Nkv, hd, scale, _ptr(out),
                                             _stream_ptr(q.device))
    _native.check(rc, "sv_op_attention_probs")
    return out


def gauss5x5(x: torch.Tensor) -> torch.Tensor:
    _require_cuda(x)
    B, C, H, W = x.shape
    out = torch.empty_like(x)
    rc = _native.lib().sv_op_gauss5x5(_ptr(x), _ptr(out), B * C, H, W, _stream_ptr(x.device))
    _native.check(rc, "sv_op_gauss5x5")
    return out


def bilinear_tokens(x: torch.Tensor, Ho: int, Wo: int) -> torch.Tensor:
    _require_cuda(x)
    B, H, W, C = x.shape
    out = torch.empty((B, Ho, Wo, C), dtype=torch.bfloat16, device=x.device)
    rc = _native.lib().sv_op_bilinear_tokens(_ptr(x), B, H, W, C, Ho, Wo, _ptr(out), C, _stream_ptr(x.device))
    _native.check(rc, "sv_op_bilinear_tokens")
    return out


def token_mean(x: torch.Tensor, tokens: int) -> torch.Tensor:
    _require_cuda(x)
    rows, C = x.shape
    B = rows // tokens
    out = torch.empty((B, C), dtype=torch.float32, device=x.device)
    rc = _native.lib().sv_op_token_mean(_ptr(x), B, tokens, C, _ptr(out), _stream_ptr(x.device))
    _native.check(rc, "sv_op_token_mean")
    return out


def mixffn_fc2(h1: torch.Tensor, w9c: torch.Tensor, dw_bias: torch.Tensor, wcat: torch.Tensor, bias: Optional[torch.Tensor], x: torch.Tensor,
               tail: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [B*H*W, N] fp32 (updated IN PLACE and returned) += bias + GELU(dwconv3x3(h1) + dw_bias) @ wcat[:, :hidden].T (+ tail @ wcat[:, hidden:].T).
    h1 [B,H,W,hidden] bf16, w9c [9,hidden] fp32, wcat [N, hidden(+tail cols)] bf16, tail [B*H*W, cols] bf16."""
    _require_cuda(h1, w9c, dw_bias, wcat, bias, x, tail)
    B, H, W, hidden = h1.shape
    N = wcat.shape[0]
    w10c = torch.cat([w9c.reshape(9, hidden), dw_bias.reshape(1, hidden)], 0).contiguous().float()
    tc = 0 if tail is None else tail.shape[1]
    assert wcat.shape[1] == hidden + tc and x.shape == (B * H * W, N) and x.dtype == torch.float32
    rc = _native.lib().sv_op_mixffn_fc2(_ptr(h1), _ptr(w10c), _ptr(wcat), wcat.stride(0), _ptr(bias), _ptr(tail), 0 if tail is None else tail.stride(0),
                                        tc, _ptr(x), x.stride(0), B, H, W, hidden, N, _stream_ptr(h1.device))
    _native.check(rc, "sv_op_mixffn_fc2")
    return x


def stem_conv(src: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, gamma: Optional[torch.Tensor] = None, beta: Optional[torch.Tensor] = None,
              eps: float = 1e-5, relu: bool = False):
    """src [B,Cin,H,W] fp32; weight [Cout,Cin,7,7] fp32 (packed here to the kernel's (kh,kw,cin) bf16 layout) -> (fp32, bf16) token-major
    [B*Ho*Wo, Cout] of LayerNorm(conv(src)+bias) (or ReLU(conv+bias) when relu)."""
    _require_cuda(src, weight, bias, gamma, beta)
    B, Cin, H, W = src.shape
    Cout = weight.shape[0]
    K = 49 * Cin
    ldw = (K + 7) // 8 * 8
    wp = torch.zeros((Cout, ldw), dtype=torch.bfloat16, device=src.device)
    wp[:, :K] = weight.permute(0, 2, 3, 1).reshape(Cout, K).to(torch.bfloat16)
    Ho, Wo = (H + 6 - 7) // 4 + 1, (W + 6 - 7) // 4 + 1
    of = torch.empty((B * Ho * Wo, Cout), dtype=torch.float32, device=src.device)
    ob = torch.empty((B * Ho * Wo, Cout), dtype=torch.bfloat16, device=src.device)
    rc = _native.lib().sv_op_stem_conv(_ptr(src), _ptr(wp), ldw, _ptr(bias), _ptr(gamma), _ptr(beta), eps, int(relu), B, Cin, H, W, Cout, _ptr(of),
                                       _ptr(ob), _stream_ptr(src.device))
    _native.check(rc, "sv_op_stem_conv")
    return of, ob
