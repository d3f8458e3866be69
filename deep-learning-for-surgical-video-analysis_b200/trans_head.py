"""The part of the reference's Trans-SVNet head that the reference itself defines (SURVEY.md §8f-1).

`adapter_transformer.Transformer` (adapter_transformer.py:290-352) wraps an inner `Transformer2_3_1` module whose source is
NOT in the reference (it is imported from a file that does not exist there), so that module cannot be restated or pinned.
What `Transformer.original_forward` does around it is fully specified and is reproduced here on the GPU:

  * `inputs[t] = out_features[t-len_q+1 .. t]` with zero left padding — a `[T, len_q, 14]` tensor of causal windows of the
    MS-TCN logits (adapter_transformer.py:335-344; the reference builds it with a Python loop and `.cuda()` calls);
  * `feas = tanh(fc(long_feature))` with `fc = Linear(f_dim, out_features, bias=False)` (adapter_transformer.py:325,348),
    computed by the MS-TCN stage-1 projection kernel in the SAME pass over the `[T, 2048]` features (14 extra columns).

`TransformerInputs` has the constructor arguments and the `fc.weight` state_dict key of the reference class; the inner module
is whatever the user supplies (`original_forward(..., transformer=module)`), called exactly as the reference calls it.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import _native, ops
from .mstcn import MultiStageModel_S


class TransformerInputs(nn.Module):
    def __init__(self, mstcn_f_maps, mstcn_f_dim, out_features, len_q, **kwargs):
        super().__init__()
        self.num_f_maps, self.dim, self.num_classes, self.len_q = mstcn_f_maps, mstcn_f_dim, out_features, len_q
        self.fc = nn.Linear(mstcn_f_dim, out_features, bias=False)  # adapter_transformer.py:325
        self._attached_to = None

    def attach(self, mstcn_model: MultiStageModel_S):
        """Pack `fc.weight` next to the MS-TCN stage-1 projection of `mstcn_model` (call again after changing fc.weight)."""
        mstcn_model.set_query_head(self.fc.weight)
        self._attached_to = mstcn_model
        return self

    @torch.no_grad()
    def prepare(self, mstcn_model: MultiStageModel_S, long_feature: torch.Tensor, lengths: Sequence[int]):
        """long_feature [sum(lengths), f_dim] fp32 CUDA, videos concatenated ->
        (logits [stages, C, T], inputs [T, len_q, C], feas [T, 1, C]) — the arguments of `self.transformer(inputs, feas)`."""
        if self._attached_to is not mstcn_model:
            self.attach(mstcn_model)
        logits, query = mstcn_model.forward_videos_query(long_feature, lengths)
        inputs = ops.causal_windows(logits[-1], lengths, self.len_q)
        return logits, inputs, query.unsqueeze(1)

    @torch.no_grad()
    def original_forward(self, x: torch.Tensor, long_feature: torch.Tensor, transformer: Optional[nn.Module] = None):
        """Reference signature (adapter_transformer.py:329): x = last-stage MS-TCN output [1, C, T], long_feature [1, T, f_dim].
        Returns `transformer(inputs, feas)` when the inner module is supplied, else the pair (inputs, feas)."""
        if not x.is_cuda:
            raise RuntimeError("surgvid_b200 has no CPU path: move the inputs to a CUDA (sm_100a) device")
        T = x.shape[2]
        inputs = ops.causal_windows(x[0].to(torch.float32).contiguous(), [T], self.len_q)
        lf = long_feature.reshape(T, self.dim).to(torch.float32).contiguous()
        if self._attached_to is None:
            raise RuntimeError("call attach(mstcn_model) first: the fc projection runs inside the MS-TCN stage-1 kernel")
        _, q = self._attached_to.forward_videos_query(lf, [T])
        feas = q.unsqueeze(1)
        return transformer(inputs, feas) if transformer is not None else (inputs, feas)


# ----------------------------------------------------------------------------------------------------------------------------------
# The inner module and the complete head.  `transformer2_3_1.py` is NOT part of the reference tree (adapter_transformer.py:9 imports a
# file that does not exist there), so this is built from the published upstream architecture (see oracle/trans_head_oracle.py) and its
# parity is UNPINNED: constructor arguments and the call signature are the reference's (adapter_transformer.py:317-325, 348), the
# parameter names below are this package's.
class _MultiHeadAttention(nn.Module):
    def __init__(self, d_model, d_k, d_v, n_heads, bias=True):
        super().__init__()
        self.W_Q = nn.Linear(d_model, d_k * n_heads, bias=bias)
        self.W_K = nn.Linear(d_model, d_k * n_heads, bias=bias)
        self.W_V = nn.Linear(d_model, d_v * n_heads, bias=bias)
        self.fc = nn.Linear(n_heads * d_v, d_model, bias=bias)
        self.layer_norm = nn.LayerNorm(d_model)


class _PoswiseFeedForwardNet(nn.Module):
    def __init__(self, d_model, d_ff, bias=True):
        super().__init__()
        self.fc1 = nn.Linear(d_model, d_ff, bias=bias)
        self.fc2 = nn.Linear(d_ff, d_model, bias=bias)
        self.layer_norm = nn.LayerNorm(d_model)


class _EncoderLayer(nn.Module):
    def __init__(self, d_model, d_ff, d_k, d_v, n_heads, bias):
        super().__init__()
        self.enc_self_attn = _MultiHeadAttention(d_model, d_k, d_v, n_heads, bias)
        self.pos_ffn = _PoswiseFeedForwardNet(d_model, d_ff, bias)


class _DecoderLayer(nn.Module):
    def __init__(self, d_model, d_ff, d_k, d_v, n_heads, bias):
        super().__init__()
        self.dec_enc_attn = _MultiHeadAttention(d_model, d_k, d_v, n_heads, bias)
        self.pos_ffn = _PoswiseFeedForwardNet(d_model, d_ff, bias)


class _Stack(nn.Module):
    def __init__(self, layers):
        super().__init__()
        self.layers = nn.ModuleList(layers)


class Transformer2_3_1(nn.Module):
    """`Transformer2_3_1(d_model, d_ff, d_k, d_v, n_layers, n_heads, len_q)` (adapter_transformer.py:317-325): parameter holder whose
    forward runs as ONE CUDA kernel (`sv_trans_forward`).  Two call forms:
      * `forward(enc_inputs [T, len_q, d_model], dec_inputs [T, 1, d_model])` — the reference's call (:348); the windows must be the
        causal windows of one logits sequence (they are read back as `enc_inputs[:, -1]`, and the zero padding as the video start);
      * `forward_fused(logits_last [d_model, T_total], query [T_total, d_model], lengths)` — no window tensor at all."""

    def __init__(self, d_model, d_ff, d_k, d_v, n_layers, n_heads, len_q, bias=True):
        super().__init__()
        self.d_model, self.d_ff, self.d_k, self.d_v, self.n_layers, self.n_heads, self.len_q = d_model, d_ff, d_k, d_v, n_layers, n_heads, len_q
        self.encoder = _Stack([_EncoderLayer(d_model, d_ff, d_k, d_v, n_heads, bias) for _ in range(n_layers)])
        self.decoder = _Stack([_DecoderLayer(d_model, d_ff, d_k, d_v, n_heads, bias) for _ in range(n_layers)])
        self._native = {}
        self._weights_epoch = 0

    def _apply(self, fn, *a, **k):
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1
        return super().load_state_dict(*a, **k)

    def refresh_weights(self):
        self._weights_epoch += 1

    def _state(self, device):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        st = self._native.get(idx)
        if st is not None and st["stamp"] == self._weights_epoch:
            return st
        lib = _native.lib()
        with torch.cuda.device(idx):
            if st is None:
                cfg = _native.TransCfg(self.d_model, self.d_ff, self.d_k, self.d_v, self.n_layers, self.n_heads, self.len_q)
                h = ctypes.c_void_p()
                _native.check(lib.sv_trans_create(ctypes.byref(cfg), ctypes.byref(h)), "sv_trans_create")
                st = {"handle": h}
                self._native[idx] = st
            for name, t in self.state_dict().items():
                a = np.ascontiguousarray(t.detach().to("cpu", torch.float32).numpy())
                shape = (ctypes.c_int64 * max(a.ndim, 1))(*a.shape)
                _native.check(lib.sv_trans_set_tensor(st["handle"], name.encode(), a.ctypes.data_as(ctypes.c_void_p), shape, a.ndim), "sv_trans_set_tensor")
            _native.check(lib.sv_trans_pack_weights(st["handle"]), "sv_trans_pack_weights")
        st["stamp"] = self._weights_epoch
        return st

    @torch.no_grad()
    def forward_fused(self, logits_last: torch.Tensor, query: torch.Tensor, lengths: Sequence[int]) -> torch.Tensor:
        """logits_last [d_model, T_total] fp32 CUDA (row stride may exceed T_total), query [T_total, d_model] -> [T_total, 1, d_model]."""
        if self.training:
            raise RuntimeError("surgvid_b200 models are inference-only: call .eval() first")
        if not logits_last.is_cuda:
            raise RuntimeError("surgvid_b200 has no CPU path: move the inputs to a CUDA (sm_100a) device")
        assert logits_last.dtype == torch.float32 and logits_last.shape[0] == self.d_model
        T = logits_last.shape[1]
        if T > 1 and logits_last.stride(1) != 1:
            logits_last = logits_last.contiguous()
        off = np.zeros(len(lengths) + 1, dtype=np.int64)
        off[1:] = np.cumsum(np.asarray(list(lengths), dtype=np.int64))
        if int(off[-1]) != T:
            raise ValueError("sum(lengths) must equal the number of frames")
        query = query.reshape(T, self.d_model).to(torch.float32).contiguous()
        out = torch.empty((T, self.d_model), dtype=torch.float32, device=logits_last.device)
        st = self._state(logits_last.device)
        rc = _native.lib().sv_trans_forward(st["handle"], ctypes.c_void_p(logits_last.data_ptr()), max(T, logits_last.stride(0)), ctypes.c_void_p(query.data_ptr()),
                                            off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(lengths), ctypes.c_void_p(out.data_ptr()),
                                            ctypes.c_void_p(torch.cuda.current_stream(out.device).cuda_stream))
        _native.check(rc, "sv_trans_forward")
        return out.unsqueeze(1)

    def forward(self, enc_inputs: torch.Tensor, dec_inputs: torch.Tensor) -> torch.Tensor:
        """The reference's call `self.transformer(inputs, feas)` (adapter_transformer.py:348) for ONE video: enc_inputs [T, len_q, d_model]
        are the causal windows Transformer.original_forward builds (:335-344), so window t's newest row is frame t's logits."""
        T = enc_inputs.shape[0]
        logits_last = enc_inputs[:, -1, :].t().contiguous()
        return self.forward_fused(logits_last, dec_inputs.reshape(T, self.d_model), [T])

    def __del__(self):
        try:
            for st in self._native.values():
                _native.lib().sv_trans_destroy(st["handle"])
        except (AttributeError, TypeError, ImportError):
            pass


class Transformer(TransformerInputs):
    """Drop-in for adapter_transformer.Transformer (:290-352): same constructor arguments, `fc.weight` and `transformer.*` parameters,
    `original_forward(x, long_feature)`; `forward_videos` runs MS-TCN + head for any number of concatenated videos."""

    def __init__(self, mstcn_f_maps, mstcn_f_dim, out_features, len_q, **kwargs):
        super().__init__(mstcn_f_maps, mstcn_f_dim, out_features, len_q, **kwargs)
        attn_dim = min(64, mstcn_f_maps)                                   # adapter_transformer.py:315
        self.transformer = Transformer2_3_1(d_model=out_features, d_ff=mstcn_f_maps, d_k=attn_dim, d_v=attn_dim, n_layers=1, n_heads=4, len_q=len_q)

    @torch.no_grad()
    def original_forward(self, x: torch.Tensor, long_feature: torch.Tensor, transformer: Optional[nn.Module] = None):
        """x: last-stage MS-TCN output [1, C, T]; long_feature [1, T, f_dim] -> [T, 1, C] (adapter_transformer.py:329-352)."""
        if transformer is not None:
            return super().original_forward(x, long_feature, transformer)
        if self._attached_to is None:
            raise RuntimeError("call attach(mstcn_model) first: the fc projection runs inside the MS-TCN stage-1 kernel")
        T = x.shape[2]
        lf = long_feature.reshape(T, self.dim).to(torch.float32).contiguous()
        _, q = self._attached_to.forward_videos_query(lf, [T])
        return self.transformer.forward_fused(x[0].to(torch.float32).contiguous(), q, [T])

    forward = original_forward

    @torch.no_grad()
    def forward_videos(self, mstcn_model: MultiStageModel_S, long_feature: torch.Tensor, lengths: Sequence[int]):
        """trans_SV_output.py:268-301 for all videos at once: (MS-TCN logits [stages, C, T_total], head output [T_total, 1, C])."""
        if self._attached_to is not mstcn_model:
            self.attach(mstcn_model)
        logits, query = mstcn_model.forward_videos_query(long_feature, lengths)
        return logits, self.transformer.forward_fused(logits[-1], query, lengths)

    def open_stream(self, mstcn_model: MultiStageModel_S, n_streams: int, device=None) -> "TransStream":
        """Online use of MS-TCN + head for `n_streams` videos (see `TransStream`)."""
        if self.training or self.transformer.training:
            raise RuntimeError("surgvid_b200 models are inference-only: call .eval() first")
        if self._attached_to is not mstcn_model:
            self.attach(mstcn_model)
        return TransStream(self, mstcn_model.open_stream(n_streams, device))


class TransStream:
    """`Transformer.open_stream`: an `MstcnStream` plus the head's own state (the last len_q - 1 last-stage logits rows of every stream).
    `step(feats, stream_ids, counts)` returns (logits [stages, C, n], head_out [n, 1, C]) for the step's rows, bit-identical to
    `Transformer.forward_videos` over each video's frames so far; `reset(ids)` resets both states together."""

    def __init__(self, head: Transformer, mstcn_stream):
        self._head, self.mstcn = head, mstcn_stream
        self.n_streams, self.device = mstcn_stream.n_streams, mstcn_stream.device
        nbytes = int(_native.lib().sv_trans_stream_state_bytes(self._handle(), self.n_streams))
        self._state = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self.reset()

    @property
    def seen(self) -> torch.Tensor:
        return self.mstcn.seen

    def _handle(self):
        with torch.cuda.device(self.device):
            return self._head.transformer._state(self.device)["handle"]

    def reset(self, ids=None):
        self.mstcn.reset(ids)
        cs = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        lib = _native.lib()
        if ids is None:
            _native.check(lib.sv_trans_stream_reset(self._handle(), ctypes.c_void_p(self._state.data_ptr()), self._state.numel(), self.n_streams,
                                                    None, 0, cs), "sv_trans_stream_reset")
            self._epoch = self._head.transformer._weights_epoch
            return
        a = np.ascontiguousarray(np.asarray(ids, dtype=np.int32).reshape(-1))
        _native.check(lib.sv_trans_stream_reset(self._handle(), ctypes.c_void_p(self._state.data_ptr()), self._state.numel(), self.n_streams,
                                                a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), a.size, cs), "sv_trans_stream_reset")

    @torch.no_grad()
    def step(self, feats: torch.Tensor, stream_ids, counts):
        if self._head.transformer._weights_epoch != self._epoch:
            raise RuntimeError("the head's weights changed since this stream state was computed: call reset() first")
        if self._head._attached_to is not self.mstcn._model:
            raise RuntimeError("the head's query projection was attached to another MS-TCN model: open a new stream")
        logits, query = self.mstcn.step(feats, stream_ids, counts, query=True)
        n = logits.shape[2]
        ids = np.ascontiguousarray(np.asarray(stream_ids, dtype=np.int32).reshape(-1))
        cnt = np.ascontiguousarray(np.asarray(counts, dtype=np.int64).reshape(-1))
        out = torch.empty((n, self._head.num_classes), dtype=torch.float32, device=self.device)
        last = logits[-1]
        rc = _native.lib().sv_trans_stream_forward(self._handle(), ctypes.c_void_p(self._state.data_ptr()), self._state.numel(), self.n_streams,
                                                   ctypes.c_void_p(last.data_ptr()), last.stride(0), ctypes.c_void_p(query.data_ptr()),
                                                   ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                                   ids.size, ctypes.c_void_p(out.data_ptr()),
                                                   ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        _native.check(rc, "sv_trans_stream_forward")
        return logits, out.unsqueeze(1)
