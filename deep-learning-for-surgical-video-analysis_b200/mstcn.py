"""Drop-in for the reference's `mstcn.py` on the LFB path: `MultiStageModel_S` (+ its `SingleStageModel`,
`DilatedResidualLayer` parameter holders).

Same positional constructor `MultiStageModel_S(stages, layers, f_maps, f_dim, out_features, causal_conv)`
(trans_SV_output.py:197), same 72 state_dict keys (`stage1_phase.conv_1x1.*`, `stage1_phase.layers.{i}.{conv_dilated,conv_1x1}.*`,
`stage1_phase.conv_out_classes.*`, `stages.{s}. ...`), same `forward(x)` contract: x `[1, f_dim, T]` (normally the
transposed *view* of a time-major `[1, T, f_dim]` tensor, trans_SV_output.py:271-272) -> `[stages, 1, out_features, T]`.
The arithmetic (mstcn.py:122-130, 173-178, 208-214) runs in libsurgvid.so behind `torch.ops.surgvid.mstcn_forward`;
there is no PyTorch fallback.  `forward_videos` is the batched entry point (all videos of a shard in one call).
"""
from __future__ import annotations

import copy
import ctypes
from typing import Sequence

import numpy as np
import torch
import torch.nn as nn

from . import _native, ops
from .models.segformer_head import _Holder


class DilatedResidualLayer(_Holder):
    def __init__(self, dilation, in_channels, out_channels, causal_conv=False, kernel_size=3):
        super().__init__()
        self.causal_conv, self.dilation, self.kernel_size = causal_conv, dilation, kernel_size
        pad = dilation * (kernel_size - 1) if causal_conv else dilation
        self.conv_dilated = nn.Conv1d(in_channels, out_channels, kernel_size, padding=pad, dilation=dilation)
        self.conv_1x1 = nn.Conv1d(out_channels, out_channels, 1)
        self.dropout = nn.Dropout()


class SingleStageModel(_Holder):
    def __init__(self, num_layers, num_f_maps, dim, num_classes, causal_conv=False):
        super().__init__()
        self.conv_1x1 = nn.Conv1d(dim, num_f_maps, 1)
        self.layers = nn.ModuleList([DilatedResidualLayer(2 ** i, num_f_maps, num_f_maps, causal_conv=causal_conv) for i in range(num_layers)])
        self.conv_out_classes = nn.Conv1d(num_f_maps, num_classes, 1)


class MultiStageModel_S(nn.Module):
    def __init__(self, mstcn_stages, mstcn_layers, mstcn_f_maps, mstcn_f_dim, out_features, mstcn_causal_conv):
        super().__init__()
        self.num_stages, self.num_layers, self.num_f_maps = mstcn_stages, mstcn_layers, mstcn_f_maps
        self.dim, self.num_classes, self.causal_conv = mstcn_f_dim, out_features, mstcn_causal_conv
        # the reference echoes its configuration at construction (mstcn.py:102-104); kept so logs look the same
        print(f"num_stages_classification: {self.num_stages}, num_layers: {self.num_layers}, num_f_maps: {self.num_f_maps}, dim: {self.dim}")
        if not mstcn_causal_conv:
            raise NotImplementedError("only mstcn_causal_conv=True (trans_SV_output.py:197) is implemented on the CUDA path")
        self.stage1_phase = SingleStageModel(self.num_layers, self.num_f_maps, self.dim, self.num_classes, causal_conv=self.causal_conv)
        self.stages = nn.ModuleList([
            copy.deepcopy(SingleStageModel(self.num_layers, self.num_f_maps, self.num_classes, self.num_classes, causal_conv=self.causal_conv))
            for _ in range(self.num_stages - 1)])
        self.smoothing = False
        self._native = {}
        self._weights_epoch = 0
        self._fc_weight = None  # optional Trans-SVNet query head packed next to the stage-1 projection (set_query_head)

    # ------------------------------------------------------------------ native plumbing
    def _apply(self, fn, *args, **kwargs):
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1
        return super().load_state_dict(*args, **kwargs)

    def refresh_weights(self):
        self._weights_epoch += 1

    def set_query_head(self, fc_weight):
        """Attach `Transformer.fc.weight` ([out_features, f_dim], no bias; adapter_transformer.py:325) so that
        `forward_videos_query` also returns tanh(fc(features)) from the same pass over the features.  None detaches it."""
        if fc_weight is not None:
            fc_weight = fc_weight.detach().to("cpu", torch.float32).contiguous()
            if fc_weight.dim() != 2 or fc_weight.shape[1] != self.dim or not (1 <= fc_weight.shape[0] <= 16):
                raise ValueError(f"fc weight must be [<=16, {self.dim}], got {tuple(fc_weight.shape)}")
        self._fc_weight = fc_weight
        # the native handle keeps tensors by name: rebuild it so that a detached head really disappears
        for st in self._native.values():
            if st.get("id") is not None:
                ops.unregister_handle(st["id"])
            _native.lib().sv_mstcn_destroy(st["handle"])
        self._native = {}
        self._weights_epoch += 1

    def _state(self, device: torch.device):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        st = self._native.get(idx)
        if st is not None and st["stamp"] == self._weights_epoch:
            return st
        lib = _native.lib()
        with torch.cuda.device(idx):
            if st is None:
                cfg = _native.MstcnCfg(self.num_stages, self.num_layers, self.num_f_maps, self.dim, self.num_classes, int(bool(self.causal_conv)))
                h = ctypes.c_void_p()
                _native.check(lib.sv_mstcn_create(ctypes.byref(cfg), ctypes.byref(h)), "sv_mstcn_create")
                st = {"handle": h, "workspace": None, "id": None}
                self._native[idx] = st
            for name, t in self.state_dict().items():
                a = np.ascontiguousarray(t.detach().to("cpu", torch.float32).numpy())
                shape = (ctypes.c_int64 * max(a.ndim, 1))(*a.shape)
                _native.check(lib.sv_mstcn_set_tensor(st["handle"], name.encode(), a.ctypes.data_as(ctypes.c_void_p), shape, a.ndim), "sv_mstcn_set_tensor")
            if self._fc_weight is not None:
                a = self._fc_weight.numpy()
                shape = (ctypes.c_int64 * 2)(*a.shape)
                _native.check(lib.sv_mstcn_set_tensor(st["handle"], b"fc.weight", a.ctypes.data_as(ctypes.c_void_p), shape, 2), "sv_mstcn_set_tensor")
            _native.check(lib.sv_mstcn_pack_weights(st["handle"]), "sv_mstcn_pack_weights")
        st["stamp"] = self._weights_epoch
        if st["id"] is None:
            st["id"] = ops.register_handle(_MstcnOpOwner(self, idx))
        return st

    def _native_forward(self, idx: int, feats: torch.Tensor, offsets: torch.Tensor, want_query: bool = False):
        st = self._native[idx]
        lib = _native.lib()
        T = feats.shape[0]
        nbytes = lib.sv_mstcn_workspace_bytes(st["handle"], T)
        ws = st["workspace"]
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=feats.device)
            st["workspace"] = ws
        out = torch.empty((self.num_stages, self.num_classes, T), dtype=torch.float32, device=feats.device)
        off = np.ascontiguousarray(offsets.detach().cpu().numpy().astype(np.int64))
        query = None
        if want_query:
            if self._fc_weight is None:
                raise RuntimeError("no query head attached: call set_query_head(fc_weight) first")
            query = torch.empty((T, self._fc_weight.shape[0]), dtype=torch.float32, device=feats.device)
        rc = lib.sv_mstcn_forward_query(st["handle"], ctypes.c_void_p(feats.data_ptr()), off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                        len(off) - 1, ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(0 if query is None else query.data_ptr()),
                                        ctypes.c_void_p(ws.data_ptr()), ws.numel(),
                                        ctypes.c_void_p(torch.cuda.current_stream(feats.device).cuda_stream))
        _native.check(rc, "sv_mstcn_forward_query")
        return (out, query) if want_query else out

    def last_launch_count(self, device=None) -> int:
        idx = torch.cuda.current_device() if device is None else torch.device(device).index
        st = self._native.get(idx)
        return 0 if st is None else int(_native.lib().sv_mstcn_last_launch_count(st["handle"]))

    # ------------------------------------------------------------------ forward
    def _check(self, t: torch.Tensor):
        if self.training:
            raise RuntimeError("surgvid_b200 models are inference-only: call model.eval() first (trans_SV_output.py:203)")
        if not t.is_cuda:
            raise RuntimeError("surgvid_b200 has no CPU path: move the inputs to a CUDA (sm_100a) device")

    def forward_videos(self, feats: torch.Tensor, lengths: Sequence[int]) -> torch.Tensor:
        """feats: [sum(lengths), f_dim] fp32 time-major, videos concatenated -> logits [stages, out_features, sum(lengths)]."""
        self._check(feats)
        feats = feats.to(torch.float32).contiguous()
        offsets = torch.zeros(len(lengths) + 1, dtype=torch.int64)
        offsets[1:] = torch.cumsum(torch.as_tensor(list(lengths), dtype=torch.int64), 0)
        if int(offsets[-1]) != feats.shape[0]:
            raise ValueError("sum(lengths) must equal feats.shape[0]")
        st = self._state(feats.device)
        return torch.ops.surgvid.mstcn_forward(feats, offsets, st["id"])

    def forward_videos_query(self, feats: torch.Tensor, lengths: Sequence[int]):
        """`forward_videos` plus the Trans-SVNet decoder query tanh(fc(feats)) [sum(lengths), out_features]
        (adapter_transformer.py:348), both from one pass over `feats`.  Needs `set_query_head`."""
        self._check(feats)
        feats = feats.to(torch.float32).contiguous()
        offsets = torch.zeros(len(lengths) + 1, dtype=torch.int64)
        offsets[1:] = torch.cumsum(torch.as_tensor(list(lengths), dtype=torch.int64), 0)
        if int(offsets[-1]) != feats.shape[0]:
            raise ValueError("sum(lengths) must equal feats.shape[0]")
        st = self._state(feats.device)
        return torch.ops.surgvid.mstcn_forward_query(feats, offsets, st["id"])

    def open_stream(self, n_streams: int, device=None) -> "MstcnStream":
        """Online use: `n_streams` independent videos fed a few frames at a time (see `MstcnStream`).  `device` defaults to the
        model's device, which must be a CUDA device."""
        if self.training:
            raise RuntimeError("surgvid_b200 models are inference-only: call model.eval() first (trans_SV_output.py:203)")
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("surgvid_b200 has no CPU path: open the stream on a CUDA (sm_100a) device")
        return MstcnStream(self, int(n_streams), dev)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: [B, f_dim, T] -> [stages, B, out_features, T] (mstcn.py:122-130)."""
        self._check(x)
        B, D, T = x.shape
        feats = x.transpose(1, 2).to(torch.float32).contiguous().view(B * T, D)  # zero-copy for the reference's transposed view
        out = self.forward_videos(feats, [T] * B)
        return out.view(self.num_stages, self.num_classes, B, T).permute(0, 2, 1, 3)

    def __del__(self):
        try:
            for st in self._native.values():
                if st.get("id") is not None:
                    ops.unregister_handle(st["id"])
                _native.lib().sv_mstcn_destroy(st["handle"])
        except (AttributeError, TypeError, ImportError):
            pass  # interpreter shutdown: module globals are already gone; anything else (a failing destroy) propagates as "ignored exception" text


def _step_tables(stream_ids, counts, n_rows: int):
    ids = np.ascontiguousarray(np.asarray(stream_ids, dtype=np.int64).reshape(-1))
    cnt = np.ascontiguousarray(np.asarray(counts, dtype=np.int64).reshape(-1))
    if ids.shape != cnt.shape or ids.size == 0:
        raise ValueError("stream_ids and counts must be non-empty and of the same length")
    if int(cnt.sum()) != n_rows:
        raise ValueError(f"sum(counts) = {int(cnt.sum())} must equal the number of feature rows ({n_rows})")
    if ids.min() < np.iinfo(np.int32).min or ids.max() > np.iinfo(np.int32).max:
        raise ValueError("stream id out of range")
    return np.ascontiguousarray(ids.astype(np.int32)), cnt


class MstcnStream:
    """Per-video state of `n_streams` videos on the GPU for online phase recognition (`MultiStageModel_S.open_stream`).

    `step(feats, stream_ids, counts)` takes new feature rows for some of the streams (rows of stream_ids[k], counts[k] >= 1 of them,
    grouped in that order) and returns their logits [stages, C, sum(counts)], bit-identical to `forward_videos` over each video's frames
    so far.  The state holds what the causal layers still need of each video's past (the last 2 * 2^l inputs of layer l), so a step costs
    the same whatever the history.  The state was computed with the weights of the last reset: after `load_state_dict` or `.to()`,
    `step` raises until `reset()`."""

    def __init__(self, model: MultiStageModel_S, n_streams: int, device: torch.device):
        if n_streams < 1:
            raise ValueError("n_streams >= 1")
        self._model, self.n_streams = model, n_streams
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        lib = _native.lib()
        st = model._state(self.device)
        nbytes = int(lib.sv_mstcn_stream_state_bytes(st["handle"], n_streams))
        self._state = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._ws = None
        self._seen = np.zeros(n_streams, dtype=np.int64)
        self.reset()

    @property
    def seen(self) -> torch.Tensor:
        """Frames each stream has consumed since its last reset (a CPU copy)."""
        return torch.from_numpy(self._seen.copy())

    def _handle(self):
        with torch.cuda.device(self.device):
            return self._model._state(self.device)["handle"]

    def reset(self, ids=None):
        """Make the next frame of the listed streams (all when ids is None) frame 0 of a new video.  Resetting every stream also adopts
        the model's current weights."""
        h = self._handle()
        cs = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        lib = _native.lib()
        if ids is None:
            _native.check(lib.sv_mstcn_stream_reset(h, ctypes.c_void_p(self._state.data_ptr()), self._state.numel(), self.n_streams, None, 0, cs),
                          "sv_mstcn_stream_reset")
            self._seen[:] = 0
            self._epoch = self._model._weights_epoch
            return
        a = np.ascontiguousarray(np.asarray(ids, dtype=np.int32).reshape(-1))
        _native.check(lib.sv_mstcn_stream_reset(h, ctypes.c_void_p(self._state.data_ptr()), self._state.numel(), self.n_streams,
                                                a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), a.size, cs), "sv_mstcn_stream_reset")
        self._seen[a] = 0

    def step(self, feats: torch.Tensor, stream_ids, counts, query: bool = False):
        """feats [sum(counts), f_dim] fp32 CUDA -> logits [stages, C, sum(counts)]; with query=True, (logits, query [sum(counts), q])
        (needs `set_query_head`)."""
        m = self._model
        if m._weights_epoch != self._epoch:
            raise RuntimeError("the model's weights changed since this stream state was computed: call reset() first")
        m._check(feats)
        feats = feats.to(torch.float32).contiguous()
        if feats.dim() != 2 or feats.shape[1] != m.dim:
            raise ValueError(f"feats must be [rows, {m.dim}], got {tuple(feats.shape)}")
        n = feats.shape[0]
        ids, cnt = _step_tables(stream_ids, counts, n)
        lib = _native.lib()
        h = self._handle()
        nbytes = int(lib.sv_mstcn_stream_workspace_bytes(h, n))
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        out = torch.empty((m.num_stages, m.num_classes, n), dtype=torch.float32, device=self.device)
        q = None
        if query:
            if m._fc_weight is None:
                raise RuntimeError("no query head attached: call set_query_head(fc_weight) first")
            q = torch.empty((n, m._fc_weight.shape[0]), dtype=torch.float32, device=self.device)
        rc = lib.sv_mstcn_stream_step(h, ctypes.c_void_p(self._state.data_ptr()), self._state.numel(), self.n_streams, ctypes.c_void_p(feats.data_ptr()),
                                      ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), ids.size,
                                      ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(0 if q is None else q.data_ptr()),
                                      ctypes.c_void_p(self._ws.data_ptr()), self._ws.numel(),
                                      ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        _native.check(rc, "sv_mstcn_stream_step")
        self._seen[ids] += cnt
        return (out, q) if query else out


class _MstcnOpOwner:
    def __init__(self, model: MultiStageModel_S, idx: int):
        import weakref

        self._model = weakref.ref(model)
        self._idx = idx
        self.num_stages, self.num_classes = model.num_stages, model.num_classes

    def _native_forward(self, feats, offsets, want_query=False):
        return self._model()._native_forward(self._idx, feats, offsets, want_query)

    @property
    def query_dim(self):
        m = self._model()
        return 0 if m is None or m._fc_weight is None else int(m._fc_weight.shape[0])
