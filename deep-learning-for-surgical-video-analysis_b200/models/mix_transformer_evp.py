"""Drop-in for the reference's `models/mix_transformer_evp.py` on the LFB path.

Same constructors (`mit_b0_evp()` ... `mit_b5_evp()`, `MixVisionTransformerEVP(...)`), same attribute tree, same
`state_dict()` keys and shapes (722 keys for b3; SURVEY.md §8b), same call
`model.forward(x, y, flow=None, return_features=False)` (mix_transformer_evp.py:418-449) — but the modules below are
*parameter holders only*: the arithmetic runs in libsurgvid.so (hand-written sm_100a kernels) behind the custom op
`torch.ops.surgvid.evp_lfb_forward`.  There is no PyTorch / CPU fallback: calling a holder directly, or calling the
model on a non-CUDA tensor, raises.

Differences from the reference, all deliberate:
  * any HxW is accepted (the reference hard-codes `view(-1,3,224,224)`, :354-355; SURVEY.md F8);
  * inference only (`model.eval()`, as the LFB driver does at generate_evp_LFB.py:437); train mode raises because
    DropPath / Dropout / BatchNorm batch statistics are not implemented;
  * `GaussianFilter.kernel` (a non-buffer tensor pinned to a module-level device, :463,498-509) is baked into the kernel.
"""
from __future__ import annotations

import ctypes
import math
import os
from functools import partial
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from .. import _native, ops, visualizer
from .segformer_head import SegFormerHead, _Holder


def _trunc_normal_(t, std=0.02):
    return nn.init.trunc_normal_(t, mean=0.0, std=std, a=-2.0, b=2.0)


def _ref_init(m: nn.Module):
    """The reference's `_init_weights` distributions (mix_transformer_evp.py:300-313)."""
    if isinstance(m, nn.Linear):
        _trunc_normal_(m.weight, 0.02)
        if m.bias is not None:
            nn.init.zeros_(m.bias)
    elif isinstance(m, nn.LayerNorm):
        nn.init.ones_(m.weight)
        nn.init.zeros_(m.bias)
    elif isinstance(m, nn.Conv2d):
        fan_out = m.kernel_size[0] * m.kernel_size[1] * m.out_channels // m.groups
        m.weight.data.normal_(0.0, math.sqrt(2.0 / fan_out))
        if m.bias is not None:
            m.bias.data.zero_()


class DWConv(_Holder):
    def __init__(self, dim=768):
        super().__init__()
        self.dwconv = nn.Conv2d(dim, dim, 3, 1, 1, bias=True, groups=dim)


class Mlp(_Holder):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.0):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.dwconv = DWConv(hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)


class Attention(_Holder):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0.0, proj_drop=0.0, sr_ratio=1):
        super().__init__()
        assert dim % num_heads == 0, f"dim {dim} should be divided by num_heads {num_heads}."
        if qk_scale is not None:
            raise NotImplementedError("qk_scale override is not supported by the fused attention kernel")
        self.dim, self.num_heads, self.sr_ratio = dim, num_heads, sr_ratio
        self.scale = (dim // num_heads) ** -0.5
        self.q = nn.Linear(dim, dim, bias=qkv_bias)
        self.kv = nn.Linear(dim, dim * 2, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        if sr_ratio > 1:
            self.sr = nn.Conv2d(dim, dim, kernel_size=sr_ratio, stride=sr_ratio)
            self.norm = nn.LayerNorm(dim)


class Block(_Holder):
    def __init__(self, dim, num_heads, mlp_ratio=4.0, qkv_bias=False, qk_scale=None, drop=0.0, attn_drop=0.0, drop_path=0.0,
                 act_layer=nn.GELU, norm_layer=nn.LayerNorm, sr_ratio=1):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop, proj_drop=drop,
                              sr_ratio=sr_ratio)
        self.drop_path = nn.Identity()  # stochastic depth is identity in eval; no parameters either way
        self.drop_path_prob = float(drop_path)
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)


class OverlapPatchEmbed(_Holder):
    def __init__(self, img_size=224, patch_size=7, stride=4, in_chans=3, embed_dim=768):
        super().__init__()
        self.img_size = (img_size, img_size) if isinstance(img_size, int) else tuple(img_size)
        self.patch_size = (patch_size, patch_size)
        self.H, self.W = self.img_size[0] // patch_size, self.img_size[1] // patch_size
        self.num_patches = self.H * self.W
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=stride, padding=patch_size // 2)
        self.norm = nn.LayerNorm(embed_dim)


class PromptGenerator(_Holder):
    """EVP adapter parameters (mix_transformer_evp.py:550-698) for the configuration the reference hard-codes
    (:278-285): scale_factor 4, tuning_stage '1234', input_type 'gaussian', adaptor 'adaptor'."""

    def __init__(self, scale_factor, prompt_type, embed_dims, tuning_stage, depths, input_type, freq_nums, handcrafted_tune,
                 embedding_tune, adaptor, img_size):
        super().__init__()
        if (str(tuning_stage), input_type, adaptor, bool(handcrafted_tune), bool(embedding_tune)) != ("1234", "gaussian", "adaptor", True, True):
            raise NotImplementedError("only the reference's hard-coded EVP configuration is implemented")
        self.scale_factor, self.prompt_type, self.embed_dims, self.tuning_stage = scale_factor, prompt_type, embed_dims, tuning_stage
        self.depths, self.input_type, self.freq_nums, self.adaptor, self.img_size = depths, input_type, freq_nums, adaptor, img_size
        self.handcrafted_tune, self.embedding_tune = handcrafted_tune, embedding_tune
        widths = [d // scale_factor for d in embed_dims]
        geom = [(img_size, 7, 4, 3), (img_size // 4, 3, 2, widths[0]), (img_size // 8, 3, 2, widths[1]), (img_size // 16, 3, 2, widths[2])]
        for s, (sz, k, st, cin) in enumerate(geom):
            setattr(self, f"handcrafted_generator{s + 1}", OverlapPatchEmbed(img_size=sz, patch_size=k, stride=st, in_chans=cin, embed_dim=widths[s]))
        for s in range(4):
            setattr(self, f"embedding_generator{s + 1}", nn.Linear(embed_dims[s], widths[s]))
        for s in range(4):
            for i in range(depths[s]):
                setattr(self, f"lightweight_mlp{s + 1}_{i}", nn.Sequential(nn.Linear(widths[s], widths[s]), nn.GELU()))
            setattr(self, f"shared_mlp{s + 1}", nn.Linear(widths[s], embed_dims[s]))
        self.apply(_ref_init)


class OpticalFlowEncoder(_Holder):
    def __init__(self, out_dim_s3=320, out_dim_s4=512):
        super().__init__()
        self.conv1 = nn.Conv2d(2, 64, kernel_size=7, stride=4, padding=3)
        self.bn1 = nn.BatchNorm2d(64)
        self.act = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(64, 128, kernel_size=3, stride=2, padding=1)
        self.bn2 = nn.BatchNorm2d(128)
        self.conv3 = nn.Conv2d(128, out_dim_s3, kernel_size=3, stride=2, padding=1)
        self.bn3 = nn.BatchNorm2d(out_dim_s3)
        self.conv4 = nn.Conv2d(out_dim_s3, out_dim_s4, kernel_size=3, stride=2, padding=1)
        self.bn4 = nn.BatchNorm2d(out_dim_s4)


class MotionGuidedCrossAttention(_Holder):
    def __init__(self, dim, num_heads=8, attn_drop=0.0, proj_drop=0.0):
        super().__init__()
        if num_heads != 8:
            raise NotImplementedError("the fused cross-attention is built for 8 heads (mix_transformer_evp.py:863)")
        self.cross_attn = nn.MultiheadAttention(embed_dim=dim, num_heads=num_heads, dropout=attn_drop, batch_first=True)
        self.proj_drop = nn.Dropout(proj_drop)
        self.norm = nn.LayerNorm(dim)


class MixVisionTransformerEVP(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=14, embed_dims=[64, 128, 256, 512],
                 num_heads=[1, 2, 4, 8], mlp_ratios=[4, 4, 4, 4], qkv_bias=False, qk_scale=None, drop_rate=0.0,
                 attn_drop_rate=0.0, drop_path_rate=0.0, norm_layer=nn.LayerNorm, depths=[3, 4, 6, 3], sr_ratios=[8, 4, 2, 1], **kwargs):
        super().__init__()
        if in_chans != 3:
            raise NotImplementedError("in_chans must be 3")
        if len(set(mlp_ratios)) != 1:
            raise NotImplementedError("one mlp_ratio for all stages")
        eps = getattr(norm_layer(8), "eps", None)
        if eps is None or abs(eps - 1e-6) > 1e-12:
            raise NotImplementedError("block/stage LayerNorm eps must be 1e-6 (as every mit_bX_evp uses)")
        self.num_classes, self.depths, self.embed_dims = num_classes, list(depths), list(embed_dims)
        self.num_heads, self.sr_ratios, self.mlp_ratio = list(num_heads), list(sr_ratios), int(mlp_ratios[0])
        # `patch_size` is accepted and ignored exactly like the reference (:228-235)
        geom = [(img_size, 7, 4, in_chans), (img_size // 4, 3, 2, embed_dims[0]), (img_size // 8, 3, 2, embed_dims[1]),
                (img_size // 16, 3, 2, embed_dims[2])]
        for s, (sz, k, st, cin) in enumerate(geom):
            setattr(self, f"patch_embed{s + 1}", OverlapPatchEmbed(img_size=sz, patch_size=k, stride=st, in_chans=cin, embed_dim=embed_dims[s]))
        dpr = [x.item() for x in torch.linspace(0, drop_path_rate, sum(depths))]
        cur = 0
        for s in range(4):
            blocks = nn.ModuleList([
                Block(dim=embed_dims[s], num_heads=num_heads[s], mlp_ratio=mlp_ratios[s], qkv_bias=qkv_bias, qk_scale=qk_scale, drop=drop_rate,
                      attn_drop=attn_drop_rate, drop_path=dpr[cur + i], norm_layer=norm_layer, sr_ratio=sr_ratios[s]) for i in range(depths[s])])
            setattr(self, f"block{s + 1}", blocks)
            setattr(self, f"norm{s + 1}", norm_layer(embed_dims[s]))
            cur += depths[s]
        self.head = SegFormerHead(embed_dims, num_classes)
        self.apply(_ref_init)  # reference applies its init BEFORE creating the modules below (:275)
        self.scale_factor, self.prompt_type, self.tuning_stage, self.input_type = 4, "highpass", str(1234), "gaussian"
        self.freq_nums, self.handcrafted_tune, self.embedding_tune, self.adaptor = 0.25, True, True, "adaptor"
        self.prompt_generator = PromptGenerator(self.scale_factor, self.prompt_type, self.embed_dims, self.tuning_stage, self.depths,
                                                self.input_type, self.freq_nums, self.handcrafted_tune, self.embedding_tune, self.adaptor, img_size)
        self.flow_encoder = OpticalFlowEncoder(out_dim_s3=embed_dims[2], out_dim_s4=embed_dims[3])
        self.cross_attn_s3 = MotionGuidedCrossAttention(dim=embed_dims[2])
        self.cross_attn_s4 = MotionGuidedCrossAttention(dim=embed_dims[3])
        # ---- native state (not parameters, not in state_dict)
        self.embedding_dim = self.head.embedding_dim
        # frames per launch plan inside one forward call; 1159 frames x 196 stage-3 tokens = 11.99 full waves of 128-row GEMM tiles on
        # 148 SMs (800 = 8.28 waves wasted 8 % of the last one); 16 GB of workspace at 224x224
        self.micro_batch = int(os.environ.get("SURGVID_MICRO_BATCH", "1159"))
        self.fold_head = bool(int(os.environ.get("SURGVID_FOLD_HEAD", "0")))
        self._native = {}  # device index -> dict(handle, stamp, workspace)

    # ------------------------------------------------------------------ reference API surface
    def reset_drop_path(self, drop_path_rate):
        dpr = [x.item() for x in torch.linspace(0, drop_path_rate, sum(self.depths))]
        cur = 0
        for s in range(4):
            for i, blk in enumerate(getattr(self, f"block{s + 1}")):
                blk.drop_path_prob = dpr[cur + i]
            cur += self.depths[s]

    def freeze_patch_emb(self):
        self.patch_embed1.requires_grad = False

    @torch.jit.ignore
    def no_weight_decay(self):
        return {"pos_embed1", "pos_embed2", "pos_embed3", "pos_embed4", "cls_token"}

    def get_classifier(self):
        return self.head

    # ------------------------------------------------------------------ native plumbing
    def _apply(self, fn, *args, **kwargs):  # .to() / .cuda() / .float() ...
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1
        return super().load_state_dict(*args, **kwargs)

    def refresh_weights(self):
        """Call after modifying parameters in place (anything other than load_state_dict / .to()): forces a re-pack."""
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1

    def _cfg(self) -> _native.EvpCfg:
        cfg = _native.EvpCfg()
        for s in range(4):
            cfg.embed_dims[s], cfg.num_heads[s] = self.embed_dims[s], self.num_heads[s]
            cfg.depths[s], cfg.sr_ratios[s] = self.depths[s], self.sr_ratios[s]
        cfg.mlp_ratio, cfg.embedding_dim, cfg.fold_head = self.mlp_ratio, self.embedding_dim, int(self.fold_head)
        return cfg

    def attention_maps_layout(self, B: int, H: int, W: int):
        """Host only: ([n_blocks + 1] element offsets of each encoder block's [B, heads, N, N_kv] fp32 maps in one buffer, the last being
        the total, [(heads, N, N_kv)] per block), blocks in call order (sv_evp_attention_maps_layout)."""
        lib = _native.lib()
        cfg = self._cfg()
        nb = ctypes.c_int32(0)
        _native.check(lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), B, H, W, None, None, 0, ctypes.byref(nb)), "sv_evp_attention_maps_layout")
        off = (ctypes.c_int64 * (nb.value + 1))()
        dims = (ctypes.c_int32 * (3 * nb.value))()
        _native.check(lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), B, H, W, off, dims, nb.value, ctypes.byref(nb)),
                      "sv_evp_attention_maps_layout")
        return list(off), [tuple(dims[3 * i:3 * i + 3]) for i in range(nb.value)]

    def _state(self, device: torch.device):
        """Per-device native handle with packed weights; re-packed after load_state_dict / .to() / refresh_weights()."""
        idx = device.index if device.index is not None else torch.cuda.current_device()
        st = self._native.get(idx)
        stamp = (getattr(self, "_weights_epoch", 0), self.fold_head)
        if st is not None and st["stamp"] == stamp:
            return st
        lib = _native.lib()
        with torch.cuda.device(idx):
            if st is None:
                cfg = self._cfg()
                h = ctypes.c_void_p()
                _native.check(lib.sv_evp_create(ctypes.byref(cfg), ctypes.byref(h)), "sv_evp_create")
                st = {"handle": h, "workspace": {}, "fold_head": self.fold_head, "id": None}
                self._native[idx] = st
            elif st["fold_head"] != self.fold_head:
                raise RuntimeError("fold_head cannot change after the first forward on a device")
            for name, t in self.state_dict().items():
                a = np.ascontiguousarray(t.detach().to("cpu", torch.float32).numpy())
                shape = (ctypes.c_int64 * max(a.ndim, 1))(*a.shape)
                _native.check(lib.sv_evp_set_tensor(st["handle"], name.encode(), a.ctypes.data_as(ctypes.c_void_p), shape, a.ndim), "sv_evp_set_tensor")
            _native.check(lib.sv_evp_pack_weights(st["handle"]), "sv_evp_pack_weights")
        st["stamp"] = stamp
        if st["id"] is None:
            st["id"] = ops.register_handle(_EvpOpOwner(self, idx))
        return st

    def _native_forward(self, idx: int, x, seg, flow, micro_batch, maps=None):
        """maps: None, or an fp32 buffer of the layout's total element count (then the capture forward also fills it)."""
        st = self._native[idx]
        lib = _native.lib()
        B, _, H, W = x.shape
        mb = max(1, min(int(micro_batch), B))
        # one grow-only workspace per device and resolution: smaller batches reuse it, so the cached launch plans (keyed by
        # frame count and workspace address inside the handle) stay valid across calls with different B
        key = (H, W)
        nbytes = lib.sv_evp_workspace_bytes(st["handle"], mb, H, W)
        if nbytes == 0:
            raise RuntimeError("sv_evp_workspace_bytes failed: " + _native.last_error())
        ws = st["workspace"].get(key)
        if ws is None or ws.numel() < nbytes:
            ws = None
            st["workspace"].pop(key, None)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            st["workspace"][key] = ws
        out = torch.empty((B, self.embedding_dim), dtype=torch.float32, device=x.device)
        args = (ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(seg.data_ptr()), ctypes.c_void_p(0 if flow is None else flow.data_ptr()),
                ctypes.c_void_p(out.data_ptr()))
        tail = (B, H, W, mb, ctypes.c_void_p(ws.data_ptr()), ws.numel(), ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
        if maps is None:
            _native.check(lib.sv_evp_forward(st["handle"], *args, *tail), "sv_evp_forward")
        else:
            _native.check(lib.sv_evp_forward_attention(st["handle"], *args, ctypes.c_void_p(maps.data_ptr()), maps.numel(), *tail),
                          "sv_evp_forward_attention")
        return out

    def last_launch_count(self, device=None) -> int:
        idx = torch.cuda.current_device() if device is None else torch.device(device).index
        st = self._native.get(idx)
        return 0 if st is None else int(_native.lib().sv_evp_last_launch_count(st["handle"]))

    def read_tap(self, name: str, device=None) -> torch.Tensor:
        """Debug/parity tap of the last micro-batch, fp32 1-D (e.g. 'stage3_tokens', 'fused4_tokens')."""
        idx = torch.cuda.current_device() if device is None else torch.device(device).index
        st = self._native[idx]
        lib = _native.lib()
        n = ctypes.c_int64(0)
        probe = torch.empty(1, dtype=torch.float32, device=f"cuda:{idx}")
        lib.sv_evp_read_tap(st["handle"], name.encode(), ctypes.c_void_p(probe.data_ptr()), 0, ctypes.byref(n), None)
        if n.value <= 0:
            raise RuntimeError("read_tap: " + _native.last_error())
        out = torch.empty(n.value, dtype=torch.float32, device=f"cuda:{idx}")
        rc = lib.sv_evp_read_tap(st["handle"], name.encode(), ctypes.c_void_p(out.data_ptr()), n.value, ctypes.byref(n),
                                 ctypes.c_void_p(torch.cuda.current_stream(out.device).cuda_stream))
        _native.check(rc, "sv_evp_read_tap")
        return out

    # ------------------------------------------------------------------ forward
    def forward_features(self, x, y):
        raise RuntimeError("forward_features is fused into torch.ops.surgvid.evp_lfb_forward; per-stage tensors are available "
                           "through model.read_tap('stage{1..4}_tokens') after a forward")

    def _inputs(self, x, y, flow):
        if self.training:
            raise RuntimeError("surgvid_b200 models are inference-only: call model.eval() first (generate_evp_LFB.py:437)")
        if not x.is_cuda:
            raise RuntimeError("surgvid_b200 has no CPU path: move the model inputs to a CUDA (sm_100a) device")
        H, W = x.shape[-2], x.shape[-1]
        x = x.reshape(-1, 3, H, W).to(torch.float32).contiguous()
        y = y.reshape(-1, 3, H, W).to(device=x.device, dtype=torch.float32).contiguous()
        if flow is not None:
            flow = flow.reshape(-1, 2, H, W).to(device=x.device, dtype=torch.float32).contiguous()
        return x, y, flow

    def extract_features(self, x, y, flow=None) -> torch.Tensor:
        x, y, flow = self._inputs(x, y, flow)
        st = self._state(x.device)
        return torch.ops.surgvid.evp_lfb_forward(x, y, flow, st["id"], self.micro_batch)

    def attention_maps(self, x, y, flow=None):
        """-> (features [B, E] as `extract_features`, maps): maps is a list of sum(depths) fp32 CUDA tensors [B, heads, N, N_kv], the
        post-softmax attention of each encoder block in call order (stage 1's blocks first), views into one buffer.  The features are
        bit-identical to `extract_features` on the same inputs.  Flow cross-attention maps are not captured."""
        x, y, flow = self._inputs(x, y, flow)
        B, _, H, W = x.shape
        off, dims = self.attention_maps_layout(B, H, W)
        buf = torch.empty(off[-1], dtype=torch.float32, device=x.device)
        self._state(x.device)
        idx = x.device.index if x.device.index is not None else torch.cuda.current_device()
        feats = self._native_forward(idx, x, y, flow, self.micro_batch, maps=buf)
        maps = [buf[off[i]:off[i + 1]].view(B, *dims[i]) for i in range(len(dims))]
        return feats, maps

    def forward(self, x, y, flow=None, return_features=False):
        caches = visualizer.active_caches()
        if caches:  # visualizer.get_local.activate(): record what the reference's decorated Attention.forward would
            feats, maps = self.attention_maps(x, y, flow)
            arrays = [m.cpu().numpy() for m in maps]
            for cache in caches:
                cache.setdefault(visualizer.QUALNAME, []).extend(arrays)
        else:
            feats = self.extract_features(x, y, flow)
        if return_features:
            return feats
        return self.head.classify(self, feats)

    def __del__(self):
        try:
            for st in self._native.values():
                if st.get("id") is not None:
                    ops.unregister_handle(st["id"])
                _native.lib().sv_evp_destroy(st["handle"])
        except (AttributeError, TypeError, ImportError):
            pass  # interpreter shutdown: module globals are already gone; anything else (a failing destroy) propagates as "ignored exception" text


class _EvpOpOwner:
    """What the custom op sees behind its integer handle (one per model x device)."""

    def __init__(self, model: MixVisionTransformerEVP, idx: int):
        import weakref

        self._model = weakref.ref(model)
        self._idx = idx
        self.embedding_dim = model.embedding_dim

    def _native_forward(self, x, seg, flow, micro_batch):
        return self._model()._native_forward(self._idx, x, seg, flow, micro_batch)


# (embed_dims, depths) of the six published variants (mix_transformer_evp.py:894-943); everything else is shared:
# heads [1,2,5,8], mlp_ratio 4, qkv_bias, LayerNorm eps 1e-6, sr_ratios [8,4,2,1], drop_path_rate 0.1, patch_size ignored.
_VARIANTS = {
    "mit_b0_evp": ([32, 64, 160, 256], [2, 2, 2, 2]),
    "mit_b1_evp": ([64, 128, 320, 512], [2, 2, 2, 2]),
    "mit_b2_evp": ([64, 128, 320, 512], [3, 4, 6, 3]),
    "mit_b3_evp": ([64, 128, 320, 512], [3, 4, 18, 3]),
    "mit_b4_evp": ([64, 128, 320, 512], [3, 8, 27, 3]),
    "mit_b5_evp": ([64, 128, 320, 512], [3, 6, 40, 3]),
}


def _make_variant(name, dims, depths):
    def __init__(self, **kwargs):
        MixVisionTransformerEVP.__init__(self, patch_size=4, embed_dims=list(dims), num_heads=[1, 2, 5, 8], mlp_ratios=[4, 4, 4, 4],
                                         qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), depths=list(depths),
                                         sr_ratios=[8, 4, 2, 1], drop_rate=0.0, drop_path_rate=0.1, **kwargs)

    return type(name, (MixVisionTransformerEVP,), {"__init__": __init__, "__module__": __name__,
                                                   "__doc__": f"{name}(): embed_dims {dims}, depths {depths}"})


for _n, (_d, _dp) in _VARIANTS.items():
    globals()[_n] = _make_variant(_n, _d, _dp)
del _n, _d, _dp
