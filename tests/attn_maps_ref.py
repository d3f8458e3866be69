"""Reference attention maps of the EVP encoder: the oracle's forward_features (oracle/evp_oracle.py) with each block's post-softmax
`attn` (Attention.forward, mix_transformer_evp.py:123-125) recorded, in call order.  It is built from the oracle's own functions;
only `attention` is restated here, with the recording added, so the oracle itself stays as it is.  tests/test_attention_maps_cpu.py
checks that the stage tokens this produces are bit-identical to the oracle's."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle import evp_oracle as E


def _attention(cx, sd, p, x, H, W, heads, sr, maps):
    """evp_oracle.attention, plus maps.append(attn) after the softmax."""
    B, N, C = x.shape
    hd = C // heads
    q = E._linear(cx, sd, p + ".q", x).reshape(B, N, heads, hd).permute(0, 2, 1, 3)
    if sr > 1:
        x_ = x.permute(0, 2, 1).reshape(B, C, H, W)
        x_ = F.conv2d(cx.r(x_), cx.r(sd[p + ".sr.weight"]), sd[p + ".sr.bias"], stride=sr)
        x_ = x_.reshape(B, C, -1).permute(0, 2, 1)
        x_ = E._ln(sd, p + ".norm", x_, 1e-5)
    else:
        x_ = x
    kv = E._linear(cx, sd, p + ".kv", x_).reshape(B, -1, 2, heads, hd).permute(2, 0, 3, 1, 4)
    k, v = kv[0], kv[1]
    attn = (cx.r(q) @ cx.r(k).transpose(-2, -1)) * (hd ** -0.5)
    attn = attn.softmax(dim=-1)
    maps.append(attn)
    o = (cx.r(attn) @ cx.r(v)).transpose(1, 2).reshape(B, N, C)
    return E._linear(cx, sd, p + ".proj", o)


@torch.no_grad()
def encoder_maps(sd, cfg, x, seg, emulate_bf16=False):
    """-> (maps: list of sum(depths) [B, heads, N, N_kv] fp32 tensors, taps: {'stage{s}_tokens': [B, N, C]}) for frames x, seg
    [B, 3, H, W], following evp_oracle.forward_features step for step."""
    cx = E._Ctx(emulate_bf16)
    H0, W0 = x.shape[-2], x.shape[-1]
    x = x.reshape(-1, 3, H0, W0).float()
    seg = seg.reshape(-1, 3, H0, W0).float()
    dims, heads, depths, srs = cfg["embed_dims"], cfg["num_heads"], cfg["depths"], cfg["sr_ratios"]
    B = x.shape[0]
    hc = E.handcrafted_prompts(cx, sd, seg)
    ks, st = [7, 3, 3, 3], [4, 2, 2, 2]
    maps, taps = [], {}
    for s in range(4):
        x, H, W = E.overlap_patch_embed(cx, sd, f"patch_embed{s + 1}", x, ks[s], st[s])
        psum = hc[s] + E._linear(cx, sd, f"prompt_generator.embedding_generator{s + 1}", x)
        for i in range(depths[s]):
            x = E.adapter(cx, sd, x, psum, s + 1, i)
            p = f"block{s + 1}.{i}"
            x = x + _attention(cx, sd, p + ".attn", E._ln(sd, p + ".norm1", x, 1e-6), H, W, heads[s], srs[s], maps)
            x = x + E.mix_ffn(cx, sd, p + ".mlp", E._ln(sd, p + ".norm2", x, 1e-6), H, W)
        x = E._ln(sd, f"norm{s + 1}", x, 1e-6)
        taps[f"stage{s + 1}_tokens"] = x
        x = x.reshape(B, H, W, -1).permute(0, 3, 1, 2).contiguous()
    return maps, taps
