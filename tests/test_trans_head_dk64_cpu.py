"""Trans-SVNet head at d_k = d_v = 64 (mstcn_f_maps 64, adapter_transformer.py:315) without a device: the oracle's generic-d_k path
against an independent float64 formulation, the state_dict of `Transformer(64, ...)`, and the configurations `sv_trans_create` rejects."""
import ctypes

import pytest
import torch

import surgvid_b200  # noqa: F401
from oracle import trans_head_oracle as tho
from surgvid_b200 import _native
from surgvid_b200.trans_head import Transformer, Transformer2_3_1

SV_ERR_UNSUPPORTED = 4


def _random_inner(d_k, d_ff, bias, seed):
    m = Transformer2_3_1(d_model=14, d_ff=d_ff, d_k=d_k, d_v=d_k, n_layers=1, n_heads=4, len_q=30, bias=bias)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("layer_norm.weight"):
                p.copy_(1.0 + 0.2 * torch.randn(p.shape, generator=g))
            elif n.endswith("bias"):
                p.copy_(0.3 * torch.randn(p.shape, generator=g))
            else:
                p.copy_(torch.randn(p.shape, generator=g) * (1.5 / p.shape[1] ** 0.5))
    return m


def _einsum_forward(sd, enc, dec, n_heads, d_k):
    """Float64, written without the oracle's helpers: explicit per-head einsums, LayerNorm from its definition."""
    def lin(p, x):
        y = torch.einsum("...i,oi->...o", x, sd[p + ".weight"])
        return y + sd[p + ".bias"] if p + ".bias" in sd else y

    def norm(p, x):
        mu = x.mean(-1, keepdim=True)
        var = ((x - mu) ** 2).mean(-1, keepdim=True)
        return (x - mu) / torch.sqrt(var + 1e-5) * sd[p + ".weight"] + sd[p + ".bias"]

    def attn(p, xq, xkv):
        q = lin(p + ".W_Q", xq).unflatten(-1, (n_heads, d_k))          # [T, Lq, H, d]
        k = lin(p + ".W_K", xkv).unflatten(-1, (n_heads, d_k))         # [T, Lk, H, d]
        v = lin(p + ".W_V", xkv).unflatten(-1, (n_heads, d_k))
        s = torch.einsum("tqhd,tkhd->thqk", q, k) / d_k ** 0.5
        w = torch.exp(s - s.amax(-1, keepdim=True))
        w = w / w.sum(-1, keepdim=True)
        ctx = torch.einsum("thqk,tkhd->tqhd", w, v).flatten(-2)
        return norm(p + ".layer_norm", lin(p + ".fc", ctx) + xq)

    def ffn(p, x):
        return norm(p + ".layer_norm", lin(p + ".fc2", torch.clamp(lin(p + ".fc1", x), min=0.0)) + x)

    e = ffn("encoder.layers.0.pos_ffn", attn("encoder.layers.0.enc_self_attn", enc, enc))
    return ffn("decoder.layers.0.pos_ffn", attn("decoder.layers.0.dec_enc_attn", dec, e))


@pytest.mark.parametrize("d_k,d_ff,bias", [(64, 64, True), (64, 64, False), (64, 32, True), (32, 32, True)])
def test_oracle_generic_dk_matches_einsum_float64(d_k, d_ff, bias):
    m = _random_inner(d_k, d_ff, bias, seed=7 + d_k + d_ff)
    sd = {k: v.detach().to(torch.float64) for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(d_k)
    T = 45
    logits = 3.0 * torch.randn(1, 14, T, generator=g, dtype=torch.float64)
    inputs, _ = tho.original_forward_inputs(logits, torch.zeros(1, T, 8, dtype=torch.float64), torch.zeros(14, 8, dtype=torch.float64), 30)
    query = torch.tanh(torch.randn(T, 1, 14, generator=g, dtype=torch.float64))
    got = tho.transformer2_3_1_forward(sd, inputs, query, 4, d_k, d_k)
    want = _einsum_forward(sd, inputs, query, 4, d_k)
    assert got.shape == (T, 1, 14)
    err = float((got - want).abs().max())
    assert err <= 1e-12, err
    # d_k enters the arithmetic (head split and 1/sqrt(d_k)), so the d_k = 64 weights read as d_k = 32 heads give another result
    if d_k == 64:
        assert float((tho.transformer2_3_1_forward(sd, inputs, query, 8, 32, 32) - want).abs().max()) > 1e-3


def test_transformer_f_maps_64_state_dict():
    head = Transformer(64, 2048, 14, 30)
    sd = head.state_dict()
    assert head.transformer.d_k == 64 and head.transformer.d_v == 64 and head.transformer.d_ff == 64 and head.transformer.len_q == 30
    assert sd["fc.weight"].shape == (14, 2048)
    for blk in ("transformer.encoder.layers.0.enc_self_attn", "transformer.decoder.layers.0.dec_enc_attn"):
        for p in ("W_Q", "W_K", "W_V"):
            assert sd[f"{blk}.{p}.weight"].shape == (256, 14) and sd[f"{blk}.{p}.bias"].shape == (256,)
        assert sd[f"{blk}.fc.weight"].shape == (14, 256)
        assert sd[f"{blk}.layer_norm.weight"].shape == (14,)
    for blk in ("transformer.encoder.layers.0.pos_ffn", "transformer.decoder.layers.0.pos_ffn"):
        assert sd[f"{blk}.fc1.weight"].shape == (64, 14) and sd[f"{blk}.fc2.weight"].shape == (14, 64)
    # mstcn_f_maps above 64 keeps d_k = 64 (min(64, f_maps)) and d_ff = f_maps
    assert Transformer(128, 2048, 14, 30).transformer.d_k == 64


@pytest.mark.parametrize("d_k,d_v,n_heads", [(48, 48, 4), (64, 32, 4), (32, 64, 4), (64, 64, 8), (128, 128, 4), (16, 16, 4)])
def test_create_rejects_unsupported_without_device(d_k, d_v, n_heads):
    lib = _native.lib()
    cfg = _native.TransCfg(14, 64, d_k, d_v, 1, n_heads, 30)
    h = ctypes.c_void_p()
    assert lib.sv_trans_create(ctypes.byref(cfg), ctypes.byref(h)) == SV_ERR_UNSUPPORTED
    assert b"d_k = d_v = 32 or 64" in lib.sv_last_error()
