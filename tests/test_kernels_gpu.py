"""Per-kernel parity (GPU): each hand-written sm_100a kernel, called through the C ABI, against a plain PyTorch fp32
reference of the same op on the same seeded inputs.  bf16-in / fp32-accumulate kernels are compared against fp32 math on
the bf16-rounded operands, so the tolerance only has to cover accumulation order and the final bf16 rounding."""
import math

import pytest
import torch
import torch.nn.functional as F

import attn_ref
import gemm_ref
import surgvid_b200  # noqa: F401
from surgvid_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand(shape, seed, scale=1.0, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(DEV).to(dtype)


GEMM_SHAPES = [
    # (M, N, K)   — shapes the model really launches, plus ragged edges
    (128, 64, 64), (256, 128, 64), (200, 64, 64), (3136 * 2, 64, 64), (3136 * 2, 256, 64), (3136, 64, 256),
    (784 * 2, 128, 128), (784 * 2, 512, 128), (784, 128, 512), (98, 128, 2048), (98, 256, 128),
    (196 * 3, 320, 320), (196 * 3, 1280, 320), (196 * 3, 320, 1280), (147, 320, 1280), (147, 640, 320),
    (49 * 4, 512, 512), (49 * 4, 2048, 512), (49 * 4, 512, 2048), (49 * 4, 1024, 512),
    (3136, 16, 152), (3136, 16, 16), (3136, 64, 16), (784, 32, 144), (784, 32, 32), (196, 80, 288), (196, 80, 80),
    (196, 320, 80), (49, 128, 720), (49, 128, 128), (49, 512, 128), (3136, 64, 104), (98, 64, 4096), (98, 2048, 8192),
    (98, 2048, 1024), (1, 16, 8), (129, 24, 72), (300, 40, 24), (5000, 2048, 64),
]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_gemm_plain(M, N, K):
    a = _rand((M, K), 1, dtype=torch.bfloat16)
    w = _rand((N, K), 2, 1.0 / math.sqrt(K), dtype=torch.bfloat16)
    out = ops.gemm_bf16(a, w, out_dtype=torch.float32)
    ref, mag = gemm_ref.reference(a, w, None, 0, None)
    gemm_ref.assert_gate(out, ref, mag, 0, True, f"{M}x{N}x{K}")


@pytest.mark.parametrize("act", [0, 1, 2])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_gemm_epilogues(act, out_dtype):
    M, N, K = 1000, 320, 200
    a = _rand((M, K), 3, dtype=torch.bfloat16)
    w = _rand((N, K), 4, 1.0 / math.sqrt(K), dtype=torch.bfloat16)
    bias = _rand((N,), 5, 0.5)
    resid = _rand((M, N), 6)
    out = ops.gemm_bf16(a, w, bias=bias, act=act, residual=resid, out_dtype=out_dtype)
    ref, mag = gemm_ref.reference(a, w, bias, act, resid)
    gemm_ref.assert_gate(out, ref, mag, act, out_dtype == torch.float32, f"act {act} {out_dtype}")


def test_gemm_residual_in_place_and_strided_output():
    M, N, K = 777, 64, 256
    a = _rand((M, K), 7, dtype=torch.bfloat16)
    w = _rand((N, K), 8, 1.0 / math.sqrt(K), dtype=torch.bfloat16)
    x = _rand((M, N), 9)
    ref, mag = gemm_ref.reference(a, w, None, 0, x)
    ops.gemm_bf16(a, w, residual=x, out=x)  # x += a @ w.T  (residual aliases out)
    gemm_ref.assert_gate(x, ref, mag, 0, True, "in place")
    # write into a column slice of a wider matrix (head concat buffer) and read A / W with padded row strides
    big = torch.zeros((M, 4 * N), dtype=torch.bfloat16, device=DEV)
    a_pad = torch.zeros((M, K + 24), dtype=torch.bfloat16, device=DEV)
    a_pad[:, :K] = a
    w_pad = torch.zeros((N, K + 8), dtype=torch.bfloat16, device=DEV)
    w_pad[:, :K] = w
    ops.gemm_bf16(a_pad[:, :K], w_pad[:, :K], out=big[:, 2 * N:3 * N])
    ref, mag = gemm_ref.reference(a, w, None, 0, None)
    gemm_ref.assert_gate(big[:, 2 * N:3 * N], ref, mag, 0, False, "strided bf16 output")
    assert big[:, :2 * N].abs().max().item() == 0 and big[:, 3 * N:].abs().max().item() == 0


def test_gemm_many_tiles_reuses_pipeline_state():
    """Enough tiles that every CTA loops several times through the smem ring and both TMEM accumulators."""
    M, N, K = 148 * 128 * 3 + 77, 256, 192
    a = _rand((M, K), 10, dtype=torch.bfloat16)
    w = _rand((N, K), 11, 1.0 / math.sqrt(K), dtype=torch.bfloat16)
    out = ops.gemm_bf16(a, w, out_dtype=torch.float32)
    ref, mag = gemm_ref.reference(a, w, None, 0, None)
    gemm_ref.assert_gate(out, ref, mag, 0, True, "many tiles")


@pytest.mark.parametrize("C", [16, 32, 64, 80, 128, 320, 512])
@pytest.mark.parametrize("eps", [1e-5, 1e-6])
def test_layernorm(C, eps):
    rows = 1237
    x = _rand((rows, C), 20, 3.0) + 0.7
    g, b = _rand((C,), 21) * 0.2 + 1.0, _rand((C,), 22, 0.3)
    of, ob = ops.layernorm(x, g, b, eps, want_f32=True, want_bf16=True)
    torch.cuda.synchronize()
    ref = F.layer_norm(x, (C,), g, b, eps)
    assert (of - ref).abs().max().item() < 2e-5
    assert (ob.float() - ref).abs().max().item() < 2e-2


@pytest.mark.parametrize("cfg", [(3, 7, 4, 3, 56, 60), (2, 7, 4, 3, 64, 48), (16, 3, 2, 1, 28, 30), (64, 3, 2, 1, 14, 14),
                                 (64, 8, 8, 0, 56, 56), (128, 4, 4, 0, 30, 27), (320, 2, 2, 0, 7, 9)])
def test_im2col(cfg):
    Cin, k, stride, pad, H, W = cfg
    B = 3
    x = _rand((B, Cin, H, W), 30)
    if Cin % 8 == 0:
        src = x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)  # NHWC bf16
        xr = src.float().permute(0, 3, 1, 2)
    else:
        src, xr = x, x.to(torch.bfloat16).float()
    out = ops.im2col(src, k, stride, pad)
    torch.cuda.synchronize()
    cols = F.unfold(xr, k, padding=pad, stride=stride)          # [B, Cin*k*k, L], index (cin, kh, kw)
    L = cols.shape[-1]
    ref = cols.view(B, Cin, k * k, L).permute(0, 3, 2, 1).reshape(B * L, k * k * Cin)  # -> (kh,kw,cin)
    K = k * k * Cin
    assert torch.equal(out[:, :K].float(), ref)
    assert out[:, K:].abs().max().item() == 0 if out.shape[1] > K else True


@pytest.mark.parametrize("shape", [(2, 56, 56, 256), (3, 28, 28, 512), (2, 14, 14, 1280), (5, 7, 7, 2048), (1, 15, 27, 64), (2, 9, 5, 8)])
def test_dwconv3x3_gelu(shape):
    B, H, W, C = shape
    x = _rand(shape, 40, dtype=torch.bfloat16)
    w = _rand((C, 1, 3, 3), 41, 0.4)
    bias = _rand((C,), 42, 0.2)
    out = ops.dwconv3x3_gelu(x, w.view(C, 9).t().contiguous(), bias)
    torch.cuda.synchronize()
    ref = F.gelu(F.conv2d(x.float().permute(0, 3, 1, 2), w, bias, padding=1, groups=C)).permute(0, 2, 3, 1)
    assert (out.float() - ref).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("cfg", [(3, 1, 3136, 49, 64), (2, 2, 784, 49, 64), (2, 5, 196, 49, 64), (3, 8, 49, 49, 64), (2, 8, 196, 196, 40),
                                 (1, 1, 1000, 390, 64), (2, 8, 405, 405, 64), (2, 5, 160, 70, 32), (1, 2, 5, 3, 64),
                                 (2, 8, 196, 196, 20), (3, 8, 49, 49, 20), (1, 8, 300, 330, 20),   # head_dim 20: mit_b0_evp flow cross-attention
                                 # tcgen05 path (head_dim 64, N_kv <= 448): several query tiles per CTA, exact / ragged tile edges, 1..7 key tiles
                                 (40, 1, 3136, 49, 64), (3, 2, 128, 64, 64), (3, 2, 129, 65, 64), (2, 3, 300, 128, 64), (2, 2, 257, 448, 64),
                                 (1, 2, 700, 200, 64), (2, 1, 1620, 405, 64), (1, 2, 64, 449, 64)])
def test_attention(cfg):
    B, heads, Nq, Nkv, hd = cfg
    C = heads * hd
    q = _rand((B * Nq, C), 50, dtype=torch.bfloat16)
    kv = _rand((B * Nkv, 2 * C), 51, dtype=torch.bfloat16)
    scale = hd ** -0.5
    o = ops.attention(q, kv[:, :C], kv[:, C:], B, heads, hd, scale)
    ref = attn_ref.reference(q, kv[:, :C], kv[:, C:], B, heads, hd, scale)
    attn_ref.assert_gate(o, ref, heads, hd, Nq, str(cfg))


def test_gauss5x5():
    x = _rand((2, 3, 37, 41), 60)
    out = ops.gauss5x5(x)
    torch.cuda.synchronize()
    k1 = torch.tensor([1.0, 4.0, 6.0, 4.0, 1.0], device=DEV)
    k = (k1[:, None] * k1[None, :] / 256.0).expand(3, 1, 5, 5).contiguous()
    ref = F.conv2d(F.pad(x, (2, 2, 2, 2), mode="reflect"), k, groups=3)
    assert (out - ref).abs().max().item() < 1e-5


@pytest.mark.parametrize("cfg", [(56, 56, 7, 7, 64), (28, 28, 7, 7, 128), (14, 14, 7, 7, 320), (120, 214, 15, 27, 64), (30, 54, 15, 27, 320)])
def test_bilinear_tokens(cfg):
    H, W, Ho, Wo, C = cfg
    x = _rand((2, H, W, C), 70, dtype=torch.bfloat16)
    out = ops.bilinear_tokens(x, Ho, Wo)
    torch.cuda.synchronize()
    ref = F.interpolate(x.float().permute(0, 3, 1, 2), size=(Ho, Wo), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    assert (out.float() - ref).abs().max().item() < 3e-2


def test_token_mean():
    x = _rand((5 * 49, 2048), 80)
    out = ops.token_mean(x, 49)
    torch.cuda.synchronize()
    assert (out - x.view(5, 49, 2048).mean(1)).abs().max().item() < 1e-5


@pytest.mark.parametrize("cfg", [(3, 64, 224, 224, False), (3, 16, 224, 224, False), (2, 64, 224, 224, True), (3, 64, 100, 76, False), (2, 32, 61, 37, True)])
def test_stem_conv(cfg):
    Cin, Cout, H, W, relu = cfg
    B = 3
    x = _rand((B, Cin, H, W), 90)
    w = _rand((Cout, Cin, 7, 7), 91, 1.0 / math.sqrt(49 * Cin))
    bias = _rand((Cout,), 92, 0.3)
    g, b = _rand((Cout,), 93) * 0.2 + 1.0, _rand((Cout,), 94, 0.3)
    of, ob = ops.stem_conv(x, w, bias, None if relu else g, None if relu else b, 1e-5, relu)
    torch.cuda.synchronize()
    y = F.conv2d(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), bias, stride=4, padding=3)   # bf16 operands, fp32 accumulate
    y = y.flatten(2).transpose(1, 2)
    ref = (F.relu(y) if relu else F.layer_norm(y, (Cout,), g, b, 1e-5)).reshape(-1, Cout)
    assert (of - ref).abs().max().item() < 2e-3 * max(1.0, ref.abs().max().item())
    assert (ob.float() - ref).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("M,N,K", [(256, 64, 64), (129, 24, 72), (1000, 320, 1280), (39200, 320, 1360), (5000, 1280, 320), (777, 512, 2048), (148 * 256 * 2 + 300, 256, 192)])
def test_gemm_cta_pair_mode(M, N, K, monkeypatch):
    """tcgen05 cta_group::2 path (2-CTA clusters, 256-row tiles) forced on; must agree with the single-CTA path bit for bit."""
    a = _rand((M, K), 101, dtype=torch.bfloat16)
    w = _rand((N, K), 102, 1.0 / math.sqrt(K), dtype=torch.bfloat16)
    bias = _rand((N,), 103, 0.5)
    resid = _rand((M, N), 104)
    monkeypatch.setenv("SURGVID_GEMM_PAIR", "0")
    single = ops.gemm_bf16(a, w, bias=bias, residual=resid, out_dtype=torch.float32)
    monkeypatch.setenv("SURGVID_GEMM_PAIR", "1")
    pair = ops.gemm_bf16(a, w, bias=bias, residual=resid, out_dtype=torch.float32)
    pair_bf16 = ops.gemm_bf16(a, w, bias=bias, act=1)
    ref, mag = gemm_ref.reference(a, w, bias, 0, resid)
    gemm_ref.assert_gate(pair, ref, mag, 0, True, "pair, fp32 + residual")
    assert torch.equal(pair, single)
    ref2, mag2 = gemm_ref.reference(a, w, bias, 1, None)
    gemm_ref.assert_gate(pair_bf16, ref2, mag2, 1, False, "pair, bf16 GELU")


@pytest.mark.parametrize("M,N,K1,K2", [(39200, 320, 1280, 80), (1000, 128, 512, 32), (70000, 64, 256, 16)])
def test_gemm_cat_cta_pair_mode(M, N, K1, K2, monkeypatch):
    """The fc2 form the model launches in CTA-pair mode: A given as two K segments, fp32 result accumulated IN PLACE into the residual
    stream.  Pair mode (forced on, and as the plan selects it by itself) must agree with single-CTA tiles bit for bit."""
    a = _rand((M, K1), 111, dtype=torch.bfloat16)
    a2 = _rand((M, K2), 112, dtype=torch.bfloat16)
    w = _rand((N, K1 + K2), 113, 1.0 / math.sqrt(K1 + K2), dtype=torch.bfloat16)
    bias = _rand((N,), 114, 0.5)
    x0 = _rand((M, N), 115)
    outs = {}
    for mode in ("0", "1", None):
        if mode is None:
            monkeypatch.delenv("SURGVID_GEMM_PAIR", raising=False)
        else:
            monkeypatch.setenv("SURGVID_GEMM_PAIR", mode)
        x = x0.clone()
        ops.gemm_bf16_cat(a, a2, w, bias=bias, residual=x, out=x)
        outs[mode] = x
    ref, mag = gemm_ref.reference(a, w, bias, 0, x0, a2)
    gemm_ref.assert_gate(outs["1"], ref, mag, 0, True, "pair, two segments, in place")
    assert torch.equal(outs["1"], outs["0"]) and torch.equal(outs[None], outs["0"])


@pytest.mark.parametrize("cfg", [
    # (frames, H, W, hidden, N, tail_cols): the three fusable stages of mit_b3_evp at 224^2, a no-tail case, ragged row tiles,
    # and enough frames that every CTA of the persistent grid walks several tiles
    (3, 14, 14, 1280, 320, 80), (2, 56, 56, 256, 64, 16), (2, 28, 28, 512, 128, 32), (2, 14, 14, 1280, 320, 0),
    (2, 11, 12, 128, 64, 0), (1, 9, 14, 64, 32, 8), (200, 14, 14, 1280, 320, 80), (3, 30, 54, 1280, 320, 80)])
def test_mixffn_fc2_fused(cfg):
    """x += bias + GELU(dwconv3x3(h1) + b_dw) @ W[:, :hidden].T + tail @ W[:, hidden:].T as one kernel (mixffn.cu) against the same math
    in fp32 on the bf16-rounded operands (the hidden tensor is rounded to bf16 before the GEMM, exactly as the unfused path stores it)."""
    B, H, W, hid, N, tc = cfg
    h1 = _rand((B, H, W, hid), 70, dtype=torch.bfloat16)
    w = _rand((hid, 1, 3, 3), 71, 0.4)
    bdw = _rand((hid,), 72, 0.2)
    wcat = _rand((N, hid + tc), 73, 1.0 / math.sqrt(hid), dtype=torch.bfloat16)
    bias = _rand((N,), 74, 0.3)
    tail = _rand((B * H * W, tc), 75, dtype=torch.bfloat16) if tc else None
    x0 = _rand((B * H * W, N), 76)
    x = x0.clone()
    ops.mixffn_fc2(h1, w.view(hid, 9).t().contiguous(), bdw, wcat, bias, x, tail)
    torch.cuda.synchronize()
    h2 = F.gelu(F.conv2d(h1.float().permute(0, 3, 1, 2), w, bdw, padding=1, groups=hid)).permute(0, 2, 3, 1).reshape(B * H * W, hid)
    ref = x0 + bias + h2.bfloat16().float() @ wcat[:, :hid].float().t()
    if tc:
        ref = ref + tail.float() @ wcat[:, hid:].float().t()
    err = (x - ref).abs().max().item()
    assert err < 2e-2 * max(1.0, ref.abs().max().item()), err
    # and against the stand-alone kernels (DWConv+GELU kernel -> tcgen05 GEMM with fp32 residual)
    h2k = ops.dwconv3x3_gelu(h1, w.view(hid, 9).t().contiguous(), bdw).reshape(B * H * W, hid)
    a = torch.cat([h2k, tail], 1).contiguous() if tc else h2k
    unf = ops.gemm_bf16(a, wcat, bias, residual=x0, out_dtype=torch.float32)
    assert (x - unf).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("M,N,K1,K2,strided", [(300, 64, 256, 16, False), (1000, 320, 1280, 80, True), (129, 128, 512, 32, True), (5000, 320, 64, 8, False)])
def test_gemm_two_segment_a_operand(M, N, K1, K2, strided):
    """[A | A2] @ W^T with the two K segments read from different buffers == the GEMM on the materialised concatenation (bit-identical:
    same tiles, same accumulation order), in the residual fp32 form the model uses for fc2 + adapter."""
    a = _rand((M, K1), 80, dtype=torch.bfloat16)
    big = _rand((M, 3 * K2 + 8), 81, dtype=torch.bfloat16)       # a2 is a column slice of a wider tensor (row stride > K2), like T_all
    a2 = big[:, K2:2 * K2] if strided else big[:, :K2].contiguous()
    w = _rand((N, K1 + K2), 82, 1.0 / math.sqrt(K1 + K2), dtype=torch.bfloat16)
    bias = _rand((N,), 83, 0.2)
    x0 = _rand((M, N), 84)
    got = ops.gemm_bf16_cat(a, a2, w, bias, residual=x0, out_dtype=torch.float32)
    want = ops.gemm_bf16(torch.cat([a, a2], 1).contiguous(), w, bias, residual=x0, out_dtype=torch.float32)
    assert torch.equal(got, want)
    ref, mag = gemm_ref.reference(a, w, bias, 0, x0, a2)
    gemm_ref.assert_gate(got, ref, mag, 0, True, "two segments")
