"""Implicit-GEMM convolutions on the B200: `sv_op_conv_gemm_bf16` (A tiles gathered by im2col-mode TMA from the NHWC input) is
bit-identical to `sv_op_im2col` + `sv_op_gemm_bf16` over the same weights — the MMAs see the same bf16 tiles in the same k order —
at every geometry the model runs and at ragged ones (odd H / W, M ending mid-tile and mid-frame, 128-row tiles spanning frame
boundaries, where the padding of one frame must not read the next), single-CTA and CTA-pair plans, every epilogue form, with NaN
around the input and NaN output margins that must keep their bits.  And mit_b3_evp with flow runs its patch-embed, flow and sr convs
without an im2col buffer: 6 gathers fewer per micro-batch, and a smaller workspace."""
import ctypes

import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native, ops

pytestmark = pytest.mark.gpu

ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
# (C, k, stride, pad, N): the model's convs (patch embed 2-4 / flow 2-4: k3 s2 p1; sr: k = s = 8 / 4 / 2, p 0) and one more width
GEOMS = [(64, 3, 2, 1, 128), (128, 3, 2, 1, 320), (320, 3, 2, 1, 512), (512, 3, 2, 1, 64), (64, 8, 8, 0, 64), (128, 4, 4, 0, 128),
         (320, 2, 2, 0, 320), (512, 2, 2, 0, 96)]
# (B, H, W): even and odd sizes; M = B*Ho*Wo is never a multiple of 128 here, so tiles straddle frames and the last one ends mid-frame
SIZES = [(3, 28, 28), (2, 31, 45), (5, 17, 23)]
# (out_fp32, residual, act): fp32 result (patch embed, sr), bf16 + ReLU (flow), fp32 + residual, bf16 + GELU
FORMS = [(True, False, ACT_NONE), (False, False, ACT_RELU), (True, True, ACT_NONE), (False, False, ACT_GELU)]


def _padded(shape, dtype, fill, dev, front=24, back=40):
    """A contiguous tensor of `shape` inside a larger buffer filled with `fill` (offset a multiple of 8 elements: 16-byte aligned)."""
    n = 1
    for s in shape:
        n *= s
    buf = torch.full((front + n + back,), fill, dtype=dtype, device=dev)
    return buf, buf[front:front + n].view(shape)


def _run(fn, x, w, bias, act, residual, out_fp32, M, N, dev):
    """Result written into a [M, N + 24] NaN buffer (ldc > N); returns the whole buffer so the margins can be compared too."""
    dt = torch.float32 if out_fp32 else torch.bfloat16
    full = torch.full((M, N + 24), float("nan"), dtype=dt, device=dev)
    out = full[:, :N]
    res = None
    if residual is not None:
        out.copy_(residual)   # in place, as the model's x += ... GEMMs
        res = out
    fn(x, w, bias, act, res, out)
    return full


@pytest.mark.parametrize("pair", [0, 1], ids=["single", "pair"])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: f"C{g[0]}k{g[1]}s{g[2]}p{g[3]}N{g[4]}")
def test_conv_gemm_matches_im2col_gemm(geom, size, pair, monkeypatch):
    C, k, st, pad, N = geom
    B, H, W = size
    if H + 2 * pad < k or W + 2 * pad < k:
        pytest.skip("window larger than the input")
    monkeypatch.setenv("SURGVID_GEMM_PAIR", str(pair))
    dev = torch.device("cuda")
    g = torch.Generator(device="cpu").manual_seed(C * 1000 + k * 10 + B)
    _, x = _padded((B, H, W, C), torch.bfloat16, float("nan"), dev)
    x.copy_(torch.randn(B, H, W, C, generator=g).to(torch.bfloat16))
    K = k * k * C
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(torch.bfloat16).to(dev)
    bias = torch.randn(N, generator=g).to(dev)
    Ho, Wo = (H + 2 * pad - k) // st + 1, (W + 2 * pad - k) // st + 1
    M = B * Ho * Wo
    plan = ops.conv_gemm_plan_info(B, H, W, C, k, st, pad, N, True, False, pair, torch.cuda.get_device_properties(0).multi_processor_count)
    assert plan["a_form"] == "im2col" and plan["gemm"]["pair"] == pair, plan
    for out_fp32, resid, act in FORMS:
        residual = torch.randn(M, N, generator=g).to(dev) if resid else None
        col = ops.im2col(x, k, st, pad)

        def ref(x_, w_, b_, a_, r_, o_):
            ops.gemm_bf16(col, w_, b_, a_, r_, o_.dtype, out=o_)

        def imp(x_, w_, b_, a_, r_, o_):
            ops.conv_gemm(x_, w_, k, st, pad, b_, a_, r_, o_.dtype, out=o_)

        want = _run(ref, x, w, bias, act, residual, out_fp32, M, N, dev)
        got = _run(imp, x, w, bias, act, residual, out_fp32, M, N, dev)
        torch.cuda.synchronize()
        assert torch.isfinite(got[:, :N].float()).all(), (out_fp32, resid, act)
        iv = torch.int32 if out_fp32 else torch.int16
        assert torch.equal(got.view(iv), want.view(iv)), (out_fp32, resid, act, (got[:, :N].float() - want[:, :N].float()).abs().max().item())


def _evp_counts(H, W, n=2):
    from surgvid_b200 import synthetic as S
    from surgvid_b200.models.mix_transformer_evp import mit_b3_evp

    dev = torch.device("cuda:0")
    sd = S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=0, mode="stress")
    model = mit_b3_evp()
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()
    x, seg, flow = S.synth_frames(n, seed=7, H=H, W=W)
    with torch.no_grad():
        model(x.to(dev), seg.to(dev), flow.to(dev), return_features=True)   # one micro-batch: builds the plan
    lib = _native.lib()
    h = model._native[0]["handle"]
    _native.check(lib.sv_evp_set_profile(h, 1), "sv_evp_set_profile")
    with torch.no_grad():
        model(x.to(dev), seg.to(dev), flow.to(dev), return_features=True)
    torch.cuda.synchronize()
    ms = (ctypes.c_double * 9)()
    launches = (ctypes.c_int64 * 9)()
    flops = ctypes.c_double()
    _native.check(lib.sv_evp_get_profile(h, ms, launches, ctypes.byref(flops), None), "sv_evp_get_profile")
    _native.check(lib.sv_evp_set_profile(h, 0), "sv_evp_set_profile")
    ws = lib.sv_evp_workspace_bytes(h, n, H, W)
    return list(launches), model.last_launch_count(), ws


# sv_evp_workspace_bytes of mit_b3_evp (micro-batch 2) in the build that gathered every conv of stages 2-4 into an im2col buffer and had
# LN1 write a second, sr-patch-ordered bf16 copy for the sr convs (measured with that build; 365 launches per micro-batch there)
PREV_WORKSPACE = {(224, 224): 26380288, (480, 854): 216342016}


@pytest.mark.parametrize("hw", [(224, 224), (480, 854)], ids=["224", "480x854"])
def test_evp_launches_and_workspace(hw):
    launches, total, ws = _evp_counts(*hw)
    # classes: 0 GEMM, 1 LayerNorm, 2 im2col, ...  Only the handcrafted-prompt convs of stages 2-4 (C_in = 16 / 32 / 80) still gather:
    # 3 im2col launches per micro-batch instead of 9 (patch embed, handcrafted and flow conv of each of stages 2-4)
    assert launches[2] == 3, launches
    assert sum(launches) == total == 365 - 6, (launches, total)
    assert 0 < ws < PREV_WORKSPACE[hw], (ws, PREV_WORKSPACE[hw])
