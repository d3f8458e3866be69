"""Implicit-GEMM convolutions without a device: which convs of mit_b0..b5 read their NHWC input through an im2col-mode TMA map
(`sv_op_conv_gemm_plan_info`), the output grid each reports against the usual conv arithmetic, and argument errors of
`sv_op_conv_gemm_bf16`, which come back before any device is touched."""
import ctypes

import pytest

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native, ops
from surgvid_b200 import synthetic as S

SV_ERR_INVALID, SV_ERR_UNSUPPORTED = 1, 4
SHAPES = [(224, 224), (480, 854)]


def conv_out_dim(n, k, s, p):
    return (n + 2 * p - k) // s + 1


def model_convs(name, H, W, n=3):
    """(what, B, H, W, C_in, k, stride, pad, C_out) of every conv after the stems, in the order the model runs them."""
    cfg = S.EVP_CONFIGS[name]
    dims, srs = cfg["embed_dims"], cfg["sr_ratios"]
    grid, h, w = [], H, W
    for s, (k, st) in enumerate([(7, 4), (3, 2), (3, 2), (3, 2)]):
        h, w = conv_out_dim(h, k, st, k // 2), conv_out_dim(w, k, st, k // 2)
        grid.append((h, w))
    fch = [2, 64, 128, dims[2], dims[3]]
    out = []
    for s in range(1, 4):
        hi, wi = grid[s - 1]
        out.append((f"patch_embed{s + 1}", n, hi, wi, dims[s - 1], 3, 2, 1, dims[s]))
        out.append((f"handcrafted{s + 1}", n, hi, wi, dims[s - 1] // 4, 3, 2, 1, dims[s] // 4))
        out.append((f"flow_conv{s + 1}", n, hi, wi, fch[s], 3, 2, 1, fch[s + 1]))
    for s in range(4):
        if srs[s] > 1:
            hi, wi = grid[s]
            out.append((f"sr{s + 1}", n, hi, wi, dims[s], srs[s], srs[s], 0, dims[s]))
    return out


@pytest.mark.parametrize("hw", SHAPES, ids=lambda t: f"{t[0]}x{t[1]}")
@pytest.mark.parametrize("name", sorted(S.EVP_CONFIGS))
def test_model_convs_plan(name, hw):
    for what, B, H, W, C, k, st, pad, N in model_convs(name, *hw):
        d = ops.conv_gemm_plan_info(B, H, W, C, k, st, pad, N, out_fp32=not what.startswith("flow"), num_sms=148)
        Ho, Wo = conv_out_dim(H, k, st, pad), conv_out_dim(W, k, st, pad)
        assert (d["Ho"], d["Wo"], d["M"], d["K"]) == (Ho, Wo, B * Ho * Wo, k * k * C), (what, d)
        # eligible: whole 64-channel k-blocks; k3 s2 p1 and k = s <= 8, p 0 fit the 4-D map's corner and stride limits
        assert d["a_form"] == ("im2col" if C % 64 == 0 else "tiled"), (name, what, C, d)
        if what.startswith("sr"):   # the sr conv's grid is the attention's key grid: floor(H / sr) x floor(W / sr)
            assert (Ho, Wo) == (H // k, W // k)
        # the GEMM it runs is the one gemm_plan_info picks for the same problem
        K = d["K"] if d["a_form"] == "im2col" else (d["K"] + 7) // 8 * 8
        g = ops.gemm_plan_info(d["M"], N, K, 0, not what.startswith("flow"), False, -1, num_sms=148)
        assert d["gemm"] == g, (what, d["gemm"], g)


def test_mit_b3_forms():
    """mit_b3 at 480x854: patch embeds 2-4, flow convs 2-4 and all three sr convs go through the map; the handcrafted-prompt convs
    (C_in = 16 / 32 / 80) do not.  Stage 1 there is 120 x 214, so the k = s = 8 sr conv truncates to 15 x 26."""
    forms = {c[0]: ops.conv_gemm_plan_info(*c[1:], num_sms=148) for c in model_convs("mit_b3_evp", 480, 854)}
    im2col = sorted(w for w, d in forms.items() if d["a_form"] == "im2col")
    assert im2col == sorted(["patch_embed2", "patch_embed3", "patch_embed4", "flow_conv2", "flow_conv3", "flow_conv4", "sr1", "sr2", "sr3"])
    assert (forms["sr1"]["Ho"], forms["sr1"]["Wo"]) == (15, 26)
    assert (forms["patch_embed2"]["Ho"], forms["patch_embed2"]["Wo"]) == (60, 107)
    assert (forms["patch_embed3"]["Ho"], forms["patch_embed3"]["Wo"]) == (30, 54)   # odd width 107 -> 54


@pytest.mark.parametrize("geom, ok", [
    ((1, 16, 16, 64, 3, 2, 1), True), ((1, 16, 16, 128, 8, 8, 0), True), ((1, 16, 16, 64, 9, 9, 0), False),   # stride 9 > 8
    ((1, 16, 16, 96, 3, 2, 1), False),
    ((1, 300, 300, 64, 3, 1, 128), True), ((1, 300, 300, 64, 3, 1, 129), False),   # lower corner -pad: -128 fits, -129 does not
    ((1, 300, 300, 64, 1, 1, 127), True), ((1, 300, 300, 64, 1, 1, 128), False),   # upper corner pad - (k - 1): 127 fits, 128 does not
    ((1, 300, 300, 64, 129, 1, 0), True), ((1, 300, 300, 64, 130, 1, 0), False)])   # ... -128 fits, -129 does not
def test_eligibility_limits(geom, ok):
    d = ops.conv_gemm_plan_info(*geom, N=64, num_sms=148)
    assert d["a_form"] == ("im2col" if ok else "tiled"), (geom, d)


def _conv_rc(**kw):
    a = dict(x=1, B=2, H=16, W=16, C=64, k=3, stride=2, pad=1, w=1, ldw=576, N=64, bias=None, act=0, res=None, ldr=0, out=1, ldc=64, f32=1)
    a.update(kw)
    p = lambda v: ctypes.c_void_p(v)   # noqa: E731 - never dereferenced: every case fails its argument checks first
    lib = _native.lib()
    rc = lib.sv_op_conv_gemm_bf16(p(a["x"]), a["B"], a["H"], a["W"], a["C"], a["k"], a["stride"], a["pad"], p(a["w"]), a["ldw"], a["N"], p(a["bias"]),
                                  a["act"], p(a["res"]), a["ldr"], p(a["out"]), a["ldc"], a["f32"], None)
    return rc, _native.last_error()


@pytest.mark.parametrize("kw", [dict(x=None), dict(w=None), dict(out=None), dict(B=0), dict(C=-64), dict(k=0), dict(stride=0), dict(pad=-1),
                                dict(H=1, pad=0), dict(N=60), dict(ldw=575), dict(ldc=32), dict(act=3)],
                         ids=lambda kw: ",".join(f"{k}={v}" for k, v in kw.items()))
def test_conv_gemm_argument_errors(kw):
    rc, msg = _conv_rc(**kw)
    assert rc == SV_ERR_INVALID, (kw, rc, msg)
    assert "conv GEMM" in msg, msg


def test_conv_gemm_unsupported_geometry():
    rc, msg = _conv_rc(C=96, ldw=9 * 96)
    assert rc == SV_ERR_UNSUPPORTED and "C % 64" in msg, (rc, msg)


def test_plan_info_argument_errors():
    ci, gi = (ctypes.c_int32 * 5)(), (ctypes.c_int32 * len(ops.GEMM_PLAN_FIELDS))()
    lib = _native.lib()
    assert lib.sv_op_conv_gemm_plan_info(1, 16, 16, 64, 0, 1, 0, 64, 1, 0, -1, 148, ci, gi) == SV_ERR_INVALID
    assert lib.sv_op_conv_gemm_plan_info(1, 2, 2, 64, 7, 1, 0, 64, 1, 0, -1, 148, ci, gi) == SV_ERR_INVALID   # window larger than the input
    assert lib.sv_op_conv_gemm_plan_info(1, 16, 16, 64, 3, 1, 1, 64, 1, 0, -1, 148, None, gi) == SV_ERR_INVALID
