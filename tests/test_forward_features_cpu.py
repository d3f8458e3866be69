"""forward_features without a GPU: the host-only stage shapes and the argument checks of the new C ABI entry points."""
import ctypes

import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native
from surgvid_b200.models.mix_transformer_evp import mit_b0_evp, mit_b3_evp


def _conv(n, k, s, p):
    return (n + 2 * p - k) // s + 1


def _expected(dims, H, W):
    out, h, w = [], H, W
    for s, (k, st, p) in enumerate(((7, 4, 3), (3, 2, 1), (3, 2, 1), (3, 2, 1))):
        h, w = _conv(h, k, st, p), _conv(w, k, st, p)
        out.append((dims[s], h, w))
    return out


@pytest.mark.parametrize("H,W", [(224, 224), (480, 854), (225, 301), (29, 29), (97, 31)])
def test_stage_shapes_follow_the_conv_formula(H, W):
    for m in (mit_b3_evp(), mit_b0_evp()):
        assert m.stage_shapes(H, W) == _expected(m.embed_dims, H, W)


def test_stage_shapes_of_the_reference_sizes():
    m = mit_b3_evp()
    assert m.stage_shapes(224, 224) == [(64, 56, 56), (128, 28, 28), (320, 14, 14), (512, 7, 7)]
    assert m.stage_shapes(480, 854) == [(64, 120, 214), (128, 60, 107), (320, 30, 54), (512, 15, 27)]


def test_stage_shapes_reject_bad_arguments():
    lib = _native.lib()
    cfg = mit_b3_evp()._cfg()
    dims = (ctypes.c_int32 * 12)()
    # 28 x 28 gives a 7 x 7 stage-1 map, smaller than its 8 x 8 spatial-reduction window; 29 is the smallest size that runs
    for H, W in ((0, 224), (224, -1), (28, 224), (224, 28), (16, 16), (1, 1)):
        assert lib.sv_evp_stage_shapes(ctypes.byref(cfg), H, W, dims) == 1, (H, W)
        assert len(lib.sv_last_error()) > 0
    assert b"too small" in (lib.sv_evp_stage_shapes(ctypes.byref(cfg), 28, 28, dims), lib.sv_last_error())[1]
    assert lib.sv_evp_stage_shapes(None, 224, 224, dims) == 1
    assert lib.sv_evp_stage_shapes(ctypes.byref(cfg), 224, 224, None) == 1
    bad = mit_b3_evp()._cfg()
    bad.num_heads[1] = 3  # 128 is not divisible by 3
    assert lib.sv_evp_stage_shapes(ctypes.byref(bad), 224, 224, dims) == 1
    assert lib.sv_evp_stage_shapes(ctypes.byref(cfg), 29, 29, dims) == 0
    with pytest.raises(RuntimeError, match="too small"):
        mit_b3_evp().stage_shapes(28, 28)


def test_forward_features_rejects_null_arguments():
    lib = _native.lib()
    ptrs = (ctypes.c_void_p * 4)(256, 512, 768, 1024)
    elems = (ctypes.c_int64 * 4)(*([1 << 30] * 4))
    assert lib.sv_evp_forward_features(None, None, None, None, None, None, 0, 1, 224, 224, 1, None, 0, None) == 1
    assert b"null" in lib.sv_last_error()
    assert lib.sv_evp_forward_features(None, ctypes.c_void_p(256), ctypes.c_void_p(512), ptrs, elems, None, 0, 1, 224, 224, 1,
                                       ctypes.c_void_p(1024), 1 << 30, None) == 1
    assert b"null" in lib.sv_last_error()


def test_layernorm_nchw_argument_errors_without_a_device():
    lib = _native.lib()
    x, g, b, o, ob = (ctypes.c_void_p(a) for a in (256, 512, 768, 1024, 2048))

    def call(x=x, g=g, b=b, rows=98, C=64, tokens=49, o=o, ob=ob):
        return lib.sv_op_layernorm_nchw(x, g, b, 1e-6, rows, C, tokens, o, ob, None)

    cases = [dict(x=None), dict(o=None), dict(g=None), dict(C=66), dict(C=0), dict(C=516), dict(tokens=0), dict(rows=0), dict(rows=97),
             dict(rows=1 << 23, tokens=1 << 13, C=512), dict(x=ctypes.c_void_p(260)), dict(o=ctypes.c_void_p(1026)),
             dict(ob=ctypes.c_void_p(2052))]
    for kw in cases:
        assert call(**kw) == 1, kw
        assert len(lib.sv_last_error()) > 0, kw
    assert b"multiple of the tokens" in (call(rows=97), lib.sv_last_error())[1]
    assert b"2^31" in (call(rows=1 << 23, tokens=1 << 13, C=512), lib.sv_last_error())[1]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour WITHOUT a CUDA device")
def test_layernorm_nchw_fails_with_cuda_error_without_a_device():
    lib = _native.lib()
    rc = lib.sv_op_layernorm_nchw(ctypes.c_void_p(256), ctypes.c_void_p(512), ctypes.c_void_p(768), 1e-6, 98, 64, 49, ctypes.c_void_p(1024),
                                  None, None)
    assert rc == 2 and len(lib.sv_last_error()) > 0


def test_forward_features_has_no_cpu_path():
    m = mit_b3_evp().eval()
    x = torch.zeros(1, 3, 224, 224)
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.forward_features(x, x)
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m.forward_features(x, x)
