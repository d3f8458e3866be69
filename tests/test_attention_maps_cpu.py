"""Attention-map capture without a GPU: the host-only layout call, argument checks of the new C ABI entry points, the `get_local`
drop-in and the reference maps of tests/attn_maps_ref.py."""
import ctypes
import importlib.util
import os
import sys

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from oracle import evp_oracle
from surgvid_b200 import _native, visualizer
from surgvid_b200 import synthetic as S
from surgvid_b200.models.mix_transformer_evp import mit_b0_evp, mit_b3_evp
from attn_maps_ref import encoder_maps

# the list vs_attn.py plots for mit_b3_evp at 224x224: (heads, N, N_kv) of the 3 + 4 + 18 + 3 blocks
B3_224 = [(1, 3136, 49)] * 3 + [(2, 784, 49)] * 4 + [(5, 196, 49)] * 18 + [(8, 49, 49)] * 3
B3_480 = [(1, 25680, 390)] * 3 + [(2, 6420, 390)] * 4 + [(5, 1620, 405)] * 18 + [(8, 405, 405)] * 3


def _offsets(B, dims):
    off = [0]
    for h, n, nk in dims:
        off.append(off[-1] + B * h * n * nk)
    return off


def test_layout_b3_224_is_the_vs_attn_list():
    off, dims = mit_b3_evp().attention_maps_layout(1, 224, 224)
    assert dims == B3_224
    assert off == _offsets(1, B3_224)
    assert off[-1] == 1_690_304  # 6.76 MB of fp32 per frame
    off4, _ = mit_b3_evp().attention_maps_layout(4, 224, 224)
    assert off4 == [4 * o for o in off]


def test_layout_b0_224_head_dim_32():
    m = mit_b0_evp()
    off, dims = m.attention_maps_layout(2, 224, 224)
    assert dims == [(1, 3136, 49)] * 2 + [(2, 784, 49)] * 2 + [(5, 196, 49)] * 2 + [(8, 49, 49)] * 2
    assert [m.embed_dims[s] // m.num_heads[s] for s in range(4)] == [32, 32, 32, 32]
    assert off == _offsets(2, dims)


def test_layout_480x854_offsets_past_2_31():
    m = mit_b3_evp()
    off1, dims = m.attention_maps_layout(1, 480, 854)
    assert dims == B3_480
    assert off1[-1] == 113_061_600  # 452 MB per frame
    off, dims = m.attention_maps_layout(19, 480, 854)
    assert off == _offsets(19, B3_480)
    assert off[-1] == 19 * 113_061_600 > 2 ** 31


def _cfg():
    return mit_b3_evp()._cfg()


def test_layout_rejects_bad_arguments():
    lib = _native.lib()
    cfg = _cfg()
    nb = ctypes.c_int32(-1)
    off = (ctypes.c_int64 * 29)()
    dims = (ctypes.c_int32 * 84)()
    assert lib.sv_evp_attention_maps_layout(None, 1, 224, 224, off, dims, 28, ctypes.byref(nb)) == 1
    assert lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), 1, 224, 224, off, dims, 28, None) == 1
    for B, H, W in ((0, 224, 224), (1, 0, 224), (1, 224, -1)):
        assert lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), B, H, W, off, dims, 28, ctypes.byref(nb)) == 1, (B, H, W)
    assert lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), 1, 224, 224, off, dims, 27, ctypes.byref(nb)) == 1
    assert b"max_blocks" in lib.sv_last_error() and nb.value == 28
    assert lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), 1, 224, 224, off, None, 28, ctypes.byref(nb)) == 1
    bad = _cfg()
    bad.depths[2] = 0
    assert lib.sv_evp_attention_maps_layout(ctypes.byref(bad), 1, 224, 224, off, dims, 28, ctypes.byref(nb)) == 1
    assert lib.sv_evp_attention_maps_layout(ctypes.byref(cfg), 1, 224, 224, off, dims, 28, ctypes.byref(nb)) == 0


def test_forward_attention_rejects_null_handle():
    lib = _native.lib()
    assert lib.sv_evp_forward_attention(None, None, None, None, None, None, 0, 1, 224, 224, 1, None, 0, None) == 1
    assert b"null" in lib.sv_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour WITHOUT a CUDA device")
def test_probs_op_fails_with_cuda_error_without_a_device():
    lib = _native.lib()
    # well-formed arguments (aligned dummy addresses): the launch itself is what fails, with SV_ERR_CUDA
    rc = lib.sv_op_attention_probs(ctypes.c_void_p(256), 64, ctypes.c_void_p(512), 128, 1, 1, 49, 49, 64, 0.125, ctypes.c_void_p(1024), None)
    assert rc == 2 and len(lib.sv_last_error()) > 0
    assert lib.sv_op_attention_probs(ctypes.c_void_p(256), 64, ctypes.c_void_p(512), 128, 1, 1, 49, 49, 40, 0.125, ctypes.c_void_p(1024), None) == 4


def test_attention_maps_has_no_cpu_path():
    m = mit_b3_evp().eval()
    x = torch.zeros(1, 3, 224, 224)
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.attention_maps(x, x)
    with pytest.raises(RuntimeError, match="inference-only"):
        m.train().attention_maps(x, x)


@pytest.fixture
def fresh_get_local():
    gl = visualizer.get_local
    saved = (dict(gl.cache), gl.is_activate)
    gl.cache.clear()
    gl.is_activate = False
    yield gl
    gl.cache.clear()
    gl.cache.update(saved[0])
    gl.is_activate = saved[1]


def test_get_local_surface(fresh_get_local):
    gl = fresh_get_local

    def f(a):
        return a + 1

    assert gl("attn")(f) is f
    assert gl.cache == {} and gl.is_activate is False
    assert visualizer.active_caches() == []
    gl.activate()
    assert gl.is_activate is True
    assert visualizer.active_caches() == [gl.cache]
    gl.cache["Attention.forward"] = [np.zeros(3), np.ones(2)]
    gl.clear()
    assert gl.cache == {"Attention.forward": []}


def test_get_local_under_its_reference_module_name(fresh_get_local):
    """Imported as `visualizer` (the sys.path switch), the same file's get_local is seen by the model's forward."""
    path = visualizer.__file__
    spec = importlib.util.spec_from_file_location("visualizer", path)
    mod = importlib.util.module_from_spec(spec)
    old = sys.modules.get("visualizer")
    sys.modules["visualizer"] = mod
    try:
        spec.loader.exec_module(mod)
        assert visualizer.active_caches() == []
        mod.get_local.activate()
        assert visualizer.active_caches() == [mod.get_local.cache]
        fresh_get_local.activate()
        assert len(visualizer.active_caches()) == 2
    finally:
        if old is None:
            sys.modules.pop("visualizer", None)
        else:
            sys.modules["visualizer"] = old


@pytest.mark.parametrize("variant", ["mit_b3_evp", "mit_b0_evp"])
def test_reference_maps_shapes_rows_and_features(variant):
    cfg = S.EVP_CONFIGS[variant]
    sd = S.synth_state_dict(S.evp_key_shapes(variant), seed=0, mode="stress")
    x, seg, _ = S.synth_frames(2, seed=5, H=64, W=96)
    maps, taps = encoder_maps(sd, cfg, x, seg)
    model = mit_b3_evp() if variant == "mit_b3_evp" else mit_b0_evp()
    _, dims = model.attention_maps_layout(2, 64, 96)
    assert [tuple(m.shape) for m in maps] == [(2,) + d for d in dims]
    for m in maps:
        assert torch.isfinite(m).all()
        assert (m.sum(-1) - 1).abs().max().item() < 1e-5
    ref_taps = {}
    evp_oracle.evp_forward(sd, cfg, x, seg, None, taps=ref_taps)
    for k, v in ref_taps.items():
        assert torch.equal(v, taps[k]), k
