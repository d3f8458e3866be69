"""CPU-side checks of the drop-in surface: state_dict contract, C-ABI exports, loud failure without CUDA, sharding."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native, lfb
from surgvid_b200 import synthetic as S
from surgvid_b200.models.mix_transformer_evp import mit_b0_evp, mit_b3_evp
from surgvid_b200.mstcn import MultiStageModel_S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_evp_state_dict_contract():
    m = mit_b3_evp()
    sd = m.state_dict()
    shapes = S.evp_key_shapes("mit_b3_evp")
    assert len(sd) == 722
    assert list(sd.keys()) == list(shapes.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(shapes[k]), k
    assert sum(p.numel() for p in m.parameters()) == 68_941_518
    # strict round trip with a foreign state_dict
    synth = S.synth_state_dict(shapes, seed=5, mode="stress")
    missing, unexpected = m.load_state_dict(synth, strict=True)
    assert not missing and not unexpected
    assert torch.equal(m.state_dict()["block3.7.attn.kv.weight"], synth["block3.7.attn.kv.weight"])


def test_evp_b0_keys():
    m = mit_b0_evp()
    assert list(m.state_dict().keys()) == list(S.evp_key_shapes("mit_b0_evp").keys())


def test_mstcn_state_dict_contract(capsys):
    m = MultiStageModel_S(2, 8, 32, 2048, 14, True)
    assert "num_stages_classification: 2, num_layers: 8, num_f_maps: 32, dim: 2048" in capsys.readouterr().out
    sd = m.state_dict()
    shapes = S.mstcn_key_shapes(2, 8, 32, 2048, 14)
    assert len(sd) == 72 and list(sd.keys()) == list(shapes.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(shapes[k]), k
    assert sum(p.numel() for p in m.parameters()) == 133_532
    m.load_state_dict(S.synth_mstcn_state_dict(mode="stress"), strict=True)
    with pytest.raises(NotImplementedError):
        MultiStageModel_S(2, 8, 32, 2048, 14, False)


def test_init_follows_reference():
    """Same init distributions as the reference (mix_transformer_evp.py:300-313): Linear weights trunc_normal(std 0.02), conv
    weights normal(0, sqrt(2 / fan_out)).  MS-TCN under manual_seed(0) draws the reference module's weights: the sum of its
    stage-1 input projection is the known answer recorded from the reference (SURVEY.md §8c)."""
    mine = mit_b3_evp()
    assert abs(float(mine.block3[5].mlp.fc1.weight.std()) - 0.02) < 2e-3
    w = mine.patch_embed2.proj.weight
    assert abs(float(w.std()) - (2.0 / (w.shape[0] * w.shape[2] * w.shape[3])) ** 0.5) < 5e-3
    torch.manual_seed(0)
    sd = MultiStageModel_S(2, 8, 32, 2048, 14, True).state_dict()
    assert abs(float(sd["stage1_phase.conv_1x1.weight"].double().sum()) - 0.688543) < 2e-6


def test_no_cpu_fallback():
    m = mit_b3_evp().eval()
    x = torch.zeros(1, 1, 3, 224, 224)
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(x, x, None, return_features=True)
    with pytest.raises(RuntimeError, match="parameter holder"):
        m.block1[0](torch.zeros(1, 4, 64))
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m(x, x)
    t = MultiStageModel_S(2, 8, 32, 2048, 14, True).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        t(torch.zeros(1, 2048, 10))


def test_c_abi_exports_every_declared_symbol():
    """The shared library loads (no GPU needed) and exports every function include/surgvid.h declares."""
    header = open(os.path.join(ROOT, "include", "surgvid.h")).read()
    declared = sorted(set(re.findall(r"\b(sv_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 26
    assert sorted(_native.EXPORTED_SYMBOLS) == declared
    lib = _native.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.sv_abi_version() == 2
    # argument validation works without a device and reports through sv_last_error
    assert lib.sv_evp_create(None, None) != 0
    assert b"null" in lib.sv_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour WITHOUT a CUDA device")
def test_compute_entry_points_fail_loudly_without_cuda():
    lib = _native.lib()
    cfg = _native.MstcnCfg(2, 8, 32, 2048, 14, 1)
    h = ctypes.c_void_p()
    rc = lib.sv_mstcn_create(ctypes.byref(cfg), ctypes.byref(h))
    assert rc == 2 and len(lib.sv_last_error()) > 0  # SV_ERR_CUDA: no device, and no CPU fallback


def test_video_lengths_and_lpt():
    L = S.cholec80_video_lengths()
    assert len(L) == 80 and L[:40].sum() == 86344 and L[40:].sum() == 98234 and L.sum() == 184578
    assert L.min() >= 600 and L.max() <= 7000
    for n in (1, 2, 4, 8):
        a = lfb.lpt_assign(L, n)
        assert sorted(v for b in a for v in b) == list(range(80))
        loads = [int(L[b].sum()) for b in a]
        assert max(loads) / (L.sum() / n) < 1.02  # < 2 % imbalance (SURVEY.md §8e)


def test_gather_in_video_order():
    L = [5, 3, 7, 2, 4]
    a = lfb.lpt_assign(L, 2)
    blocks = [[np.full((L[v], 4), v, dtype=np.float32) for v in vids] for vids in a]
    out = lfb.gather_in_video_order(blocks, a, len(L))
    expect = np.concatenate([np.full((L[v], 4), v, dtype=np.float32) for v in range(len(L))])
    assert np.array_equal(out, expect)
    with pytest.raises(ValueError):
        lfb.gather_in_video_order([blocks[0], blocks[1][:-1]], a, len(L))


def test_gemm_tile_picker_is_legal():
    lib = _native.lib()  # noqa: F841  (library must at least load)
    # legal UMMA N for M=128: multiple of 16 in [16, 256]; mirrored in Python for the shapes the model uses
    from surgvid_b200.synthetic import EVP_CONFIGS
    for C in EVP_CONFIGS["mit_b3_evp"]["embed_dims"]:
        for N in (C // 4, C, 2 * C, 4 * C, 2048):
            assert N % 8 == 0


def test_ramp_schedule_covers_every_frame_once():
    from surgvid_b200.lfb import ramp_schedule
    for n, b, r in [(2300, 800, 100), (2300, 200, 25), (7, 4, 1), (1, 800, 100), (800, 800, 800), (0, 800, 100)]:
        sched = ramp_schedule(n, b, r)
        assert sum(c for _, c in sched) == n
        pos = 0
        for b0, c in sched:
            assert b0 == pos and 1 <= c <= b
            pos += c
        if n >= r:
            assert sched[0][1] == min(r, b)
    assert ramp_schedule(2300, 800, 100) == [(0, 100), (100, 200), (300, 400), (700, 800), (1500, 800)]


def test_numa_binding_is_a_no_op_without_a_gpu():
    import os
    from surgvid_b200.lfb import bind_to_gpu_numa_node
    before = os.sched_getaffinity(0)
    assert bind_to_gpu_numa_node(0) is None or isinstance(bind_to_gpu_numa_node(0), list)
    if not __import__("torch").cuda.is_available():
        assert os.sched_getaffinity(0) == before


def test_trans_head_holder_keys_and_no_cpu_path():
    """adapter_transformer.Transformer's constructor arguments (adapter_transformer.py:290-325); the inner module's source is absent
    from the reference, so its parameter names are this package's (documented as parity-unpinned)."""
    import pytest
    import torch
    from surgvid_b200.trans_head import Transformer
    head = Transformer(32, 2048, 14, 30)
    keys = set(head.state_dict())
    assert "fc.weight" in keys and head.fc.weight.shape == (14, 2048) and head.fc.bias is None
    for blk in ("transformer.encoder.layers.0.enc_self_attn", "transformer.decoder.layers.0.dec_enc_attn"):
        for p in ("W_Q", "W_K", "W_V", "fc"):
            assert f"{blk}.{p}.weight" in keys
        assert head.state_dict()[f"{blk}.W_Q.weight"].shape == (4 * 32, 14)
    assert head.transformer.d_k == 32 and head.transformer.d_ff == 32 and head.transformer.len_q == 30
    with pytest.raises(RuntimeError):
        head.eval().transformer.forward_fused(torch.zeros(14, 5), torch.zeros(5, 14), [5])
