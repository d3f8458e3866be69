"""End-to-end parity of the CUDA LFB path (drop-in mit_b3_evp -> torch.ops.surgvid.evp_lfb_forward -> C ABI) against
  * the committed golden vectors (outputs of the real reference), and
  * the fp32 oracle (oracle/evp_oracle.py) run on the same seeded inputs and weights.
Tolerances (SURVEY.md §8d "parity gates"; bf16 operands, fp32 accumulate, fp32 residual stream):
  rel-L2 <= 1.5e-2 and max-abs <= 3e-2 * max|ref|.  The oracle with bf16-rounded operands sits at rel-L2 ~2-3.5e-3."""
import os

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from oracle import evp_oracle as EO
from surgvid_b200 import synthetic as S
from surgvid_b200.models.mix_transformer_evp import mit_b3_evp

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CFG = S.EVP_CONFIGS["mit_b3_evp"]
REL_L2_TOL = 1.5e-2
MAXABS_TOL = 3e-2


def _rel_l2(a, b):
    return float((a - b).norm() / b.norm())


def _check(out, ref, what=""):
    out, ref = out.float().cpu(), ref.float().cpu()
    rel, mx = _rel_l2(out, ref), float((out - ref).abs().max())
    print(f"[parity] {what}: rel-L2 {rel:.3e}  max-abs {mx:.3e}  (max|ref| {float(ref.abs().max()):.3f})")
    assert rel <= REL_L2_TOL, (what, rel)
    assert mx <= MAXABS_TOL * float(ref.abs().max()), (what, mx)


_MODELS = {}


def _model(mode, fold=False):
    key = (mode, fold)
    if key not in _MODELS:
        m = mit_b3_evp()
        sd = S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=0, mode=mode)
        m.load_state_dict(sd, strict=True)
        m.fold_head = fold
        _MODELS[key] = (m.to(DEV).eval(), sd)
    return _MODELS[key]


def _tap_sample(t, n=2048):
    flat = t.reshape(-1)
    idx = torch.linspace(0, flat.numel() - 1, n).long().to(flat.device)
    return flat[idx].float().cpu().numpy()


@pytest.mark.parametrize("mode", ["ref_init", "stress"])
def test_lfb_features_match_golden_and_taps(golden_dir, mode):
    g = np.load(os.path.join(golden_dir, f"evp_b3_{mode}_224.npz"))
    m, _ = _model(mode)
    x, seg, flow = S.synth_frames(int(g["n"]), seed=int(g["input_seed"]), device=DEV)
    with torch.no_grad():
        feats = m(x, seg, flow, return_features=True)
    torch.cuda.synchronize()
    assert feats.shape == (2, 2048) and feats.dtype == torch.float32
    # localise errors first: per-stage taps against the reference's own intermediate activations
    for k in ("stage1_tokens", "stage2_tokens", "stage3_tokens", "stage4_tokens", "fused3_tokens", "fused4_tokens"):
        got, ref = _tap_sample(m.read_tap(k)), g[k]
        rel = float(np.linalg.norm(got - ref) / np.linalg.norm(ref))
        print(f"[tap] {mode} {k}: rel-L2 {rel:.3e}")
        assert rel < 3e-2, (k, rel)
    _check(feats, torch.from_numpy(g["feats"]), f"{mode} feats vs golden")
    with torch.no_grad():
        nf = m(x, seg, None, return_features=True)
        y, y_ant = m(x, seg, flow)  # return_features=False -> (fc, fc_ant)
    _check(nf, torch.from_numpy(g["feats_noflow"]), f"{mode} feats (flow=None) vs golden")
    assert y.shape == (2, 7) and y_ant.shape == (2, 7)
    assert float((y.cpu() - torch.from_numpy(g["y"])).abs().max()) < 3e-2 * max(1.0, float(np.abs(g["y"]).max()))
    assert float((y_ant.cpu() - torch.from_numpy(g["y_ant"])).abs().max()) < 3e-2 * max(1.0, float(np.abs(g["y_ant"]).max()))


@pytest.mark.parametrize("mode", ["ref_init", "stress"])
def test_lfb_features_match_oracle_with_ragged_microbatches(mode):
    """7 frames with micro_batch 3 -> plans for n=3 and a tail n=1; frames must not bleed into each other."""
    m, sd = _model(mode)
    x, seg, flow = S.synth_frames(7, seed=101)
    ref = EO.evp_forward(sd, CFG, x, seg, flow)
    m.micro_batch = 3
    with torch.no_grad():
        out = m(x.to(DEV), seg.to(DEV), flow.to(DEV), return_features=True)
        m.micro_batch = 7
        out7 = m(x.to(DEV), seg.to(DEV), flow.to(DEV), return_features=True)
    m.micro_batch = 32
    _check(out, ref, f"{mode} B=7 mb=3 vs oracle")
    _check(out7, ref, f"{mode} B=7 mb=7 vs oracle")
    # per-frame independence: same frame, different batch composition -> bit-identical features
    with torch.no_grad():
        single = m(x[4:5].to(DEV), seg[4:5].to(DEV), flow[4:5].to(DEV), return_features=True)
    assert torch.equal(single[0], out7[4])


def test_folded_head_matches_oracle():
    m, sd = _model("stress", fold=True)
    x, seg, flow = S.synth_frames(3, seed=55)
    ref = EO.evp_forward(sd, CFG, x, seg, flow)
    with torch.no_grad():
        out = m(x.to(DEV), seg.to(DEV), flow.to(DEV), return_features=True)
    _check(out, ref, "folded head vs oracle")


def test_480x854_matches_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "evp_b3_stress_480x854.npz"))
    m, _ = _model("stress")
    x, seg, flow = S.synth_frames(1, seed=int(g["input_seed"]), H=480, W=854, device=DEV)
    with torch.no_grad():
        out = m(x, seg, flow, return_features=True)
    _check(out, torch.from_numpy(g["feats"]), "480x854 vs golden")


def test_reload_state_dict_repacks():
    m, sd = _model("ref_init")
    x, seg, flow = S.synth_frames(1, seed=9, device=DEV)
    with torch.no_grad():
        a = m(x, seg, flow, return_features=True).clone()
        sd2 = S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=1, mode="ref_init")
        m.load_state_dict(sd2, strict=True)
        b = m(x, seg, flow, return_features=True).clone()
        m.load_state_dict(sd, strict=True)
        c = m(x, seg, flow, return_features=True)
    assert not torch.allclose(a, b) and torch.equal(a, c)


@pytest.mark.parametrize("variant,hw,with_flow", [("mit_b0_evp", (224, 224), True), ("mit_b0_evp", (96, 160), False), ("mit_b2_evp", (128, 128), True),
                                                  ("mit_b1_evp", (224, 224), True)])
def test_other_variants_match_oracle(variant, hw, with_flow):
    """The reference exports mit_b0..b5_evp (mix_transformer_evp.py:897-939); the LFB driver uses b3, the others share the code path.
    b0 has different widths everywhere (32/64/160/256; adapter 8/16/40/64; block head_dim 32, flow cross-attention head_dim 20 and 32);
    b1/b2 differ in depth only."""
    from surgvid_b200.models import mix_transformer_evp as M
    cfg = S.EVP_CONFIGS[variant]
    m = getattr(M, variant)()
    sd = S.synth_state_dict(S.evp_key_shapes(variant), seed=2, mode="stress")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval()
    x, seg, flow = S.synth_frames(3, seed=77, H=hw[0], W=hw[1])
    if not with_flow:
        flow = None
    ref = EO.evp_forward(sd, cfg, x, seg, flow)
    with torch.no_grad():
        out = m(x.to(DEV), seg.to(DEV), None if flow is None else flow.to(DEV), return_features=True)
    _check(out, ref, f"{variant} {hw[0]}x{hw[1]} flow={with_flow} vs oracle")


def test_simt_dwconv_and_im2col_from_input_match_oracle(tmp_path):
    """Two launch forms no mit_bX_evp reaches: stage 1's MixFFN width 96 x 2 = 192 is not a multiple of 128, so its DWConv runs the
    SIMT kernel instead of the TMA one, and stage 1's patch embed (Cout 96) cannot use the fused stem, so im2col reads the call's x.
    The plan's profile shows both: im2col with Cin 3 for the handcrafted prompt and the patch embed, DWConv with C 192."""
    import csv
    from collections import OrderedDict
    from functools import partial

    from surgvid_b200 import _native
    from surgvid_b200.models.mix_transformer_evp import MixVisionTransformerEVP
    cfg = dict(embed_dims=[96, 192, 320, 512], num_heads=[3, 3, 5, 8], depths=[2, 2, 2, 2], sr_ratios=[8, 4, 2, 1])
    m = MixVisionTransformerEVP(patch_size=4, mlp_ratios=[2] * 4, qkv_bias=True, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6),
                                drop_rate=0.0, drop_path_rate=0.1, **cfg)
    sd = S.synth_state_dict(OrderedDict((k, tuple(v.shape)) for k, v in m.state_dict().items()), seed=2, mode="stress")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval()
    x, seg, flow = S.synth_frames(3, seed=77)
    ref = EO.evp_forward(sd, cfg, x, seg, flow)
    with torch.no_grad():
        out = m(x.to(DEV), seg.to(DEV), flow.to(DEV), return_features=True)
    _check(out, ref, "embed_dims 96/192/320/512, mlp_ratio 2 vs oracle")
    lib, h = _native.lib(), m._native[0]["handle"]
    _native.check(lib.sv_evp_set_profile(h, 1), "sv_evp_set_profile")
    with torch.no_grad():
        m(x.to(DEV), seg.to(DEV), flow.to(DEV), return_features=True)
    torch.cuda.synchronize()
    path = tmp_path / "ops.csv"
    _native.check(lib.sv_evp_dump_profile(h, str(path).encode()), "sv_evp_dump_profile")
    _native.check(lib.sv_evp_set_profile(h, 0), "sv_evp_set_profile")
    rows = list(csv.DictReader(open(path)))
    assert sum(r["kind"] == "im2col" and r["i1"] == "3" for r in rows) == 2, rows
    assert any(r["kind"] == "dwconv" and r["i3"] == "192" for r in rows), rows


def test_full_size_video_properties():
    """BASELINE configs[1] at full size (one 2 300-frame video, the bench's micro-batch of 800) through size-independent properties:
    (1) frames are independent, so the features of the whole video are bit-identical to those of any sub-range processed on its own
        and do not depend on the micro-batch size (800 / 200 / 37);
    (2) a sample of frames matches the fp32 oracle within the parity tolerance."""
    m, sd = _model("stress")
    T = 2300
    x, seg, flow = S.synth_frames(T, seed=4242, device=DEV)
    with torch.no_grad():
        m.micro_batch = 800
        full = m(x, seg, flow, return_features=True).clone()
        m.micro_batch = 200
        part = m(x[1500:2100], seg[1500:2100], flow[1500:2100], return_features=True).clone()
        m.micro_batch = 37
        tail = m(x[2200:], seg[2200:], flow[2200:], return_features=True).clone()
    m.micro_batch = 800
    assert full.shape == (T, 2048) and bool(torch.isfinite(full).all())
    assert torch.equal(full[1500:2100], part)
    assert torch.equal(full[2200:], tail)
    idx = [0, 799, 800, 1601, 2299]
    ref = EO.evp_forward(sd, CFG, x[idx].cpu(), seg[idx].cpu(), flow[idx].cpu())
    _check(full[idx], ref, "2300-frame video, sampled frames vs oracle")
