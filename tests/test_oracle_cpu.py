"""Pins the oracle (oracle/*.py, a CPU restatement of the reference) against
  (a) the committed golden vectors, which are outputs of the REAL reference (tests/golden/make_golden.py), and
  (b) a known answer recorded from the reference's own MS-TCN module.
The reference ships no tests or golden vectors of its own (SURVEY.md F4)."""
import os

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from oracle import evp_oracle as EO
from oracle import mstcn_oracle as MO
from surgvid_b200 import synthetic as S
from surgvid_b200.mstcn import MultiStageModel_S

CFG = S.EVP_CONFIGS["mit_b3_evp"]


def _tap_sample(t, n=2048):
    flat = t.reshape(-1)
    idx = torch.linspace(0, flat.numel() - 1, n).long()
    return flat[idx].numpy()


@pytest.mark.parametrize("mode", ["ref_init", "stress"])
def test_evp_oracle_matches_golden(golden_dir, mode):
    g = np.load(os.path.join(golden_dir, f"evp_b3_{mode}_224.npz"))
    sd = S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=int(g["weight_seed"]), mode=mode)
    x, seg, flow = S.synth_frames(int(g["n"]), seed=int(g["input_seed"]))
    taps = {}
    feats = EO.evp_forward(sd, CFG, x, seg, flow, taps=taps)
    assert np.abs(feats.numpy() - g["feats"]).max() < 5e-5
    for k in ("stage1_tokens", "stage2_tokens", "stage3_tokens", "stage4_tokens", "fused3_tokens", "fused4_tokens"):
        assert np.abs(_tap_sample(taps[k]) - g[k]).max() < 1e-3, k
    assert np.abs(EO.evp_forward(sd, CFG, x, seg, None).numpy() - g["feats_noflow"]).max() < 5e-5
    y, y_ant = EO.evp_forward(sd, CFG, x, seg, flow, return_features=False)
    assert np.abs(y.numpy() - g["y"]).max() < 5e-5 and np.abs(y_ant.numpy() - g["y_ant"]).max() < 5e-5


def test_evp_oracle_matches_golden_480x854(golden_dir):
    g = np.load(os.path.join(golden_dir, "evp_b3_stress_480x854.npz"))
    sd = S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=int(g["weight_seed"]), mode="stress")
    x, seg, flow = S.synth_frames(1, seed=int(g["input_seed"]), H=480, W=854)
    feats = EO.evp_forward(sd, CFG, x, seg, flow)
    assert np.abs(feats.numpy() - g["feats"]).max() < 1e-4


@pytest.mark.parametrize("f_maps", [32, 64])
@pytest.mark.parametrize("mode", ["ref_init", "stress", "phase"])
def test_mstcn_oracle_matches_golden(golden_dir, f_maps, mode):
    g = np.load(os.path.join(golden_dir, f"mstcn_f{f_maps}_{mode}_T700.npz"))
    sd = S.synth_mstcn_state_dict(2, 8, f_maps, 2048, 14, seed=int(g["weight_seed"]), mode=mode)
    feats = S.synth_lfb_features(int(g["T"]), seed=int(g["feat_seed"]))
    out = MO.mstcn_forward(sd, feats.unsqueeze(0).transpose(2, 1))
    scale = max(1.0, float(np.abs(g["logits"]).max()))
    assert np.abs(out.numpy() - g["logits"]).max() < 2e-5 * scale
    taps = MO.mstcn_forward_taps(sd, feats)  # the causal-tap form the CUDA kernel implements
    assert np.abs(taps.numpy() - g["logits"][:, 0]).max() < 1e-4 * scale


def test_mstcn_phase_weights_give_nondegenerate_argmax(golden_dir):
    g = np.load(os.path.join(golden_dir, "mstcn_f32_phase_T700.npz"))
    hist = np.bincount(g["logits"][-1, 0, :7].argmax(0), minlength=7)
    assert (hist > 0).sum() >= 5 and hist.max() < 0.6 * hist.sum()


def test_mstcn_causality():
    sd = S.synth_mstcn_state_dict(mode="stress")
    a = S.synth_lfb_features(600, seed=5)
    b = a.clone()
    b[400:] = S.synth_lfb_features(200, seed=6)
    oa, ob = MO.mstcn_forward_taps(sd, a), MO.mstcn_forward_taps(sd, b)
    assert torch.equal(oa[..., :400], ob[..., :400])


def test_oracle_matches_reference_known_answer():
    """Known answer of the reference's MS-TCN (SURVEY.md §8c): its own init under manual_seed(0), applied to a seeded 2 300-frame
    sequence, gives logits summing to -4348.2007 with mean |logit| 0.256878.  The drop-in module draws the same initial weights
    (tests/test_host_cpu.py), so the oracle must reproduce both numbers.  The EVP oracle is pinned to the reference's outputs by the
    golden tests above."""
    torch.manual_seed(0)
    sd = MultiStageModel_S(2, 8, 32, 2048, 14, True).state_dict()
    gen = torch.Generator().manual_seed(1234)
    xx = torch.randn(1, 2300, 2048, generator=gen).transpose(2, 1)
    with torch.no_grad():
        o = MO.mstcn_forward(sd, xx)
    assert abs(float(o.double().sum()) - (-4348.2007)) < 5e-3
    assert abs(float(o.abs().mean()) - 0.256878) < 1e-6
