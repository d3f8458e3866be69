"""Attention-map capture on the GPU: `sv_op_attention_probs` against float64 softmax(Q K^T * scale) of the same bf16 operands, the
capture forward against the reference maps of tests/attn_maps_ref.py, features unchanged by the capture, invariance of the maps to
micro-batching and batch composition, the `get_local` drop-in, and argument errors."""
import ctypes

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native, ops, visualizer
from surgvid_b200 import synthetic as S
from surgvid_b200.models.mix_transformer_evp import mit_b0_evp, mit_b3_evp
import attn_ref as AR
from attn_maps_ref import encoder_maps

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Gate of the op (fp32 probabilities, fp32 accumulation of the bf16 products, exp2 with log2(e) folded into the scale).
# Largest honest errors measured on one B200 (1000 W power limit) over these cases: max-abs 4.6e-6 and row-sum error 4.6e-6 (both on
# plant_first, where one probability is ~1).  The gate sits 4.3x above them and 475x below the smallest error of a softmax whose scale
# is 2 % off (9.5e-3, test_probs_gate_rejects_a_scale_bug).
PROBS_MAX_ABS = 2e-5
PROBS_ROWSUM = 2e-5
# Model maps vs the oracle with bf16-rounded operands (activations round to bf16 in different places), per block.  Measured worst on the
# same B200: rel-L2 6.9e-3, max-abs 3.7e-3, argmax agreement 0.965 (near-tied rows of the 480x854 stage-3 blocks); a map of the wrong
# block, head or frame agrees on about 1/N_kv of the rows.
MODEL_REL_L2 = 2e-2
MODEL_MAX_ABS = 1.5e-2
MODEL_ARGMAX_AGREE = 0.90

NKV = (1, 49, 63, 64, 65, 390, 405, 448, 500)
NQ = (1, 49, 65, 127, 196, 3136)


def _strided(x: torch.Tensor) -> torch.Tensor:
    """The same values in a buffer of row stride 2C (the layout of the kv / q buffers of the model)."""
    buf = torch.full((x.shape[0], 2 * x.shape[1]), float("nan"), dtype=x.dtype, device=x.device)
    buf[:, :x.shape[1]] = x
    return buf[:, :x.shape[1]]


def _ref_probs(q, k, B, heads, hd, scale):
    Q, K = (AR._heads_view(t, B, heads, hd).double() for t in (q, k))
    return torch.softmax((Q @ K.transpose(-1, -2)) * scale, dim=-1)


def _errors(p, ref):
    assert bool(torch.isfinite(p).all()), "non-finite probabilities"
    return float((p.double() - ref).abs().max()), float((p.double().sum(-1) - 1.0).abs().max())


@pytest.mark.parametrize("hd", [32, 64])
def test_probs_op_matches_float64(hd):
    B, heads = 2, 2
    worst = {}
    for Nkv in NKV:
        for Nq in NQ:
            for kind in AR.STRESS:
                if kind == "bigv" or (kind != "randn" and Nq > 196):
                    continue  # bigv only changes V; the 3136-row cases run on randn
                q, k, _ = AR.make_inputs(kind, B, heads, Nq, Nkv, hd, seed=Nkv * 7 + Nq, device=DEV)
                q, k = _strided(q), _strided(k)
                scale = hd ** -0.5
                p = ops.attention_probs(q, k, B, heads, Nq, Nkv, hd, scale)
                ref = _ref_probs(q, k, B, heads, hd, scale)
                mx, rs = _errors(p, ref)
                w = worst.setdefault(kind, [0.0, 0.0])
                w[0], w[1] = max(w[0], mx), max(w[1], rs)
                assert mx <= PROBS_MAX_ABS and rs <= PROBS_ROWSUM, (kind, Nq, Nkv, mx, rs)
    print(f"[probs] hd {hd} worst max-abs / row-sum error per input kind: " +
          ", ".join(f"{k} {v[0]:.2e}/{v[1]:.2e}" for k, v in worst.items()))


def test_probs_gate_rejects_a_scale_bug():
    """softmax with the scale off by 2 % (a bug the attention gate also targets) is far outside the op's gate."""
    for hd in (32, 64):
        for Nkv in (49, 405):
            q, k, _ = AR.make_inputs("randn", 2, 2, 196, Nkv, hd, seed=3, device=DEV)
            ref = _ref_probs(q, k, 2, 2, hd, hd ** -0.5)
            bug = _ref_probs(q, k, 2, 2, hd, 1.02 * hd ** -0.5)
            mx = float((bug - ref).abs().max())
            print(f"[probs] scale x1.02 hd {hd} Nkv {Nkv}: max-abs {mx:.2e} = {mx / PROBS_MAX_ABS:.0f}x the gate")
            assert mx > 20 * PROBS_MAX_ABS


_MODELS = {}


def _model(variant="mit_b3_evp"):
    if variant not in _MODELS:
        m = mit_b3_evp() if variant == "mit_b3_evp" else mit_b0_evp()
        sd = S.synth_state_dict(S.evp_key_shapes(variant), seed=0, mode="stress")
        m.load_state_dict(sd, strict=True)
        _MODELS[variant] = (m.to(DEV).eval(), sd)
    return _MODELS[variant]


@pytest.mark.parametrize("variant,H,W,n,with_flow", [
    ("mit_b3_evp", 224, 224, 2, True),
    ("mit_b3_evp", 224, 224, 2, False),
    ("mit_b0_evp", 224, 224, 2, True),
    ("mit_b3_evp", 480, 854, 2, True),
])
def test_model_maps_match_oracle(variant, H, W, n, with_flow):
    m, sd = _model(variant)
    x, seg, flow = S.synth_frames(n, seed=11, H=H, W=W)
    with torch.no_grad():
        feats, maps = m.attention_maps(x.to(DEV), seg.to(DEV), flow.to(DEV) if with_flow else None)
        plain = m(x.to(DEV), seg.to(DEV), flow.to(DEV) if with_flow else None, return_features=True)
    assert torch.equal(feats, plain)
    ref, _ = encoder_maps(sd, S.EVP_CONFIGS[variant], x, seg, emulate_bf16=True)
    assert len(maps) == len(ref) == sum(S.EVP_CONFIGS[variant]["depths"])
    worst = [0.0, 0.0, 1.0]
    for i, (got, r) in enumerate(zip(maps, ref)):
        got = got.cpu()
        assert got.shape == r.shape and bool(torch.isfinite(got).all())
        rel = float((got - r).norm() / r.norm())
        mx = float((got - r).abs().max())
        agree = float((got.argmax(-1) == r.argmax(-1)).float().mean())
        worst = [max(worst[0], rel), max(worst[1], mx), min(worst[2], agree)]
        assert rel <= MODEL_REL_L2 and mx <= MODEL_MAX_ABS and agree >= MODEL_ARGMAX_AGREE, (i, rel, mx, agree)
        assert float((got.sum(-1) - 1).abs().max()) <= PROBS_ROWSUM
    print(f"[maps] {variant} {H}x{W} flow={with_flow}: worst block rel-L2 {worst[0]:.2e}, max-abs {worst[1]:.2e}, "
          f"argmax agreement {worst[2]:.4f}")


def test_capture_leaves_features_and_plain_plans_unchanged():
    m, _ = _model()
    x, seg, flow = (t.to(DEV) for t in S.synth_frames(3, seed=21))
    with torch.no_grad():
        before = m(x, seg, flow, return_features=True)
        n_plain = m.last_launch_count()
        feats, _ = m.attention_maps(x, seg, flow)
        n_capture = m.last_launch_count()
        after = m(x, seg, flow, return_features=True)
    assert torch.equal(feats, before) and torch.equal(after, before)
    assert m.last_launch_count() == n_plain
    assert n_capture == n_plain + sum(m.depths)


def test_maps_invariant_to_micro_batch_calls_and_batch_composition():
    m, _ = _model()
    B = 10
    x, seg, flow = (t.to(DEV) for t in S.synth_frames(B, seed=31))
    runs = []
    try:
        for mb in (3, 7, B, B):  # ragged micro-batches; the last two are two calls with the same plans
            m.micro_batch = mb
            with torch.no_grad():
                runs.append(m.attention_maps(x, seg, flow))
        m.micro_batch = B
        with torch.no_grad():
            alone = m.attention_maps(x[6:7], seg[6:7], flow[6:7])
    finally:
        m.micro_batch = 1159
    f0, maps0 = runs[0]
    for f, maps in runs[1:]:
        assert torch.equal(f, f0)
        assert all(torch.equal(a, b) for a, b in zip(maps, maps0))
    assert torch.equal(alone[0][0], f0[6])
    assert all(torch.equal(a[0], b[6]) for a, b in zip(alone[1], maps0))


def test_get_local_drop_in():
    m, _ = _model()
    gl = visualizer.get_local
    x, seg, flow = (t.to(DEV) for t in S.synth_frames(1, seed=41))
    saved = (dict(gl.cache), gl.is_activate)
    try:
        gl.cache.clear()
        gl.activate()
        with torch.no_grad():
            feats = m(x, seg, flow, return_features=True)
        cache = gl.cache["Attention.forward"]
        assert len(cache) == 28
        with torch.no_grad():
            f2, maps = m.attention_maps(x, seg, flow)
        assert torch.equal(feats, f2)
        for a, t in zip(cache, maps):
            assert isinstance(a, np.ndarray) and a.dtype == np.float32 and a.shape == tuple(t.shape)
            assert np.array_equal(a, t.cpu().numpy())
        assert [a.shape for a in cache] == [(1, 1, 3136, 49)] * 3 + [(1, 2, 784, 49)] * 4 + [(1, 5, 196, 49)] * 18 + [(1, 8, 49, 49)] * 3
        gl.clear()
        assert gl.cache["Attention.forward"] == []
    finally:
        gl.cache.clear()
        gl.cache.update(saved[0])
        gl.is_activate = saved[1]


def test_argument_errors():
    m, _ = _model()
    lib = _native.lib()
    x, seg, _ = (t.to(DEV) for t in S.synth_frames(1, seed=51))
    x, seg = x.reshape(1, 3, 224, 224), seg.reshape(1, 3, 224, 224)
    m.attention_maps(x, seg)  # packs the weights
    st = m._native[torch.device(DEV).index or 0]
    off, _ = m.attention_maps_layout(1, 224, 224)
    ws = next(iter(st["workspace"].values()))
    out = torch.empty(1, 2048, device=DEV)
    maps = torch.empty(off[-1] + 4, device=DEV)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ptr, elems):
        return lib.sv_evp_forward_attention(st["handle"], ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(seg.data_ptr()), None,
                                            ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ptr), elems, 1, 224, 224, 1,
                                            ctypes.c_void_p(ws.data_ptr()), ws.numel(), stream)

    assert call(maps.data_ptr(), off[-1] - 1) == 1 and b"too small" in lib.sv_last_error()
    assert call(maps.data_ptr() + 4, off[-1]) == 1 and b"aligned" in lib.sv_last_error()
    assert call(maps.data_ptr(), off[-1]) == 0
    torch.cuda.synchronize()
    q, k, _ = AR.make_inputs("randn", 1, 2, 49, 49, 40, device=DEV)
    with pytest.raises(RuntimeError, match="head_dim"):
        ops.attention_probs(q, k, 1, 2, 49, 49, 40, 40 ** -0.5)
    q, k, _ = AR.make_inputs("randn", 1, 2, 49, 49, 64, device=DEV)
    p = torch.empty(2 * 49 * 49 + 1, device=DEV)
    rc = lib.sv_op_attention_probs(ctypes.c_void_p(q.data_ptr()), 128, ctypes.c_void_p(k.data_ptr() + 2), 128, 1, 2, 49, 49, 64, 0.125,
                                   ctypes.c_void_p(p.data_ptr()), stream)
    assert rc == 1 and b"alignment" in lib.sv_last_error()
