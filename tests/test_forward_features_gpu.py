"""MixVisionTransformerEVP.forward_features on the GPU: the four fp32 NCHW stage maps of the encoder-only launch plans against the golden
vectors of the real reference and the fp32 oracle, bit-identity with the stage norm of the full forward, frame independence, no effect
on the plans of the full forward, the attention-map capture through `get_local`, the channel-major LayerNorm kernel, and errors."""
import ctypes
import os

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from oracle import evp_oracle as EO
from surgvid_b200 import _native, ops, visualizer
from surgvid_b200 import synthetic as S
from surgvid_b200.models import mix_transformer_evp as M

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
REL_L2_TOL = 1.5e-2
MAXABS_TOL = 3e-2
B3_224 = [(64, 56, 56), (128, 28, 28), (320, 14, 14), (512, 7, 7)]

_MODELS = {}


def _model(variant="mit_b3_evp", mode="stress"):
    key = (variant, mode)
    if key not in _MODELS:
        m = getattr(M, variant)()
        sd = S.synth_state_dict(S.evp_key_shapes(variant), seed=0, mode=mode)
        m.load_state_dict(sd, strict=True)
        _MODELS[key] = (m.to(DEV).eval(), sd)
    return _MODELS[key]


def _ff(m, x, seg, micro_batch=None):
    saved = m.micro_batch
    if micro_batch is not None:
        m.micro_batch = micro_batch
    try:
        with torch.no_grad():
            return m.forward_features(x.to(DEV), seg.to(DEV))
    finally:
        m.micro_batch = saved


def _oracle(sd, variant, x, seg, emulate_bf16=False):
    H, W = x.shape[-2:]
    return EO.forward_features(EO._Ctx(emulate_bf16), sd, S.EVP_CONFIGS[variant], x.reshape(-1, 3, H, W).float(),
                               seg.reshape(-1, 3, H, W).float())


def _check_stages(outs, refs, what):
    for s, (o, r) in enumerate(zip(outs, refs)):
        o = o.cpu()
        assert o.shape == r.shape, (what, s, o.shape, r.shape)
        rel = float((o - r).norm() / r.norm())
        mx = float((o - r).abs().max())
        print(f"[features] {what} stage {s + 1} {tuple(o.shape)}: rel-L2 {rel:.3e}  max-abs {mx:.3e}  (max|ref| {float(r.abs().max()):.3f})")
        assert rel <= REL_L2_TOL, (what, s, rel)
        assert mx <= MAXABS_TOL * float(r.abs().max()), (what, s, mx)


def _tap_sample(t, n=2048):
    flat = t.reshape(-1)
    idx = torch.linspace(0, flat.numel() - 1, n).long().to(flat.device)
    return flat[idx].float().cpu().numpy()


@pytest.mark.parametrize("mode", ["ref_init", "stress"])
def test_stage_maps_match_golden(golden_dir, mode):
    g = np.load(os.path.join(golden_dir, f"evp_b3_{mode}_224.npz"))
    m, _ = _model(mode=mode)
    x, seg, _ = S.synth_frames(int(g["n"]), seed=int(g["input_seed"]))
    outs = _ff(m, x, seg)
    assert [tuple(o.shape) for o in outs] == [(2,) + d for d in B3_224]
    for s, o in enumerate(outs):
        assert o.dtype == torch.float32 and o.is_cuda and o.is_contiguous()
        got, ref = _tap_sample(o.permute(0, 2, 3, 1)), g[f"stage{s + 1}_tokens"]
        rel = float(np.linalg.norm(got - ref) / np.linalg.norm(ref))
        print(f"[golden] {mode} stage {s + 1}: rel-L2 {rel:.3e}")
        assert rel < 3e-2, (s, rel)


def test_ragged_micro_batches_match_oracle():
    m, sd = _model()
    x, seg, _ = S.synth_frames(7, seed=101)
    outs = _ff(m, x, seg, micro_batch=3)
    _check_stages(outs, _oracle(sd, "mit_b3_evp", x, seg), "B=7 mb=3 vs oracle")
    for s, (o, r) in enumerate(zip(outs, _oracle(sd, "mit_b3_evp", x, seg, emulate_bf16=True))):
        print(f"[features] stage {s + 1} vs oracle with bf16 operands: rel-L2 {float((o.cpu() - r).norm() / r.norm()):.3e}")


def test_same_values_as_the_stage_norm_of_the_full_forward():
    m, _ = _model()
    x, seg, _ = (t.to(DEV) for t in S.synth_frames(3, seed=17))
    outs = _ff(m, x, seg, micro_batch=3)
    with torch.no_grad():
        m.extract_features(x, seg, None)
    for s, o in enumerate(outs):
        tap = m.read_tap(f"stage{s + 1}_tokens")
        assert torch.equal(o.permute(0, 2, 3, 1).reshape(-1).to(torch.bfloat16).float(), tap), s


def test_frames_are_independent():
    m, _ = _model()
    x, seg, _ = S.synth_frames(7, seed=101)
    outs = _ff(m, x, seg, micro_batch=3)
    alone = _ff(m, x[4:5], seg[4:5], micro_batch=3)
    for s in range(4):
        assert torch.equal(alone[s][0], outs[s][4]), s


def test_full_forward_plans_unchanged():
    m, _ = _model()
    x, seg, flow = (t.to(DEV) for t in S.synth_frames(3, seed=21))
    with torch.no_grad():
        f_flow = m.extract_features(x, seg, flow)
        n_flow = m.last_launch_count()
        f_none = m.extract_features(x, seg, None)
        n_none = m.last_launch_count()
        m.forward_features(x, seg)
        n_ff = m.last_launch_count()
        m.forward_features(x, seg)
        after_flow = m.extract_features(x, seg, flow)
        assert m.last_launch_count() == n_flow
        after_none = m.extract_features(x, seg, None)
        assert m.last_launch_count() == n_none
    assert torch.equal(after_flow, f_flow) and torch.equal(after_none, f_none)
    print(f"[launches] with flow {n_flow}, without flow {n_none}, forward_features {n_ff}")
    assert 0 < n_ff < n_none


def test_480x854_shapes_and_oracle():
    m, sd = _model()
    x, seg, _ = S.synth_frames(2, seed=5, H=480, W=854)
    outs = _ff(m, x, seg, micro_batch=1)
    assert [tuple(o.shape) for o in outs] == [(2, 64, 120, 214), (2, 128, 60, 107), (2, 320, 30, 54), (2, 512, 15, 27)]
    _check_stages(outs, _oracle(sd, "mit_b3_evp", x, seg), "480x854 mb=1 vs oracle")


@pytest.mark.parametrize("variant,hw", [("mit_b0_evp", (224, 224)), ("mit_b0_evp", (96, 160)), ("mit_b2_evp", (128, 128))])
def test_other_variants_match_oracle(variant, hw):
    """b0 (widths 32/64/160/256) takes the paths without im2col maps; b2 differs from b3 in depth only."""
    m, sd = _model(variant)
    x, seg, _ = S.synth_frames(3, seed=77, H=hw[0], W=hw[1])
    outs = _ff(m, x, seg)
    assert [tuple(o.shape)[1:] for o in outs] == m.stage_shapes(*hw)
    _check_stages(outs, _oracle(sd, variant, x, seg), f"{variant} {hw[0]}x{hw[1]} vs oracle")


def test_get_local_records_the_maps():
    m, _ = _model()
    gl = visualizer.get_local
    x, seg, _ = (t.to(DEV) for t in S.synth_frames(2, seed=41))
    with torch.no_grad():
        plain = m.forward_features(x, seg)
    saved = (dict(gl.cache), gl.is_activate)
    try:
        gl.cache.clear()
        gl.activate()
        with torch.no_grad():
            captured = m.forward_features(x, seg)
        cache = list(gl.cache["Attention.forward"])
    finally:
        gl.cache.clear()
        gl.cache.update(saved[0])
        gl.is_activate = saved[1]
    with torch.no_grad():
        _, maps = m.attention_maps(x, seg)
    assert len(cache) == len(maps) == sum(m.depths)
    for a, t in zip(cache, maps):
        assert isinstance(a, np.ndarray) and a.dtype == np.float32
        assert np.array_equal(a, t.cpu().numpy())
    assert all(torch.equal(a, b) for a, b in zip(captured, plain))


@pytest.mark.parametrize("C", [32, 64, 128, 160, 256, 320, 512])
def test_layernorm_nchw_op(C):
    g = torch.Generator(device="cpu").manual_seed(C)
    gamma = (1.0 + 0.5 * torch.randn(C, generator=g)).to(DEV)
    beta = (0.3 * torch.randn(C, generator=g)).to(DEV)
    for tokens in (49, 196, 405, 3136):
        for frames in (1, 3):   # 3 x 49 = 147 rows: not a multiple of any CTA tile (8 ... 128 rows)
            rows = frames * tokens
            x = (2.0 * torch.randn(rows, C, generator=g) + 0.7).to(DEV)
            out, ob = ops.layernorm_nchw(x, gamma, beta, 1e-6, tokens, want_bf16=True)
            ref_f32, ref_b16 = ops.layernorm(x, gamma, beta, 1e-6, want_f32=True, want_bf16=True)
            assert out.shape == (frames, C, tokens)
            assert torch.equal(out.permute(0, 2, 1).reshape(rows, C), ref_f32), (C, tokens, frames)
            assert torch.equal(ob, ref_b16), (C, tokens, frames)
            ref = torch.nn.functional.layer_norm(x.double(), (C,), gamma.double(), beta.double(), 1e-6)
            err = float((out.permute(0, 2, 1).reshape(rows, C).double() - ref).abs().max())
            assert err <= 4e-6 * float(ref.abs().max()), (C, tokens, frames, err)


def test_errors():
    m, _ = _model()
    x, seg, _ = S.synth_frames(2, seed=3)

    def message(fn, *args):
        with pytest.raises((RuntimeError, ValueError)) as e:
            fn(*args)
        return str(e.value)

    fwd = lambda a, b: m(a, b, return_features=True)  # noqa: E731
    assert message(m.forward_features, x, seg) == message(fwd, x, seg)  # CPU tensors
    bad_y = S.synth_frames(2, seed=3, H=112, W=112)[1].to(DEV)
    assert message(m.forward_features, x.to(DEV), bad_y) == message(fwd, x.to(DEV), bad_y)
    m.train()
    try:
        assert message(m.forward_features, x.to(DEV), seg.to(DEV)) == message(fwd, x.to(DEV), seg.to(DEV))
    finally:
        m.eval()
    with pytest.raises(ValueError, match="frames"):
        m.forward_features(x.to(DEV), seg[:1].to(DEV))

    # the C ABI checks sizes and alignment before the device is touched
    lib = _native.lib()
    xd, sd_ = x.to(DEV).contiguous(), seg.to(DEV).contiguous()
    st = m._state(xd.device)
    ws = m._workspace(st, xd.device, 2, 224, 224)
    outs = [torch.empty(2 * c * h * w + 1, device=DEV) for c, h, w in B3_224]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ptrs, elems, maps=None, maps_elems=0):
        return lib.sv_evp_forward_features(st["handle"], ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(sd_.data_ptr()),
                                           (ctypes.c_void_p * 4)(*ptrs), (ctypes.c_int64 * 4)(*elems), maps, maps_elems, 2, 224, 224, 2,
                                           ctypes.c_void_p(ws.data_ptr()), ws.numel(), stream)

    ptrs = [o.data_ptr() for o in outs]
    need = [2 * c * h * w for c, h, w in B3_224]
    assert call(ptrs, [need[0], need[1], need[2] - 1, need[3]]) == 1 and b"stage_out[2] too small" in lib.sv_last_error()
    assert call([ptrs[0], ptrs[1] + 2, ptrs[2], ptrs[3]], need) == 1 and b"aligned" in lib.sv_last_error()
    assert call([ptrs[0], None, ptrs[2], ptrs[3]], need) == 1 and b"NULL" in lib.sv_last_error()
    off, _ = m.attention_maps_layout(2, 224, 224)
    maps = torch.empty(off[-1] + 4, device=DEV)
    assert call(ptrs, need, ctypes.c_void_p(maps.data_ptr()), off[-1] - 1) == 1 and b"too small" in lib.sv_last_error()
    assert call(ptrs, need, ctypes.c_void_p(maps.data_ptr() + 4), off[-1]) == 1 and b"aligned" in lib.sv_last_error()
    assert call(ptrs, need) == 0
    torch.cuda.synchronize()
