"""Trans-SVNet head at d_k = d_v = 64 (`Transformer(64, ...)`, the reference's mstcn_f_maps 64 configuration) on the GPU: the inner
module against the unpinned oracle restatement, the full head against the reference call site, streaming against the offline call,
and the configurations that stay unsupported."""
import ctypes

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from oracle import trans_head_oracle as tho
from surgvid_b200 import _native
from surgvid_b200 import synthetic as S
from surgvid_b200.mstcn import MultiStageModel_S
from surgvid_b200.trans_head import Transformer, Transformer2_3_1

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SV_ERR_UNSUPPORTED = 4


def _randomize(m, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("layer_norm.weight"):
                p.copy_(1.0 + 0.2 * torch.randn(p.shape, generator=g))
            elif n.endswith("bias"):
                p.copy_(0.3 * torch.randn(p.shape, generator=g))
            elif n == "fc.weight":   # the query projection of the LFB features
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
            else:
                p.copy_(torch.randn(p.shape, generator=g) * (1.5 / p.shape[1] ** 0.5))
    return m


def _inner(d_ff=64, len_q=30, bias=True, seed=11):
    m = Transformer2_3_1(d_model=14, d_ff=d_ff, d_k=64, d_v=64, n_layers=1, n_heads=4, len_q=len_q, bias=bias)
    return _randomize(m, seed).to(DEV).eval()


def _tcn(f_maps, seed=3):
    m = MultiStageModel_S(2, 8, f_maps, 2048, 14, True)
    m.load_state_dict(S.synth_mstcn_state_dict(2, 8, f_maps, 2048, 14, seed=seed, mode="phase"), strict=True)
    return m.to(DEV).eval()


def _head(seed=21):
    return _randomize(Transformer(64, 2048, 14, 30), seed).to(DEV).eval()


@pytest.mark.parametrize("len_q", [30, 32])
@pytest.mark.parametrize("bias,d_ff", [(True, 64), (False, 64), (True, 32)], ids=["bias", "no_bias", "d_ff32"])
def test_inner_dk64_matches_oracle(bias, d_ff, len_q):
    m = _inner(d_ff, len_q, bias, seed=11 + d_ff + len_q)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(3)
    lengths = [1, 29, 30, 31, 200, 7]
    T = sum(lengths)
    logits = 3.0 * torch.randn(14, T, generator=g)
    query = torch.tanh(torch.randn(T, 14, generator=g))
    out = m.forward_fused(logits.to(DEV), query.to(DEV), lengths)
    torch.cuda.synchronize()
    assert out.shape == (T, 1, 14)
    o, worst = 0, 0.0
    for Tv in lengths:
        inputs, _ = tho.original_forward_inputs(logits[:, o:o + Tv].unsqueeze(0), torch.zeros(1, Tv, 8), torch.zeros(14, 8), len_q)
        ref = tho.transformer2_3_1_forward(sd, inputs, query[o:o + Tv].unsqueeze(1), 4, 64, 64)
        worst = max(worst, float((out[o:o + Tv].cpu() - ref).abs().max()))
        # the reference's own call form: windows + query of ONE video
        assert torch.equal(m(inputs.to(DEV), query[o:o + Tv].unsqueeze(1).to(DEV)), out[o:o + Tv])
        o += Tv
    print(f"[parity] Transformer2_3_1 d_k=64 (bias={bias}, d_ff={d_ff}, len_q={len_q}) vs unpinned oracle: max-abs {worst:.3e}")
    assert worst <= 2e-4


@pytest.mark.parametrize("f_maps", [64, 32])
def test_full_head_dk64_forward_videos_and_reference_call_site(f_maps):
    """trans_SV_output.py:268-301 with a head built for mstcn_f_maps 64, on the logits of either MS-TCN width."""
    tcn = _tcn(f_maps)
    head = _head()
    lengths = [45, 300, 29, 1]
    T = sum(lengths)
    lfb = S.synth_lfb_features(T, seed=9).to(DEV)
    logits, out = head.forward_videos(tcn, lfb, lengths)
    assert logits.shape == (2, 14, T) and out.shape == (T, 1, 14)
    sd = {k: v.detach().cpu() for k, v in head.transformer.state_dict().items()}
    o, worst = 0, 0.0
    for Tv in lengths:
        video_fe = lfb[o:o + Tv].unsqueeze(0).transpose(2, 1)
        x = tcn(video_fe)[-1]                                            # [1, 14, Tv]
        y = head(x.detach(), lfb[o:o + Tv].unsqueeze(0))                  # [Tv, 1, 14]
        assert torch.equal(y, out[o:o + Tv])
        inputs, feas = tho.original_forward_inputs(x.cpu(), lfb[o:o + Tv].cpu().unsqueeze(0), head.fc.weight.detach().cpu(), 30)
        ref = tho.transformer2_3_1_forward(sd, inputs, feas, 4, 64, 64)
        worst = max(worst, float((y.cpu() - ref).abs().max()))
        o += Tv
    print(f"[parity] Transformer(64, ...) on MS-TCN f_maps {f_maps} vs unpinned oracle: max-abs {worst:.3e}")
    assert worst <= 3e-4


def _feed(st, videos, schedules, rng=None, reset_at=None):
    """Step one stream per video until all are done; each step feeds every unfinished stream (or, with rng, a random subset in random
    order) its next chunk (schedules[i]: chunk sizes, the last repeating).  reset_at = (i, frame): when stream i has been fed at least
    `frame` frames, it is reset and restarts its video.  Returns per stream the concatenated (logits, head_out) since its last reset."""
    n = len(videos)
    pos, nxt = [0] * n, [0] * n
    got = [[] for _ in range(n)]
    while True:
        if reset_at is not None and pos[reset_at[0]] >= reset_at[1]:
            st.reset([reset_at[0]])
            pos[reset_at[0]], nxt[reset_at[0]], got[reset_at[0]] = 0, 0, []
            reset_at = None
        live = [i for i in range(n) if pos[i] < videos[i].shape[0]]
        if not live:
            break
        ids = live if rng is None else rng.permutation(live)[: int(rng.integers(1, len(live) + 1))].tolist()
        counts = []
        for i in ids:
            sch = schedules[i]
            counts.append(int(min(sch[min(nxt[i], len(sch) - 1)], videos[i].shape[0] - pos[i])))
            nxt[i] += 1
        lg, out = st.step(torch.cat([videos[i][pos[i]:pos[i] + c] for i, c in zip(ids, counts)]), ids, counts)
        o = 0
        for i, c in zip(ids, counts):
            got[i].append((lg[..., o:o + c], out[o:o + c]))
            pos[i] += c
            o += c
    return [(torch.cat([a for a, _ in g], dim=-1), torch.cat([b for _, b in g], dim=0)) for g in got]


RAGGED = [3, 1, 29, 30, 31, 2, 64, 17]


@pytest.mark.parametrize("f_maps", [64, 32])
@pytest.mark.parametrize("plan", ["one_frame", "chunks25", "ragged", "interleaved", "reset_mid_video"])
def test_stream_dk64_equals_offline(f_maps, plan):
    tcn = _tcn(f_maps)
    head = _head()
    lengths = [150, 77, 260] if plan != "one_frame" else [70, 45]
    videos = [S.synth_lfb_features(T, seed=60 + i).to(DEV) for i, T in enumerate(lengths)]
    st = head.open_stream(tcn, len(videos))
    sched = {"one_frame": [[1]] * 2, "chunks25": [[25]] * 3, "ragged": [RAGGED, RAGGED[::-1], [31]],
             "interleaved": [RAGGED, [1], [25]], "reset_mid_video": [[25], [7], RAGGED]}[plan]
    rng = np.random.default_rng(f_maps) if plan in ("interleaved", "reset_mid_video") else None
    got = _feed(st, videos, sched, rng, reset_at=(2, 100) if plan == "reset_mid_video" else None)
    for v, (lg, out) in zip(videos, got):
        lg_off, out_off = head.forward_videos(tcn, v, [v.shape[0]])
        assert torch.equal(lg, lg_off)
        assert torch.equal(out, out_off)
    assert st.seen.tolist() == lengths


def test_stream_dk64_stale_weights_until_reset():
    tcn = _tcn(64)
    head = _head()
    st = head.open_stream(tcn, 2)
    f = S.synth_lfb_features(40, seed=2).to(DEV)
    st.step(f, [0], [40])
    head.transformer.load_state_dict(_randomize(Transformer(64, 2048, 14, 30), 99).transformer.state_dict())
    with pytest.raises(RuntimeError, match="reset"):
        st.step(f, [1], [40])
    st.reset()
    _, out = st.step(f, [1], [40])
    assert torch.equal(out, head.forward_videos(tcn, f, [40])[1])


@pytest.mark.parametrize("d_k,d_v,n_heads", [(48, 48, 4), (64, 32, 4), (64, 64, 8)], ids=["d_k48", "d_k_ne_d_v", "n_heads8"])
def test_unsupported_configurations_stay_rejected(d_k, d_v, n_heads):
    lib = _native.lib()
    cfg = _native.TransCfg(14, 64, d_k, d_v, 1, n_heads, 30)
    h = ctypes.c_void_p()
    assert lib.sv_trans_create(ctypes.byref(cfg), ctypes.byref(h)) == SV_ERR_UNSUPPORTED
    assert b"d_k = d_v = 32 or 64" in lib.sv_last_error()
    m = Transformer2_3_1(d_model=14, d_ff=64, d_k=d_k, d_v=d_v, n_layers=1, n_heads=n_heads, len_q=30).to(DEV).eval()
    with pytest.raises(RuntimeError, match="status 4"):
        m.forward_fused(torch.zeros(14, 5, device=DEV), torch.zeros(5, 14, device=DEV), [5])
