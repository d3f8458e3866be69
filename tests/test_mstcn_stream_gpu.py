"""Online MS-TCN and Trans-SVNet head (`MultiStageModel_S.open_stream`, `Transformer.open_stream`): every streamed output is
`torch.equal` to the offline call over the same video's frames, whatever the chunk schedule."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native
from surgvid_b200 import synthetic as S
from surgvid_b200.mstcn import MultiStageModel_S
from surgvid_b200.trans_head import Transformer

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(f_maps=32, mode="phase", seed=1):
    m = MultiStageModel_S(2, 8, f_maps, 2048, 14, True)
    m.load_state_dict(S.synth_mstcn_state_dict(2, 8, f_maps, 2048, 14, seed=seed, mode=mode), strict=True)
    return m.to(DEV).eval()


def _head(m, f_maps=32, seed=21):
    head = Transformer(f_maps, 2048, 14, 30)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in head.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.05 if p.dim() == 2 and p.shape[1] == 2048 else 0.2))
    return head.to(DEV).eval()


def _feed(step, videos, schedules, rng=None):
    """Drive one stream per video: each step feeds a subset of the unfinished streams (all of them, in order, without rng) their next
    chunk; schedules[i] lists stream i's chunk sizes (the last repeats) or maps its position to one.  Returns, per stream, the
    concatenation of every output of `step`: logits over their last dim, the other outputs over rows."""
    n = len(videos)
    pos, nxt = [0] * n, [0] * n
    got = [[] for _ in range(n)]
    while True:
        live = [i for i in range(n) if pos[i] < videos[i].shape[0]]
        if not live:
            break
        ids = live if rng is None else rng.permutation(live)[: int(rng.integers(1, len(live) + 1))].tolist()
        counts = []
        for i in ids:
            sch = schedules[i]
            c = sch(pos[i]) if callable(sch) else sch[min(nxt[i], len(sch) - 1)]
            counts.append(int(min(c, videos[i].shape[0] - pos[i])))
            nxt[i] += 1
        outs = step(torch.cat([videos[i][pos[i]:pos[i] + c] for i, c in zip(ids, counts)]), ids, counts)
        outs = outs if isinstance(outs, tuple) else (outs,)
        o = 0
        for i, c in zip(ids, counts):
            got[i].append((outs[0][..., o:o + c],) + tuple(x[o:o + c] for x in outs[1:]))
            pos[i] += c
            o += c
    return [tuple(torch.cat([g[j] for g in parts], dim=-1 if j == 0 else 0) for j in range(len(parts[0]))) for parts in got]


SCHEDULES = [[1], [25], [509, 510, 511, 1021], lambda p: 1 + (p * 7919) % 97]


@pytest.mark.parametrize("f_maps", [32, 64])
@pytest.mark.parametrize("mode", ["ref_init", "stress", "phase"])
def test_stream_equals_offline(f_maps, mode):
    m = _model(f_maps, mode)
    lengths = [1100, 1300, 2600, 1700]
    videos = [S.synth_lfb_features(T, seed=40 + i).to(DEV) for i, T in enumerate(lengths)]
    st = m.open_stream(len(videos))
    got = _feed(lambda f, i, c: st.step(f, i, c), videos, SCHEDULES, np.random.default_rng(f_maps))
    for v, g in zip(videos, got):
        assert torch.equal(g[0], m.forward_videos(v, [v.shape[0]]))
    assert st.seen.tolist() == lengths


def test_nine_lengths_as_nine_streams_with_query():
    m = _model(32, "phase")
    head = _head(m)
    head.attach(m)
    lengths = [700, 1531, 64, 2300, 1, 3, 255, 511, 513]
    videos = [S.synth_lfb_features(T, seed=100 + i).to(DEV) for i, T in enumerate(lengths)]
    rng = np.random.default_rng(9)
    st = m.open_stream(len(videos))
    got = _feed(lambda f, i, c: st.step(f, i, c, query=True), videos, [lambda p: int(rng.integers(1, 300))] * 9, rng)
    for v, g in zip(videos, got):
        lg, q = m.forward_videos_query(v, [v.shape[0]])
        assert torch.equal(g[0], lg) and torch.equal(g[1], q)


def test_reset_after_extreme_features():
    m = _model(32, "stress")
    st = m.open_stream(3)
    wild = S.synth_lfb_features(900, seed=5).to(DEV) * 1e4
    wild[::7] = -wild[::7]
    st.step(wild, [1], [900])
    st.step(S.synth_lfb_features(40, seed=6).to(DEV), [0], [40])
    st.reset([1])
    assert st.seen.tolist() == [40, 0, 0]
    v = S.synth_lfb_features(600, seed=7).to(DEV)
    got = _feed(lambda f, i, c: st.step(f, [1], c), [v], [[13]])
    assert torch.equal(got[0][0], m.forward_videos(v, [600]))


def test_simt_layers_in_a_child_process():
    code = (
        "import sys, torch; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import test_mstcn_stream_gpu as t\n"
        "m = t._model(32, 'phase'); v = t.S.synth_lfb_features(1400, seed=3).to(t.DEV)\n"
        "st = m.open_stream(1); g = t._feed(lambda f, i, c: st.step(f, i, c), [v], [[1] * 40 + [509, 510, 511]])\n"
        "assert torch.equal(g[0][0], m.forward_videos(v, [1400]))\n"
        "print('ok')\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, SURGVID_MSTCN_TC="0")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


@pytest.mark.parametrize("schedule", [[29, 1, 1, 5, 40], [30, 1, 30], [31, 2, 17], [1]], ids=["cut29", "cut30", "cut31", "one_frame"])
def test_head_stream_windows(schedule):
    m = _model(32, "phase")
    head = _head(m)
    v = S.synth_lfb_features(150, seed=12).to(DEV)
    st = head.open_stream(m, 2)
    got = _feed(lambda f, i, c: st.step(f, i, c), [v, v[:77]], [schedule, [3]])
    for w, g in zip([v, v[:77]], got):
        lg, out = head.forward_videos(m, w, [w.shape[0]])
        assert torch.equal(g[0], lg)
        assert torch.equal(g[1], out)


def test_cholec80_80_streams_25_frames_per_step():
    m = _model(32, "phase")
    head = _head(m)
    L = [int(x) for x in S.cholec80_video_lengths()]
    allf = torch.rand(sum(L), 2048, device=DEV, generator=torch.Generator(DEV).manual_seed(80)) * 0.57
    lg_off, out_off = head.forward_videos(m, allf, L)
    videos = list(torch.split(allf, L))
    st = head.open_stream(m, 80)
    got = _feed(lambda f, i, c: st.step(f, i, c), videos, [[25]] * 80)
    assert torch.equal(torch.cat([g[0] for g in got], dim=2), lg_off)
    assert torch.equal(torch.cat([g[1] for g in got], dim=0), out_off)
    assert st.seen.tolist() == L


def test_argument_errors():
    m = _model(32, "phase")
    st = m.open_stream(3)
    f = S.synth_lfb_features(4, seed=1).to(DEV)
    with pytest.raises(RuntimeError, match="duplicate stream id"):
        st.step(f, [1, 1], [2, 2])
    with pytest.raises(RuntimeError, match="out of range"):
        st.step(f, [3], [4])
    with pytest.raises(RuntimeError, match="counts must be >= 1"):
        st.step(f, [0, 1], [4, 0])
    with pytest.raises(ValueError, match="sum\\(counts\\)"):
        st.step(f, [0], [3])
    lib = _native.lib()
    h = m._state(torch.device(DEV))["handle"]
    small = st._state.numel() - 1
    ids, cnt = (ctypes.c_int32 * 1)(0), (ctypes.c_int64 * 1)(4)
    out = torch.empty(2, 14, 4, device=DEV)
    ws = torch.empty(lib.sv_mstcn_stream_workspace_bytes(h, 4), dtype=torch.uint8, device=DEV)
    rc = lib.sv_mstcn_stream_step(h, ctypes.c_void_p(st._state.data_ptr()), small, 3, ctypes.c_void_p(f.data_ptr()), ids, cnt, 1,
                                  ctypes.c_void_p(out.data_ptr()), None, ctypes.c_void_p(ws.data_ptr()), ws.numel(), None)
    assert rc == 1 and b"state too small" in lib.sv_last_error()
    rc = lib.sv_mstcn_stream_step(h, ctypes.c_void_p(st._state.data_ptr()), st._state.numel(), 3, ctypes.c_void_p(f.data_ptr()), ids, cnt, 1,
                                  ctypes.c_void_p(out.data_ptr()), None, ctypes.c_void_p(ws.data_ptr()), ws.numel() - 1, None)
    assert rc == 1 and b"workspace too small" in lib.sv_last_error()
    cnt_big = (ctypes.c_int64 * 1)(1 << 31)
    rc = lib.sv_mstcn_stream_step(h, ctypes.c_void_p(st._state.data_ptr()), st._state.numel(), 3, ctypes.c_void_p(f.data_ptr()), ids, cnt_big, 1,
                                  ctypes.c_void_p(out.data_ptr()), None, ctypes.c_void_p(ws.data_ptr()), ws.numel(), None)
    assert rc == 1 and b"pass 2^31" in lib.sv_last_error()
    st.step(f, [0], [4])
    m.load_state_dict(S.synth_mstcn_state_dict(mode="stress"))   # stale weights
    with pytest.raises(RuntimeError, match="reset"):
        st.step(f, [0], [4])
    st.reset()
    assert st.seen.tolist() == [0, 0, 0]
    assert torch.equal(st.step(f, [2], [4]), m.forward_videos(f, [4]))
