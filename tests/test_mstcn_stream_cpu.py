"""The stream-state design of online MS-TCN, checked without a GPU: the float64 streaming restatement (tests/mstcn_stream_ref.py)
equals the offline model for every chunk schedule, and the new C ABI entry points refuse bad arguments before touching a device."""
import ctypes

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native
from surgvid_b200 import synthetic as S
from surgvid_b200.mstcn import MultiStageModel_S
from surgvid_b200.trans_head import Transformer
from mstcn_stream_ref import MstcnStreamRef, offline

RTOL = 1e-10


def _sd64(mode="phase", f_maps=32):
    sd = S.synth_mstcn_state_dict(2, 8, f_maps, 2048, 14, seed=1, mode=mode)
    return {k: v.double() for k, v in sd.items()}


def _close(got, want):
    scale = float(want.abs().max())
    err = float((got - want).abs().max())
    assert err <= RTOL * max(1.0, scale), (err, scale)


def _run(sd, feats, chunks):
    ref = MstcnStreamRef(sd, 1)
    outs, o = [], 0
    for c in chunks:
        outs.append(ref.step(feats[o:o + c], [0], [c]))
        o += c
    assert o == feats.shape[0] and ref.seen[0] == o
    return torch.cat(outs, dim=2)


def test_one_frame_steps_over_1100_frames():
    sd = _sd64()
    feats = S.synth_lfb_features(1100, seed=11).double()
    _close(_run(sd, feats, [1] * 1100), offline(sd, feats))


@pytest.mark.parametrize("chunk", [509, 510, 511, 1021])
def test_chunks_straddling_the_receptive_field(chunk):
    sd = _sd64("stress")
    T = 2 * chunk + 37
    feats = S.synth_lfb_features(T, seed=12).double()
    _close(_run(sd, feats, [chunk, chunk, 37]), offline(sd, feats))


def test_random_interleaved_chunks_with_reset():
    sd = _sd64()
    rng = np.random.default_rng(3)
    n = 5
    lengths = [300, 1, 777, 64, 520]
    videos = [S.synth_lfb_features(T, seed=20 + i).double() for i, T in enumerate(lengths)]
    ref = MstcnStreamRef(sd, n)
    pos = [0] * n
    got = [[] for _ in range(n)]
    reset_done = False
    second = S.synth_lfb_features(400, seed=99).double()
    while any(pos[i] < videos[i].shape[0] for i in range(n)):
        live = [i for i in range(n) if pos[i] < videos[i].shape[0]]
        ids = list(rng.permutation(live)[: rng.integers(1, len(live) + 1)])
        counts = [int(min(rng.integers(1, 90), videos[i].shape[0] - pos[i])) for i in ids]
        feats = torch.cat([videos[i][pos[i]:pos[i] + c] for i, c in zip(ids, counts)])
        out = ref.step(feats, ids, counts)
        o = 0
        for i, c in zip(ids, counts):
            got[i].append(out[:, :, o:o + c])
            pos[i] += c
            o += c
        if not reset_done and pos[2] >= 300:   # stream 2 switches to a new video mid-way
            reset_done = True
            ref.reset([2])
            videos[2], pos[2], got[2] = second, 0, []
    for i in range(n):
        _close(torch.cat(got[i], dim=2), offline(sd, videos[i]))


def test_stream_state_size():
    lib = _native.lib()
    assert lib.sv_mstcn_stream_state_bytes(None, 4) == 0


def test_stream_abi_rejects_bad_arguments_without_a_device():
    lib = _native.lib()
    ids = (ctypes.c_int32 * 1)(0)
    cnt = (ctypes.c_int64 * 1)(1)
    assert lib.sv_mstcn_stream_step(None, None, 0, 1, None, ids, cnt, 1, None, None, None, 0, None) == 1
    assert b"null" in lib.sv_last_error()
    assert lib.sv_mstcn_stream_reset(None, None, 0, 1, None, 0, None) == 1
    assert b"null" in lib.sv_last_error()
    assert lib.sv_trans_stream_forward(None, None, 0, 1, None, 1, None, ids, cnt, 1, None, None) == 1
    assert b"null" in lib.sv_last_error()
    assert lib.sv_trans_stream_reset(None, None, 0, 1, None, 0, None) == 1
    assert b"null" in lib.sv_last_error()
    assert lib.sv_mstcn_stream_workspace_bytes(None, 10) == 0
    assert lib.sv_trans_stream_state_bytes(None, 3) == 0


def test_open_stream_on_a_cpu_model_has_no_cpu_path():
    m = MultiStageModel_S(2, 8, 32, 2048, 14, True).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.open_stream(4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        Transformer(32, 2048, 14, 30).eval().open_stream(m, 4)
    with pytest.raises(RuntimeError, match="inference-only"):
        m.train().open_stream(4)
