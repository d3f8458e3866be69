"""Host plumbing shared by the native handles, called through the C ABI: the stream-state registry behind sv_trans_stream_reset /
sv_trans_stream_forward (the MS-TCN side is covered by test_mstcn_stream_gpu.py), and the state-dict store behind every
sv_*_set_tensor / sv_*_pack_weights."""
import ctypes

import numpy as np
import pytest
import torch

import surgvid_b200  # noqa: F401
from surgvid_b200 import _native
from surgvid_b200 import synthetic as S
from surgvid_b200.trans_head import Transformer

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SV_ERR_INVALID, SV_ERR_STATE = 1, 3
N_STREAMS = 3


@pytest.fixture(scope="module")
def trans():
    """A packed head handle, its state size for N_STREAMS streams and device buffers for a step's operands."""
    head = Transformer(32, 2048, 14, 30).to(DEV).eval()
    lib = _native.lib()
    h = head.transformer._state(torch.device(DEV))["handle"]
    need = int(lib.sv_trans_stream_state_bytes(h, N_STREAMS))
    bufs = {"logits": torch.zeros(14, 64, device=DEV), "query": torch.zeros(64, 14, device=DEV), "out": torch.zeros(64, 14, device=DEV)}
    yield head, h, need, bufs
    torch.cuda.synchronize()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _ids(*v):
    return (ctypes.c_int32 * len(v))(*v)


def _reset(h, state, nbytes, n_streams, ids=None):
    return _native.lib().sv_trans_stream_reset(h, _ptr(state), nbytes, n_streams, ids, 0 if ids is None else len(ids), None)


def _forward(h, bufs, state, nbytes, n_streams, ids, counts):
    cnt = (ctypes.c_int64 * len(counts))(*counts)
    return _native.lib().sv_trans_stream_forward(h, _ptr(state), nbytes, n_streams, _ptr(bufs["logits"]), bufs["logits"].stride(0),
                                                 _ptr(bufs["query"]), ids, cnt, len(counts), _ptr(bufs["out"]), None)


def _expect(rc, status, text):
    msg = _native.lib().sv_last_error().decode()
    assert rc == status and msg.startswith(text), (rc, msg)


def test_trans_stream_argument_errors(trans):
    _, h, need, bufs = trans
    state = torch.empty(need, dtype=torch.uint8, device=DEV)
    # a state this handle never reset
    _expect(_forward(h, bufs, state, need, N_STREAMS, _ids(0), [4]), SV_ERR_STATE, "trans stream: the state was not reset through this handle")
    _expect(_reset(h, state, need, N_STREAMS, _ids(0)), SV_ERR_STATE, "trans stream: reset every stream of a new state (stream_ids = NULL) first")
    # state too small
    _expect(_reset(h, state, need - 1, N_STREAMS), SV_ERR_INVALID, "trans stream: state too small")
    assert _reset(h, state, need, N_STREAMS) == 0
    _expect(_forward(h, bufs, state, need - 1, N_STREAMS, _ids(0), [4]), SV_ERR_INVALID, "trans stream: state too small")
    # n_streams differs from the last full reset
    _expect(_forward(h, bufs, state, need, N_STREAMS - 1, _ids(0), [4]), SV_ERR_INVALID,
            "trans stream: n_streams differs from the state's last full reset")
    _expect(_reset(h, state, need, N_STREAMS - 1, _ids(0)), SV_ERR_INVALID, "trans stream: n_streams differs from the state's last full reset")
    # stream ids and counts
    _expect(_forward(h, bufs, state, need, N_STREAMS, _ids(1, 1), [2, 2]), SV_ERR_INVALID, "trans stream: duplicate stream id")
    _expect(_reset(h, state, need, N_STREAMS, _ids(1, 1)), SV_ERR_INVALID, "trans stream: duplicate stream id")
    _expect(_forward(h, bufs, state, need, N_STREAMS, _ids(N_STREAMS), [4]), SV_ERR_INVALID, "trans stream: stream id out of range")
    _expect(_reset(h, state, need, N_STREAMS, _ids(-1)), SV_ERR_INVALID, "trans stream: stream id out of range")
    _expect(_forward(h, bufs, state, need, N_STREAMS, _ids(0, 1), [4, 0]), SV_ERR_INVALID, "trans stream: counts must be >= 1")
    _expect(_forward(h, bufs, state, need, N_STREAMS, _ids(0), [1 << 31]), SV_ERR_INVALID, "trans stream: a stream position would pass 2^31")
    # none of the refused calls touched the state: a valid step and a partial reset still go through
    assert _forward(h, bufs, state, need, N_STREAMS, _ids(2, 0), [3, 5]) == 0
    assert _reset(h, state, need, N_STREAMS, _ids(2)) == 0
    torch.cuda.synchronize()
    assert state[:16].view(torch.int64).tolist() == [5, 0]


def _evp_handle():
    c = S.EVP_CONFIGS["mit_b0_evp"]
    cfg = _native.EvpCfg()
    for s in range(4):
        cfg.embed_dims[s], cfg.num_heads[s], cfg.depths[s], cfg.sr_ratios[s] = c["embed_dims"][s], c["num_heads"][s], c["depths"][s], c["sr_ratios"][s]
    cfg.mlp_ratio, cfg.embedding_dim, cfg.fold_head = 4, 2048, 0
    return cfg, S.synth_state_dict(S.evp_key_shapes("mit_b0_evp"), seed=0), "evp"


def _mstcn_handle():
    return _native.MstcnCfg(2, 8, 32, 2048, 14, 1), S.synth_mstcn_state_dict(2, 8, 32, 2048, 14, seed=1), "mstcn"


def _trans_handle():
    head = Transformer(32, 2048, 14, 30).transformer
    cfg = _native.TransCfg(head.d_model, head.d_ff, head.d_k, head.d_v, head.n_layers, head.n_heads, head.len_q)
    return cfg, head.state_dict(), "trans"


@pytest.fixture(params=[_evp_handle, _mstcn_handle, _trans_handle], ids=["evp", "mstcn", "trans"])
def handle(request):
    """(C ABI prefix, fresh handle, its state dict); the handle is destroyed afterwards."""
    cfg, sd, kind = request.param()
    lib = _native.lib()
    h = ctypes.c_void_p()
    torch.cuda.set_device(DEV)
    _native.check(getattr(lib, f"sv_{kind}_create")(ctypes.byref(cfg), ctypes.byref(h)), f"sv_{kind}_create")
    yield kind, h, sd
    getattr(_native.lib(), f"sv_{kind}_destroy")(h)


def test_set_tensor_rejects_bad_shapes(handle):
    kind, h, _ = handle
    set_tensor = getattr(_native.lib(), f"sv_{kind}_set_tensor")
    data = np.zeros(4, dtype=np.float32)
    ptr = data.ctypes.data_as(ctypes.c_void_p)
    assert set_tensor(h, b"x", ptr, None, 1) == SV_ERR_INVALID
    assert set_tensor(h, b"x", ptr, (ctypes.c_int64 * 2)(2, -2), 2) == SV_ERR_INVALID
    assert set_tensor(h, b"x", ptr, (ctypes.c_int64 * 2)(2, 2), 2) == 0


def test_pack_weights_missing_key_and_wrong_shape(handle):
    kind, h, sd = handle
    lib = _native.lib()
    set_tensor, pack = getattr(lib, f"sv_{kind}_set_tensor"), getattr(lib, f"sv_{kind}_pack_weights")
    names = list(sd)
    victim = next(n for n in names if n.endswith("weight") and sd[n].dim() >= 2)
    _native.set_tensors(set_tensor, h, [(n, sd[n]) for n in names if n != victim], "set_tensor")
    rc = pack(h)
    msg = lib.sv_last_error().decode()
    assert rc == SV_ERR_STATE and "missing state_dict key" in msg and victim in msg, (rc, msg)
    _native.set_tensors(set_tensor, h, [(victim, sd[victim].reshape(-1))], "set_tensor")
    rc = pack(h)
    msg = lib.sv_last_error().decode()
    # EVP reports every packing error as SV_ERR_STATE, MS-TCN and the head a wrong shape as SV_ERR_INVALID
    assert rc == (SV_ERR_STATE if kind == "evp" else SV_ERR_INVALID) and "wrong shape" in msg and victim in msg, (rc, msg)
    _native.set_tensors(set_tensor, h, [(victim, sd[victim])], "set_tensor")
    assert pack(h) == 0
