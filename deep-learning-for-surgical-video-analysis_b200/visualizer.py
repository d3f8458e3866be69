"""Drop-in for the reference's `visualizer.py` (`from visualizer import get_local`, used by `vs_attn.py` and as the decorator of
`Attention.forward` in mix_transformer_evp.py:109).

The semantics follow the upstream Visualizer `get_local` that the reference copies: `get_local('attn')` decorates a function;
after `get_local.activate()` every call appends the decorated function's local `attn` (`attn.detach().cpu().numpy()`) to
`get_local.cache[func.__qualname__]`; `get_local.clear()` empties the lists.  The reference's own `visualizer.py` is not part of
this repository, so these semantics are not pinned against that file.

Here the encoder runs in native kernels and no Python `Attention.forward` exists to decorate, so:
  * the decorator returns the function unchanged (no bytecode rewriting; the `bytecode` package is not needed);
  * while `get_local.is_activate` is true, `MixVisionTransformerEVP.forward` (and so `lfb.LFBExtractor`) runs the capture forward
    (`sv_evp_forward_attention`) and `forward_features` passes a maps buffer to `sv_evp_forward_features`; each appends one float32
    array [B, heads, N, N_kv] per encoder block per call to `get_local.cache['Attention.forward']`, in block order — what the
    reference's decorated `Attention.forward` records;
  * the switch is read at call time, so `activate()` also works after the model module has been imported (in the reference it must
    come before the import, because the decorator is applied then);
  * the flow cross-attention (`nn.MultiheadAttention`) is not decorated in the reference and is not captured here.
Capturing costs 6.76 MB of device memory per frame for mit_b3_evp at 224x224 (452 MB at 480x854) plus the copy to the host.
"""
from __future__ import annotations

import os
import sys

QUALNAME = "Attention.forward"


class get_local(object):
    cache = {}
    is_activate = False

    def __init__(self, varname):
        self.varname = varname

    def __call__(self, func):
        return func

    @classmethod
    def clear(cls):
        for key in cls.cache.keys():
            cls.cache[key] = []

    @classmethod
    def activate(cls):
        cls.is_activate = True


def active_caches():
    """The `cache` dicts of every active `get_local` of this file.  The same file may be imported twice under different names:
    `visualizer` through the `sys.path` switch of INTEGRATION §1 and `surgvid_b200.visualizer` package-style."""
    out = []
    for name in ("visualizer", __name__):
        mod = sys.modules.get(name)
        f = getattr(mod, "__file__", None)
        gl = getattr(mod, "get_local", None)
        if f and os.path.realpath(f) == os.path.realpath(__file__) and gl is not None and gl.is_activate:
            if not any(gl.cache is c for c in out):
                out.append(gl.cache)
    return out
