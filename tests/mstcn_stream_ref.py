"""Streaming restatement of the causal MS-TCN (`MultiStageModel_S`, mstcn_causal_conv=True) for tests: the state design of
`MultiStageModel_S.open_stream` / `sv_mstcn_stream_step` written out in PyTorch, in any dtype.

Per stream, per stage, per layer l (dilation d = 2^l) a ring of 2d rows keeps the layer's last inputs (position q in slot q mod 2d).
A step computes the new rows only; tap x[q - k d] comes from the step's rows when q - k d >= seen, from the ring when
0 <= q - k d < seen, and is zero when q - k d < 0.  After the step each layer's last min(2d, seen + count) inputs go to the ring.
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import torch
import torch.nn.functional as F


def _n(sd, prefix: str, fmt: str) -> int:
    n = 0
    while fmt.format(prefix=prefix, i=n) in sd:
        n += 1
    return n


class MstcnStreamRef:
    def __init__(self, sd: Dict[str, torch.Tensor], n_streams: int):
        self.sd = sd
        self.stages = ["stage1_phase"] + [f"stages.{s}" for s in range(_n(sd, "stages", "{prefix}.{i}.conv_1x1.weight"))]
        self.layers = _n(sd, "stage1_phase", "{prefix}.layers.{i}.conv_dilated.weight")
        self.f_maps = sd["stage1_phase.conv_1x1.weight"].shape[0]
        self.dtype = sd["stage1_phase.conv_1x1.weight"].dtype
        self.n_streams = n_streams
        self.seen = [0] * n_streams
        self.rings: List[List[List[torch.Tensor]]] = [[[torch.zeros(2 << l, self.f_maps, dtype=self.dtype) for l in range(self.layers)]
                                                        for _ in self.stages] for _ in range(n_streams)]

    def reset(self, ids: Sequence[int] | None = None):
        for s in (range(self.n_streams) if ids is None else ids):
            self.seen[s] = 0   # ring rows are only read at positions [0, seen)

    def _taps(self, ring: torch.Tensor, x: torch.Tensor, seen: int, d: int) -> torch.Tensor:
        """[2d + n, F]: the rows at positions seen - 2d .. seen + n - 1 (history from the ring, zero before position 0)."""
        hist = torch.zeros(2 * d, x.shape[1], dtype=x.dtype)
        for j in range(2 * d):
            q = seen - 2 * d + j
            if q >= 0:
                hist[j] = ring[q % (2 * d)]
        return torch.cat([hist, x])

    def _stage(self, s: int, g: int, p: str, x: torch.Tensor) -> torch.Tensor:
        sd, seen, n = self.sd, self.seen[s], x.shape[0]
        h = x @ sd[p + ".conv_1x1.weight"][:, :, 0].t() + sd[p + ".conv_1x1.bias"]
        inputs = []
        for l in range(self.layers):
            d = 2 ** l
            inputs.append(h)
            ext = self._taps(self.rings[s][g][l], h, seen, d)
            w = sd[f"{p}.layers.{l}.conv_dilated.weight"]
            acc = sd[f"{p}.layers.{l}.conv_dilated.bias"].expand(n, -1).clone()
            for k in range(3):   # tap k multiplies x[q - (2 - k) d]
                acc = acc + ext[k * d: k * d + n] @ w[:, :, k].t()
            h = h + F.relu(acc) @ sd[f"{p}.layers.{l}.conv_1x1.weight"][:, :, 0].t() + sd[f"{p}.layers.{l}.conv_1x1.bias"]
        for l, xin in enumerate(inputs):   # commit after the step
            R = 2 << l
            for j in range(max(0, n - R), n):
                self.rings[s][g][l][(seen + j) % R] = xin[j]
        return h @ sd[p + ".conv_out_classes.weight"][:, :, 0].t() + sd[p + ".conv_out_classes.bias"]

    @torch.no_grad()
    def step(self, feats: torch.Tensor, stream_ids: Sequence[int], counts: Sequence[int]) -> torch.Tensor:
        """feats [sum(counts), dim] -> logits [stages, C, sum(counts)]."""
        assert len(set(stream_ids)) == len(stream_ids) and all(c >= 1 for c in counts)
        outs, o = [], 0
        for s, c in zip(stream_ids, counts):
            x = feats[o:o + c].to(self.dtype)
            per = []
            for g, p in enumerate(self.stages):
                x = self._stage(s, g, p, x if g == 0 else F.softmax(x, dim=1))
                per.append(x.t())
            outs.append(torch.stack(per))
            self.seen[s] += c
            o += c
        return torch.cat(outs, dim=2)


@torch.no_grad()
def offline(sd: Dict[str, torch.Tensor], feats: torch.Tensor) -> torch.Tensor:
    """MultiStageModel_S.forward of one whole video in the dtype of `sd` (the conv1d form of oracle/mstcn_oracle.py):
    feats [T, dim] -> [stages, C, T]."""
    from oracle import mstcn_oracle as MO
    x = feats.to(sd["stage1_phase.conv_1x1.weight"].dtype).t().unsqueeze(0)
    out = MO.single_stage(sd, "stage1_phase", x)
    outs = [out]
    s = 0
    while f"stages.{s}.conv_1x1.weight" in sd:
        out = MO.single_stage(sd, f"stages.{s}", F.softmax(out, dim=1))
        outs.append(out)
        s += 1
    return torch.stack(outs)[:, 0]
