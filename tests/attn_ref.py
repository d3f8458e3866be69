"""Shared reference, accuracy gate, stress inputs and a tiled CPU emulator for `sv_op_attention` (softmax(Q K^T * scale) V).

Layout everywhere: q [B*Nq, heads*hd], k / v [B*Nkv, heads*hd]; head h owns columns [h*hd, (h+1)*hd) of every row.

* `reference`: float64 softmax(Q K^T * scale) V per (frame, head), computed from the bf16-rounded operands on their device.
* `gate_errors` / `assert_gate`: the accuracy gate of every attention kernel.  Both the relative L2 error and the largest absolute error
  (over max|ref|) must stay under the limits, over the whole output and over each head's column block.
* `make_inputs`: seeded bf16 inputs, plain randn and stress inputs aimed at masking, rescaling and range bugs.
* `emulate`: tiled online-softmax attention on the CPU with the kernels' precision (fp32 scores and sums in the exp2 domain, P rounded
  to bf16 before the PV product, bf16 output), with switches that inject known kernel bugs.  tests/test_attention_gate_cpu.py uses it
  to show that the gate accepts the honest arithmetic and rejects every one of these bugs.

Run as a script (`python attn_ref.py IN OUT`), it executes the cases saved in IN through `ops.attention` on cuda:0 and saves the outputs
and the kernel each case ran (as sv_op_attention_kernel reports the dispatch) to OUT: the GPU tests use it to run a case list in a
fresh process, where the A/B switches SURGVID_ATTN_TC / SURGVID_ATTN_ORDER (read once per process) can be set.
"""
from __future__ import annotations

import math
import os
import sys

import torch

# Limits of the gate.  The bf16 output alone contributes up to 2^-8 of max|ref| to the largest error and ~1.5e-3 to the relative L2
# error; the bf16 probabilities of the PV product add a little more.
REL_L2_GATE = 4e-3
MAX_ABS_GATE = 8e-3

KEY_TILE = 64   # keys per tile of every attention kernel

STRESS = ("randn", "neg", "plant_first", "plant_last", "wide", "uniform", "bigv")


def _heads_view(x: torch.Tensor, B: int, heads: int, hd: int) -> torch.Tensor:
    """[B*N, >= heads*hd] -> [B, heads, N, hd]"""
    return x[:, :heads * hd].reshape(B, -1, heads, hd).transpose(1, 2)


def _rows_view(x: torch.Tensor) -> torch.Tensor:
    """[B, heads, N, hd] -> [B*N, heads*hd]"""
    B, heads, N, hd = x.shape
    return x.transpose(1, 2).reshape(B * N, heads * hd)


def reference(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, heads: int, hd: int, scale: float) -> torch.Tensor:
    """float64 softmax(Q K^T * scale) V of the (bf16) operands, on their device -> [B*Nq, heads*hd] float64."""
    Q, K, V = (_heads_view(t, B, heads, hd).double() for t in (q, k, v))
    return _rows_view(torch.softmax((Q @ K.transpose(-1, -2)) * scale, dim=-1) @ V)


def gate_errors(out: torch.Tensor, ref: torch.Tensor, heads: int, hd: int) -> dict:
    """Worst relative L2 error and worst max-abs / max|ref| over the whole output and each head's column block, with where they occur.
    A non-finite output scores inf."""
    o, r = out[:, :heads * hd].double(), ref[:, :heads * hd].double()
    if not bool(torch.isfinite(o).all()):
        return {"rel_l2": math.inf, "max_abs": math.inf, "rel_l2_block": "all", "max_abs_block": "all", "max_abs_row": -1}
    res = {"rel_l2": 0.0, "max_abs": 0.0, "rel_l2_block": "all", "max_abs_block": "all", "max_abs_row": -1}
    blocks = [("all", 0, heads * hd)] + [(f"head {h}", h * hd, (h + 1) * hd) for h in range(heads)]
    for name, c0, c1 in blocks:
        d, rb = o[:, c0:c1] - r[:, c0:c1], r[:, c0:c1]
        rel = (d.norm() / rb.norm().clamp_min(1e-300)).item()
        err = d.abs()
        mx = (err.max() / rb.abs().max().clamp_min(1e-300)).item()
        if rel > res["rel_l2"]:
            res["rel_l2"], res["rel_l2_block"] = rel, name
        if mx > res["max_abs"]:
            res["max_abs"], res["max_abs_block"] = mx, name
            res["max_abs_row"] = int(err.amax(1).argmax())
    return res


def passes_gate(e: dict) -> bool:
    return e["rel_l2"] <= REL_L2_GATE and e["max_abs"] <= MAX_ABS_GATE


def gate_ratio(e: dict) -> float:
    """How far over the gate an error is (> 1: rejected)."""
    return max(e["rel_l2"] / REL_L2_GATE, e["max_abs"] / MAX_ABS_GATE)


def assert_gate(out: torch.Tensor, ref: torch.Tensor, heads: int, hd: int, Nq: int, what: str = "") -> dict:
    e = gate_errors(out, ref, heads, hd)
    row = e["max_abs_row"]
    assert passes_gate(e), (
        f"{what}: rel-L2 {e['rel_l2']:.3e} ({e['rel_l2_block']}; gate {REL_L2_GATE:.0e}), max-abs/max|ref| {e['max_abs']:.3e} "
        f"({e['max_abs_block']}, frame {row // Nq if row >= 0 else -1} row {row % Nq if row >= 0 else -1}; gate {MAX_ABS_GATE:.0e})")
    return e


# --------------------------------------------------------------------------------------------------------------- inputs
def make_inputs(kind: str, B: int, heads: int, Nq: int, Nkv: int, hd: int, seed: int = 0, device="cpu"):
    """-> q [B*Nq, heads*hd], k, v [B*Nkv, heads*hd] bf16 (contiguous) for softmax(Q K^T hd^-0.5) V.
      randn        q, k, v ~ N(0, 1): logits spread about +-3.
      neg          k = u + noise, q = -a u per (frame, head), every real logit about -30 (spread ~1.5): a zero-filled padding key that is
                   not masked scores 0 and takes all the weight.
      plant_first  one key 20+ logits above all others, at key 0 / at key Nkv-1 (inside the ragged last key tile): the output is that
      plant_last   key's V row; exercises the tail mask and the online-softmax rescale in both directions.
      wide         q, k scaled by 4: logit std ~16, a few keys carry the softmax (scale and exp-base errors show at full size).
      uniform      q = 0: the output is the mean of V over the frame's keys, per head.
      bigv         randn q, k and |V| up to 1e3 (range of the bf16 output)."""
    assert kind in STRESS, kind
    g = torch.Generator(device=device).manual_seed(seed)
    scale = hd ** -0.5

    def rn(*shape):
        return torch.randn(shape, generator=g, device=device)

    Q, K, V = rn(B, heads, Nq, hd), rn(B, heads, Nkv, hd), rn(B, heads, Nkv, hd)
    if kind == "neg":
        u = rn(B, heads, 1, hd)
        u = u / u.norm(dim=-1, keepdim=True)
        alpha = 30.0 / scale
        K = u + 0.05 * rn(B, heads, Nkv, hd)
        Q = -alpha * (u + 0.05 * rn(B, heads, Nq, hd))
    elif kind in ("plant_first", "plant_last"):
        a = rn(B, heads, 1, hd)
        a = a / a.norm(dim=-1, keepdim=True)
        Q = 3.0 * a + 0.2 * rn(B, heads, Nq, hd)
        K = 0.5 * rn(B, heads, Nkv, hd)
        j = 0 if kind == "plant_first" else Nkv - 1
        K[:, :, j] = (22.0 / (3.0 * scale)) * a[:, :, 0]
    elif kind == "wide":
        Q, K = 4.0 * Q, 4.0 * K
    elif kind == "uniform":
        Q = torch.zeros_like(Q)
    elif kind == "bigv":
        V = (torch.rand((B, heads, Nkv, hd), generator=g, device=device) * 2 - 1) * 1000.0
    return tuple(_rows_view(t).to(torch.bfloat16).contiguous() for t in (Q, K, V))


# --------------------------------------------------------------------------------------------------------------- emulator
# Known ways a tiled attention kernel goes wrong, each with the stress input that exposes it and the shapes on which it changes the
# output at all (B, heads, Nq, Nkv, query rows per tile).
BUGS = {
    "unmasked_padding": ("neg", lambda B, H, Nq, Nkv, qt: Nkv % KEY_TILE != 0),           # zero-filled tail keys score 0
    "no_rescale": ("plant_last", lambda B, H, Nq, Nkv, qt: Nkv > KEY_TILE),               # O, l not rescaled when the running max rises
    "drop_last_key_tile": ("plant_last", lambda B, H, Nq, Nkv, qt: True),
    "scale_x1.02": ("randn", lambda B, H, Nq, Nkv, qt: Nkv > 1),
    "natural_exp": ("wide", lambda B, H, Nq, Nkv, qt: Nkv > 1),                           # exp2 of un-log2e'd logits
    "last_key_tile_from_next_frame": ("plant_last", lambda B, H, Nq, Nkv, qt: B > 1),
    "head_offset_plus_one": ("uniform", lambda B, H, Nq, Nkv, qt: H > 1),
    "partial_query_tile_row_shift": ("randn", lambda B, H, Nq, Nkv, qt: Nq % qt != 0 and Nkv > 1),
}


def emulate(q, k, v, B: int, heads: int, hd: int, scale: float, q_tile: int = 64, bug: str | None = None) -> torch.Tensor:
    """Tiled attention with the kernels' arithmetic, on the CPU -> [B*Nq, heads*hd] (bf16 values, float32)."""
    assert bug is None or bug in BUGS, bug
    Q, K, V = (_heads_view(t, B, heads, hd).float() for t in (q, k, v))
    if bug == "head_offset_plus_one":
        Q, K, V = (t.roll(-1, dims=1) for t in (Q, K, V))
    Nq, Nkv = Q.shape[2], K.shape[2]
    nq_pad = -(-Nq // q_tile) * q_tile
    kt = -(-Nkv // KEY_TILE)
    Q = torch.nn.functional.pad(Q, (0, 0, 0, nq_pad - Nq))                 # zero-filled query rows of the last tile
    K = torch.nn.functional.pad(K, (0, 0, 0, kt * KEY_TILE - Nkv))        # zero-filled keys of the last key tile
    V = torch.nn.functional.pad(V, (0, 0, 0, kt * KEY_TILE - Nkv))
    if bug == "last_key_tile_from_next_frame":
        last = slice((kt - 1) * KEY_TILE, kt * KEY_TILE)
        K[:, :, last], V[:, :, last] = K.roll(-1, dims=0)[:, :, last], V.roll(-1, dims=0)[:, :, last]
    log2e = 1.4426950408889634
    scale_log2 = torch.tensor(scale * (1.0 if bug == "natural_exp" else log2e) * (1.02 if bug == "scale_x1.02" else 1.0), dtype=torch.float32)
    m = torch.full(Q.shape[:3], -math.inf)
    l = torch.zeros(Q.shape[:3])
    acc = torch.zeros(Q.shape)
    key = torch.arange(kt * KEY_TILE)
    for t in range(kt - 1 if bug == "drop_last_key_tile" else kt):
        ks = slice(t * KEY_TILE, (t + 1) * KEY_TILE)
        s = (Q @ K[:, :, ks].transpose(-1, -2)) * scale_log2
        if bug != "unmasked_padding":
            s = s.masked_fill(key[ks] >= Nkv, -math.inf)
        m_new = torch.maximum(m, s.amax(-1))
        corr = torch.ones_like(m) if bug == "no_rescale" else torch.exp2(m - m_new)
        p = torch.exp2(s - m_new[..., None])
        l = l * corr + p.sum(-1)
        acc = acc * corr[..., None] + p.to(torch.bfloat16).float() @ V[:, :, ks]
        m = m_new
    o = (acc / l[..., None]).to(torch.bfloat16).float()
    if bug == "partial_query_tile_row_shift" and Nq % q_tile:
        r0 = Nq // q_tile * q_tile
        o[:, :, r0:Nq] = o[:, :, r0 + 1:Nq + 1].clone()
    return _rows_view(o[:, :, :Nq])


# --------------------------------------------------------------------------------------------------------------- GPU runs
# sv_op_attention_kernel -> kernel name (SV_ATTN_* in include/surgvid.h)
KERNELS = ("attention_tc_single_kernel", "attention_tc_kernel", "attention_resident_kv_kernel", "attention_resident_multi_kernel",
           "attention_kernel")


def padded_ld(x: torch.Tensor) -> torch.Tensor:
    """The same values with the row stride rounded up to 8 elements (16 bytes), as `sv_op_attention` requires of its operands."""
    C = x.shape[1]
    if C % 8 == 0:
        return x
    buf = torch.zeros((x.shape[0], -(-C // 8) * 8), dtype=x.dtype, device=x.device)
    buf[:, :C] = x
    return buf[:, :C]


def _operands(case: dict, out=None):
    dev = torch.device("cuda:0")
    q, k, v = (padded_ld(case[n].to(dev)) for n in ("q", "k", "v"))
    if out is None:
        rows, C, off = q.shape[0], case["heads"] * case["hd"], case["o_offset"]
        out = torch.empty(rows * C + off, dtype=torch.bfloat16, device=dev)[off:].view(rows, C)
    return q, k, v, out


def _kernel(q, k, v, out, hd, Nkv) -> str:
    from surgvid_b200 import _native

    i = _native.lib().sv_op_attention_kernel(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), out.data_ptr(),
                                             out.stride(0), Nkv, hd)
    return KERNELS[i]


def call(case: dict, out=None, kernels=None) -> torch.Tensor:
    """ops.attention on one case: a dict with q, k, v (bf16), B, heads, hd, scale and o_offset (elements by which the output is moved
    off 16-byte alignment when `out` is not given).  The name of the kernel the call runs is appended to `kernels` when given."""
    from surgvid_b200 import ops

    q, k, v, out = _operands(case, out)
    if kernels is not None:
        kernels.append(_kernel(q, k, v, out, case["hd"], k.shape[0] // case["B"]))
    return ops.attention(q, k, v, case["B"], case["heads"], case["hd"], case["scale"], out=out)


def run_cases(cases):
    """Runs each case through `call` -> ([outputs on the CPU], [the attention kernel each case ran])."""
    kernels = []
    outs = [call(c, kernels=kernels) for c in cases]
    return [o.cpu() for o in outs], kernels


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import surgvid_b200  # noqa: F401

    outs, kernels = run_cases(torch.load(sys.argv[1]))
    torch.save({"outs": outs, "kernels": kernels}, sys.argv[2])
