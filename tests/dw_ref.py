"""Shared reference, accuracy gate, stress inputs and a CPU emulator for the depthwise 3x3 conv + bias + GELU (`sv_op_dwconv3x3_gelu`):
out = GELU(dwconv3x3(x) + bias) on NHWC bf16, zero padding per frame, w9c [9, C] fp32 tap-major (tap = kh * 3 + kw), bf16 output.

* `reference`: float64 pre-activation a, erf-GELU of it, and the magnitude m = sum |w| |x| + |b| that bounds the accumulation error.
* `gate_errors` / `assert_gate`: the gate, derived from the number formats rather than from max|ref|.  Elementwise,
      |out - ref| <= TAU_ACC * 1.13 * m + tau_gelu(mode, a) + 2^-8 |ref|
  (1.13 = max |GELU'|; 2^-8 = bf16 unit roundoff) with tau_gelu the error of the kernel's GELU form (common.cuh):
      mode 0  erf polynomial             8e-5                  (the formula's own error, 6.1e-5, plus its fp32 evaluation)
      mode 1  x * sigmoid(2 g(x))        3.0e-5 + 2^-20 |a|    (the fit's error, 3.0e-5, plus MUFU.EX2 / MUFU.RCP relative error)
      mode 2  0.5 x (1 + tanh(g(x)))     3.0e-5 + 2.5e-4 |a|   (the fit, plus tanh.approx's relative error as common.cuh states it)
  A non-finite output fails unless the reference is non-finite there too (a planted NaN).  Over the elements whose accumulation and GELU
  terms are below 2 % of a bf16 ulp, the mean signed rounding error must stay within gemm_ref.BIAS_GATE ulps (round to nearest even).
* `make_inputs`: seeded inputs, one stress input per bug class (STRESS).
* `emulate`: each kernel's fp32 arithmetic on the CPU (the SIMT kernel's single 10-term FMA chain, the TMA kernel's three 3-tap chains),
  with switches that inject known bugs (BUGS).  tests/test_dwconv_gate_cpu.py shows the gate accepts the honest arithmetic and rejects
  every one of them.

Run as a script (`python dw_ref.py IN OUT`), it executes the cases saved in IN (dicts with x, w9c, bias) through `ops.dwconv3x3_gelu` on
cuda:0 and saves the outputs and the plan each case got (sv_op_dwconv_plan_info) to OUT.  The GPU tests use it to run a case list in a
fresh process, where the switches SURGVID_DW_CPL / _GELU / _STAGES / _PREFETCH (read once per process) can be set; with SURGVID_LIB it
runs another build of the library on the same cases, for a bit-identity check of a kernel change.
"""
from __future__ import annotations

import math
import os
import re
import sys

import torch

import gemm_ref as G

TH = 7              # output rows per tile (both kernels)
# Accumulation term, relative to m = sum |w| |x| + |b|.  Each output is a 10-term fp32 sum (bias + 9 products): the SIMT kernel's one FMA
# chain and the TMA kernel's three 3-tap chains plus two adds both stay within 10 roundings of 2^-24 m; 2^-20 = 16 * 2^-24 leaves 1.6x
# over that worst case.  Measured over tests/test_dwconv_gpu.py (one B200, 1000 W power limit): no output needed this term at all, every
# error fit under the GELU and bf16 rounding terms alone (test_report_gate_terms prints what the run needed); the worst whole-gate ratio
# was 0.995, set by the bf16 rounding term, which round-to-nearest reaches by construction at the bottom of a binade.
TAU_ACC = 2.0 ** -20
GELU_LIP = 1.13
TAU_OUT = 2.0 ** -8
GELU_TAU = {0: (8e-5, 0.0), 1: (3.0e-5, 2.0 ** -20), 2: (3.0e-5, 2.5e-4)}   # mode -> (absolute, per |a|)
CHANNELS_PER_BLOCK = {"simt": 128, "tma4": 128, "tma2": 64}
GELU_G = (0.7974584707822386, 0.03705034510045914, -0.0003587323611556633)   # g(x) = x (G0 + G1 x^2 + G2 x^4) of modes 1 and 2

STRESS = ("randn", "asym_taps", "coord", "cancel", "bigbias", "gelu_sweep", "nan_plant")


# --------------------------------------------------------------------------------------------------------------- reference
def _taps(xp: torch.Tensor, H: int, W: int):
    """The nine shifted views of a padded [B, H+2, W+2, C] tensor, in tap order kh * 3 + kw."""
    return [xp[:, kh:kh + H, kw:kw + W, :] for kh in range(3) for kw in range(3)]


def gelu64(a: torch.Tensor) -> torch.Tensor:
    return 0.5 * a * (1.0 + torch.erf(a * (0.5 ** 0.5)))


def reference(x, w9c, bias):
    """-> (ref, a, m) float64 [B, H, W, C] on x's device: ref = GELU(a), a = dwconv3x3(x) + bias, m = sum |w| |x| + |b|."""
    B, H, W, C = x.shape
    xp = torch.nn.functional.pad(x.double(), (0, 0, 1, 1, 1, 1))
    w = w9c.double().to(x.device)
    b = bias.double().to(x.device)
    a = b.expand(B, H, W, C).clone()
    m = b.abs().expand(B, H, W, C).clone()
    for t, v in enumerate(_taps(xp, H, W)):
        a += v * w[t]
        m += v.abs() * w[t].abs()
    return gelu64(a), a, m


# --------------------------------------------------------------------------------------------------------------- gate
def gate_bound(ref, a, m, mode: int):
    t_abs, t_rel = GELU_TAU[mode]
    acc = TAU_ACC * GELU_LIP * m + t_abs + t_rel * a.abs()
    return acc + TAU_OUT * ref.abs(), acc


def gate_errors(out, ref, a, m, mode: int, check_bias: bool = True) -> dict:
    """Worst elementwise |out - ref| / bound, where it occurs ((b, h, w, c)), and the mean signed bf16 rounding error in ulps."""
    o = out.double().to(ref.device)
    planted = ~torch.isfinite(ref)
    bad = (~torch.isfinite(o) & ~planted) | (planted & ~torch.isnan(o))
    res = {"ratio": 0.0, "where": None, "err": 0.0, "bound": 0.0, "bias_ulp": None, "bias_ratio": 0.0, "n_bias": 0, "tau_acc_seen": 0.0}
    if bool(bad.any()):
        res.update(ratio=math.inf, where=tuple(bad.nonzero()[0].tolist()), err=math.inf, tau_acc_seen=math.inf)
        return res
    ok = ~planted
    bound, acc = gate_bound(ref, a, m, mode)
    err = torch.where(ok, (o - ref).abs(), torch.zeros((), dtype=torch.float64, device=ref.device))
    q = err / bound.clamp_min(1e-300)
    q = torch.where(ok, q, torch.zeros_like(q))
    i = int(q.argmax())
    lip_m = GELU_LIP * m
    seen = torch.where(ok, (err - (bound - TAU_ACC * lip_m)).clamp_min(0) / lip_m.clamp_min(1e-300), torch.zeros_like(q))
    res.update(ratio=float(q.max()), where=tuple(int(v) for v in torch.unravel_index(torch.tensor(i), q.shape)), err=float(err.view(-1)[i]),
               bound=float(bound.view(-1)[i]), tau_acc_seen=float(seen.max()))
    if check_bias:
        ulp = G._bf16_ulp(ref)
        elig = ok & (acc <= G.BIAS_ELIGIBLE * ulp) & (ref != 0)
        n = int(elig.sum())
        res["n_bias"] = n
        if n >= G.BIAS_MIN_ELEMS:
            b = float((((o - ref) * torch.sign(ref)) / ulp)[elig].mean())
            res["bias_ulp"], res["bias_ratio"] = b, abs(b) / G.BIAS_GATE
    return res


def gate_ratio(e: dict) -> float:
    return max(e["ratio"], e["bias_ratio"])


def passes_gate(e: dict) -> bool:
    return gate_ratio(e) <= 1.0


def describe(e: dict) -> str:
    s = f"worst |err|/bound {e['ratio']:.3g} at (b, h, w, c) = {e['where']}: |err| {e['err']:.3e}, bound {e['bound']:.3e}"
    if e["bias_ulp"] is not None:
        s += f"; rounding bias {e['bias_ulp']:+.4f} ulp over {e['n_bias']} elements (gate {G.BIAS_GATE})"
    return s


def assert_gate(out, ref, a, m, mode: int, what: str = "", check_bias: bool = True) -> dict:
    e = gate_errors(out, ref, a, m, mode, check_bias)
    assert passes_gate(e), f"{what}: {describe(e)}"
    return e


# --------------------------------------------------------------------------------------------------------------- inputs
def finite_bf16_values() -> torch.Tensor:
    """Every finite bf16 value (65 280 of them), as bf16."""
    bits = torch.arange(65536, dtype=torch.int32).to(torch.int16)
    v = bits.view(torch.bfloat16)
    return v[torch.isfinite(v.float())]


def nan_sites(B: int, H: int, W: int, C: int, tw: int) -> list:
    """(b, h, w, c) sites of nan_plant: frame corners, row-tile seams (h = 7k - 1, 7k), column-tile seams (w = tw k - 1, tw k), the first
    and last rows of each frame; channels spread over the channel blocks."""
    hs = sorted({0, H - 1} | {h for k in range(1, -(-H // TH)) for h in (TH * k - 1, TH * k)})
    ws = sorted({0, W - 1} | {w for k in range(1, -(-W // tw)) for w in (tw * k - 1, tw * k)})
    sites = []
    for b in range(B):
        for i, h in enumerate(hs):
            for j, w in enumerate(ws):
                if (i + j + b) % 2 == 0 or h in (0, H - 1) and w in (0, W - 1):
                    sites.append((b, h, w, (7 * i + 13 * j + 31 * b) % C))
    return sites


def make_inputs(kind: str, B: int, H: int, W: int, C: int, seed: int = 0, device="cpu", tw: int = 8) -> dict:
    """Seeded x bf16 [B, H, W, C], w9c fp32 [9, C], bias fp32 [C].
      randn       x ~ N(0, 1), w ~ N(0, 1) / 3, bias ~ 0.2 N(0, 1).
      asym_taps   nine distinct weights per channel (-1 ... 1 in tap order, a per-channel factor): transposed taps or a shifted halo move
                  the result by whole taps.
      coord       x encodes (frame, h, w, c) as small integers: reading a neighbouring pixel, row, frame or channel changes the sum.
      cancel      x = 8 + N(0, 1) / 4 and the nine taps of each channel sum to 0: |a| << m.
      bigbias     bias ~ U(-10, 10): pre-activations deep in both GELU tails.
      gelu_sweep  centre tap 1, other taps 0, bias 0, x = every finite bf16 value (cyclically; evenly spaced ones when there are fewer
                  elements): a == x exactly in both kernels, so the output is GELU_mode of each finite bf16 value.
      nan_plant   randn with NaN at the sites of `nan_sites`."""
    assert kind in STRESS, kind
    g = torch.Generator(device="cpu").manual_seed(seed)

    def rn(*shape):
        return torch.randn(shape, generator=g)

    x = rn(B, H, W, C)
    w = rn(9, C) / 3
    b = 0.2 * rn(C)
    if kind == "asym_taps":
        w = torch.linspace(-1.0, 1.0, 9)[:, None] * (0.5 + torch.rand((1, C), generator=g))
    elif kind == "coord":
        bb, hh, ww, cc = torch.meshgrid(*(torch.arange(n, dtype=torch.float32) for n in (B, H, W, C)), indexing="ij")
        x = ((bb * 5 + hh * 3 + ww * 7 + cc * 11) % 23 - 11) / 4
        w = torch.linspace(-1.0, 1.0, 9)[:, None] * (0.5 + torch.rand((1, C), generator=g))
    elif kind == "cancel":
        x = 8.0 + rn(B, H, W, C) / 4
        w = w - w.mean(0, keepdim=True)
    elif kind == "bigbias":
        b = torch.rand(C, generator=g) * 20 - 10
    elif kind == "gelu_sweep":
        v = finite_bf16_values().float()
        n = B * H * W * C
        x = (v.repeat(-(-n // v.numel()))[:n] if n >= v.numel() else v[torch.arange(n) * v.numel() // n]).view(B, H, W, C)
        w = torch.zeros(9, C)
        w[4] = 1.0
        b = torch.zeros(C)
    x = x.to(torch.bfloat16)
    if kind == "nan_plant":
        for s in nan_sites(B, H, W, C, tw):
            x[s] = float("nan")
    return {"x": x.to(device), "w9c": w.float().contiguous().to(device), "bias": b.float().to(device)}


# --------------------------------------------------------------------------------------------------------------- emulator
def _fma(a, b, c):
    """fp32 fused multiply-add (the product of two fp32 values is exact in float64)."""
    return (a.double() * b.double() + c.double()).float()


def gelu_f32(a: torch.Tensor, mode: int) -> torch.Tensor:
    """The GELU forms of common.cuh in fp32 (mode 2 with an exact tanh: tanh.approx's own error is what the device sweep measures)."""
    if mode == 0:
        return G.gelu_poly_f32(a)
    u = (a * a).clamp_max(49.0)
    if mode == 1:
        k = -2.8853900817779268
        q = _fma(u, torch.tensor(k * GELU_G[2]), torch.tensor(k * GELU_G[1]))
        q = _fma(q, u, torch.tensor(k * GELU_G[0]))
        return a * (1.0 / (torch.exp2(a * q) + 1.0))
    q = _fma(u, torch.tensor(GELU_G[2]), torch.tensor(GELU_G[1]))
    q = _fma(q, u, torch.tensor(GELU_G[0]))
    hx = a * 0.5
    return _fma(hx, torch.tanh(a * q), hx)


def gelu_tanh_approx_f32(a: torch.Tensor) -> torch.Tensor:
    return 0.5 * a * (1.0 + torch.tanh(0.7978845608028654 * (a + 0.044715 * a * a * a)))


# Known ways the kernels go wrong: bug -> (stress kind, predicate (B, H, W, C, form, tw) -> can the bug change the output at all).
BUGS = {
    "kh_kw_swapped": ("asym_taps", lambda B, H, W, C, f, tw: H > 1 or W > 1),
    "frame_bleed": ("coord", lambda B, H, W, C, f, tw: B > 1),
    "right_halo_from_next_row": ("coord", lambda B, H, W, C, f, tw: H > 1),
    "last_row_tile_dropped": ("randn", lambda B, H, W, C, f, tw: H % TH != 0 and H > TH),
    "last_col_tile_dropped": ("randn", lambda B, H, W, C, f, tw: W % tw != 0 and W > tw),
    "stale_channel_block_weights": ("asym_taps", lambda B, H, W, C, f, tw: C > CHANNELS_PER_BLOCK[f]),
    "bias_missing": ("bigbias", lambda B, H, W, C, f, tw: True),
    "bias_doubled": ("bigbias", lambda B, H, W, C, f, tw: True),
    "bf16_truncation": ("randn", lambda B, H, W, C, f, tw: True),
    "tanh_approx_gelu": ("gelu_sweep", lambda B, H, W, C, f, tw: True),
}


def emulate(x, w9c, bias, form: str = "tma4", mode: int = 2, tw: int = 8, bug: str | None = None) -> torch.Tensor:
    """The kernel's arithmetic on the CPU -> float32 [B, H, W, C] holding the bf16 outputs.  form: "simt" (one FMA chain from the bias, taps
    in the order 0, 3, 6, 1, 4, 7, 2, 5, 8; GELU mode 0 always), "tma4" / "tma2" (three 3-tap chains, the first from the bias, summed)."""
    assert bug is None or bug in BUGS, bug
    if form == "simt":
        mode = 0
    B, H, W, C = x.shape
    w = w9c.float().cpu().clone()
    b = bias.float().cpu().clone()
    if bug == "kh_kw_swapped":
        w = w.view(3, 3, C).transpose(0, 1).reshape(9, C)
    if bug == "stale_channel_block_weights":
        cb = CHANNELS_PER_BLOCK[form]
        for c0 in range(cb, C, cb):
            n = min(cb, C - c0)
            w[:, c0:c0 + n], b[c0:c0 + n] = w[:, c0 - cb:c0 - cb + n], b[c0 - cb:c0 - cb + n]
    if bug == "bias_missing":
        b = torch.zeros_like(b)
    elif bug == "bias_doubled":
        b = 2 * b
    xf = x.float().cpu()
    if bug == "frame_bleed":   # the frames as one tall image: a frame's halo rows come from its neighbours
        xp = torch.nn.functional.pad(xf.reshape(1, B * H, W, C), (0, 0, 1, 1, 1, 1))
        xp = torch.stack([xp[0, f * H:f * H + H + 2] for f in range(B)])
    else:
        xp = torch.nn.functional.pad(xf, (0, 0, 1, 1, 1, 1))
    if bug == "right_halo_from_next_row":   # column W of row h reads pixel 0 of row h + 1 (flat NHWC offset + C)
        xp[:, 1:H, W + 1] = xf[:, 1:H, 0]
    v = _taps(xp, H, W)
    wt = [w[t].expand(B, H, W, C) for t in range(9)]
    bb = b.expand(B, H, W, C)
    if form == "simt":
        a = bb.clone()
        for dx in range(3):
            for dy in range(3):
                a = _fma(v[dy * 3 + dx], wt[dy * 3 + dx], a)
    else:
        s = []
        for dy in range(3):
            t = _fma(v[dy * 3 + 1], wt[dy * 3 + 1], bb) if dy == 0 else v[dy * 3 + 1] * wt[dy * 3 + 1]
            t = _fma(v[dy * 3], wt[dy * 3], t)
            s.append(_fma(v[dy * 3 + 2], wt[dy * 3 + 2], t))
        a = (s[0] + s[1]) + s[2]
    y = gelu_tanh_approx_f32(a) if bug == "tanh_approx_gelu" else gelu_f32(a, mode)
    if bug == "bf16_truncation":
        y = (y.view(torch.int32) & -65536).view(torch.float32)
    else:
        y = y.to(torch.bfloat16).float()
    if bug == "last_row_tile_dropped" and H % TH and H > TH:
        y[:, H // TH * TH:] = 0.0
    if bug == "last_col_tile_dropped" and W % tw and W > tw:
        y[:, :, W // tw * tw:] = 0.0
    return y


# --------------------------------------------------------------------------------------------------------------- GELU constants
def gelu_constants(path: str | None = None) -> dict:
    """The GELU constants of common.cuh, parsed from the source: the polynomial's clamp and coefficients, and g(x)'s coefficients."""
    path = path or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "deep-learning-for-surgical-video-analysis_b200",
                                "csrc", "common.cuh")
    src = open(path).read()
    body = src[src.index("f2_gelu_erf_poly(f32x2 x)"):src.index("f2_gelu_erf_poly_x2")]
    lim = float(re.search(r"const float lim = ([0-9.e+-]+)f", body).group(1))
    coef = [float(v) for v in re.findall(r"SV_C2\(([-0-9.e]+)f\)", body) if v != "0.5"]
    g = [float(re.search(rf"#define SV_GELU_G{i} \(?([-0-9.e]+)f", src).group(1)) for i in range(3)]
    return {"lim": lim, "poly": coef, "g": g}


# --------------------------------------------------------------------------------------------------------------- GPU runs
def plan_info(case: dict, num_sms: int | None = None) -> dict:
    from surgvid_b200 import ops

    return ops.dwconv_plan_info(*case["x"].shape, num_sms)


def run_cases(cases):
    """ops.dwconv3x3_gelu on each case on cuda:0 -> ([outputs on the CPU], [plan of each case])."""
    from surgvid_b200 import ops

    outs, plans = [], []
    for c in cases:
        plans.append(plan_info(c))
        outs.append(ops.dwconv3x3_gelu(c["x"].cuda(), c["w9c"].cuda(), c["bias"].cuda()).cpu())
    return outs, plans


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import surgvid_b200  # noqa: F401

    outs, plans = run_cases(torch.load(sys.argv[1]))
    torch.save({"outs": outs, "plans": plans}, sys.argv[2])
