"""Shared reference, accuracy gate, stress inputs and a CPU emulator for LayerNorm (`sv_op_layernorm`, `sv_op_layernorm_nchw`):
y = (x - mean) / sqrt(var + eps) * gamma + beta over the last dim of fp32 [rows, C], biased variance, fp32 and / or bf16 outputs.

* `reference`: float64 LayerNorm, with the per-row quantities the gate needs.
* `gate_bound` / `gate_errors`: the gate, derived from the kernel's fp32 steps (elementwise.cu: two-pass mean and centred variance in
  fp32, rstd = MUFU.RSQ, y = v * (rstd g) + (b - mean rstd g) as two FMAs):
      |y - ref| <= TAU_MEAN * mean|x| * rstd |g|          the summed mean's error shifts every output of the row by dmu * rstd * |g|
                 + TAU_RSTD * |x - mean| * rstd |g|        the variance sum, 1/C, + eps and MUFU.RSQ (2 ulp) as a relative error of rstd
                 + 2^-23 * |x| * rstd |g| + 2^-24 |b|      the folded form's roundings (rstd * g, mean * rstd * g + b), which cancel
                 + tau_out * |ref|                         2^-24 (fp32 output, the last FMA) or 2^-8 (bf16)
  A non-finite output fails; a bf16 output must also pass gemm_ref's rounding-bias check (round to nearest even).
* `make_inputs`: seeded inputs, one stress input per way the arithmetic can go wrong (STRESS).
* `emulate`: the kernel's fp32 arithmetic on the CPU, with switches that inject known LayerNorm bugs (BUGS).
"""
from __future__ import annotations

import math

import torch

import gemm_ref as G

# 2^-20 = 16 fp32 roundings: the mean is a sum of at most 2 + 5 + 5 rounded adds (a float4 pair sum, up to 5 float4 per lane, up to 5 shuffle
# levels) times a rounded 1/C; rstd adds the variance sum (same depth), + eps and 2 ulp of MUFU.RSQ, halved by the square root.  Over
# tests/test_layernorm_gpu.py on one B200 (1000 W power limit) the worst whole-gate ratio was 0.21 for fp32 outputs of randn rows, 0.27 at
# |mean| / std = 1e3, 0.28 with the variance near eps and 0.53 on constant rows (the mean's rounding times rstd = 1 / sqrt(eps)).
TAU_MEAN = 2.0 ** -20
TAU_RSTD = 2.0 ** -20
TAU_OUT = {True: 2.0 ** -24, False: 2.0 ** -8}   # keyed by fp32 output

STRESS = ("randn", "bigmean", "const", "var_near_eps", "huge", "tiny")


def reference(x, gamma, beta, eps):
    """-> dict of float64 tensors on x's device: ref [rows, C] and the per-row / per-element magnitudes of the gate."""
    X = x.double()
    g, b = gamma.double().to(x.device), beta.double().to(x.device)
    mu = X.mean(1, keepdim=True)
    var = ((X - mu) ** 2).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    ref = (X - mu) * rstd * g + b
    return {"ref": ref, "mean_abs": X.abs().mean(1, keepdim=True), "xc": (X - mu).abs(), "x": X.abs(), "rstd": rstd, "g": g.abs(), "b": b.abs()}


def gate_bound(r, fp32: bool):
    s = r["rstd"] * r["g"]
    terms = {"mean": TAU_MEAN * r["mean_abs"] * s, "rstd": TAU_RSTD * r["xc"] * s, "fold": 2.0 ** -23 * r["x"] * s + 2.0 ** -24 * r["b"],
             "out": TAU_OUT[fp32] * r["ref"].abs()}
    return sum(terms.values()), terms


def gate_errors(out, r, fp32: bool, check_bias: bool = True) -> dict:
    """check_bias=False where the outputs sit on a few values (const, tiny: every row is ~beta), which the bias check cannot average."""
    o = out.double().to(r["ref"].device)
    if not bool(torch.isfinite(o).all()):
        return {"ratio": math.inf, "where": tuple((~torch.isfinite(o)).nonzero()[0].tolist()), "err": math.inf, "bound": 0.0}
    bound, terms = gate_bound(r, fp32)
    err = (o - r["ref"]).abs()
    q = err / bound.clamp_min(1e-300)
    i = int(q.argmax())
    res = {"ratio": float(q.max()), "where": divmod(i, q.shape[1]), "err": float(err.view(-1)[i]), "bound": float(bound.view(-1)[i]),
           "bias_ulp": None}
    if not fp32 and check_bias:   # gemm_ref's rounding-bias check: round to nearest even averages 0, truncation -0.5 ulp
        ulp = G._bf16_ulp(r["ref"])
        elig = (bound - terms["out"] <= G.BIAS_ELIGIBLE * ulp) & (r["ref"] != 0)
        if int(elig.sum()) >= G.BIAS_MIN_ELEMS:
            res["bias_ulp"] = float((((o - r["ref"]) * torch.sign(r["ref"])) / ulp)[elig].mean())
            res["ratio"] = max(res["ratio"], abs(res["bias_ulp"]) / G.BIAS_GATE)
    return res


def assert_gate(out, r, fp32: bool, what: str = "", check_bias: bool = True) -> dict:
    e = gate_errors(out, r, fp32, check_bias)
    assert e["ratio"] <= 1.0, f"{what}: worst |err|/bound {e['ratio']:.3g} at (row, c) = {e['where']}: |err| {e['err']:.3e}, bound {e['bound']:.3e}"
    return e


def make_inputs(kind: str, rows: int, C: int, seed: int = 0, device="cpu") -> dict:
    """Seeded x fp32 [rows, C], gamma, beta fp32 [C].
      randn         x ~ 3 N(0, 1) + 0.7, gamma ~ 1 + 0.2 N(0, 1), beta ~ 0.3 N(0, 1).
      bigmean       |mean| / std = 1e3: a one-pass variance E[x^2] - mean^2 loses every digit.
      const         every row constant: var = 0, the output is beta up to the mean's rounding.
      var_near_eps  std ~ sqrt(eps): eps outside the square root, or dropped, moves rstd by O(1).
      huge, tiny    |x| ~ 1e4 and ~ 1e-20 (squares far below fp32's normal range: the variance is eps)."""
    assert kind in STRESS, kind
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(s, generator=g)
    x = 3 * rn(rows, C) + 0.7
    gamma, beta = 1 + 0.2 * rn(C), 0.3 * rn(C)
    if kind == "bigmean":
        x = 1000.0 * torch.sign(rn(rows, 1)) + rn(rows, C)
    elif kind == "const":
        x = (5 * rn(rows, 1)).expand(rows, C).contiguous()
    elif kind == "var_near_eps":
        x = rn(rows, 1) + 3e-3 * rn(rows, C)
    elif kind == "huge":
        x = 1e4 * rn(rows, C)
    elif kind == "tiny":
        x = 1e-20 * rn(rows, C)
    return {"x": x.float().to(device), "gamma": gamma.float().to(device), "beta": beta.float().to(device)}


# Known ways LayerNorm goes wrong: bug -> (stress kind, fp32 output).
BUGS = {
    "one_pass_variance": ("bigmean", True),
    "unbiased_variance": ("randn", True),
    "eps_outside_sqrt": ("var_near_eps", True),
    "last_slot_dropped": ("randn", True),
    "bf16_truncation": ("randn", False),
}


def emulate(x, gamma, beta, eps: float, fp32: bool = True, bug: str | None = None) -> torch.Tensor:
    """The kernel's arithmetic in fp32 on the CPU (mean and centred variance as fp32 sums, rstd rounded to fp32, the folded two-FMA form)."""
    assert bug is None or bug in BUGS, bug
    X = x.float().cpu()
    C = X.shape[1]
    if bug == "last_slot_dropped":
        X = X[:, :C - 4]
    n = X.shape[1]
    inv_c = torch.tensor(1.0 / C, dtype=torch.float32)   # a dropped slot still counts in 1/C
    mean = (X.sum(1, keepdim=True) * inv_c).float()
    if bug == "one_pass_variance":
        var = ((X * X).sum(1, keepdim=True) * inv_c - mean * mean).float()
    else:
        var = (((X - mean) ** 2).sum(1, keepdim=True) * (inv_c if bug != "unbiased_variance" else torch.tensor(1.0 / (n - 1)))).float()
    if bug == "eps_outside_sqrt":
        rstd = (1.0 / (torch.sqrt(var.clamp_min(0).double()) + eps)).float()
    else:
        rstd = torch.rsqrt((var + eps).double()).float()
    g, b = gamma.float().cpu()[:n], beta.float().cpu()[:n]
    a = (rstd * g).float()
    c = ((-mean * rstd).double() * g.double() + b.double()).float()
    y = (X.double() * a.double() + c.double()).float()
    if bug == "last_slot_dropped":
        y = torch.cat([y, torch.zeros(y.shape[0], 4)], 1)
    if not fp32:
        y = (y.view(torch.int32) & -65536).view(torch.float32) if bug == "bf16_truncation" else y.to(torch.bfloat16).float()
    return y
