"""Shared reference, accuracy gate, stress inputs and a CPU emulator for the tcgen05 GEMM (`sv_op_gemm_bf16` / `sv_op_gemm_bf16_cat`):
out = act(A W^T + bias) (+ residual), A = [a | a2] bf16 [M, K], W bf16 [N, K], bias / residual fp32, bf16 or fp32 output.

* `reference`: float64 act(A W^T + bias) + residual of the values the kernel reads (GELU in its erf form), on the operands' device, and
  the magnitude |A| |W|^T + |bias| that bounds the accumulation error.
* `gate_errors` / `assert_gate`: the gate, derived from the number formats rather than from max|ref|.  Elementwise,
      |out - ref| <= TAU_ACC * L * (|A| |W|^T + |bias|) + tau_out * |ref| + tau_abs
  with L = 1.13 (max |GELU'|) under GELU, else 1; tau_out = 2^-8 (bf16 unit roundoff) or 4 * 2^-24 (fp32); tau_abs = the error of the packed
  erf polynomial of bf16 GELU outputs (common.cuh: <= 6.1e-5), else 0.  A bf16 output must also round without bias: over the elements
  whose accumulation bound is below 2 % of a bf16 ulp, the mean signed error toward zero must stay within BIAS_GATE ulps (round to
  nearest even averages 0, truncation -0.5).  A non-finite output fails.
* `make_inputs`: seeded inputs, plain randn and one stress input per bug class.
* `emulate`: the kernel's arithmetic on the CPU (fp32 accumulation in 16-deep k-steps, fp32 epilogue, round to nearest even), with switches
  that inject known GEMM bugs.  tests/test_gemm_gate_cpu.py uses it to show that the gate accepts the honest arithmetic and rejects every
  one of these bugs.

Run as a script (`python gemm_ref.py IN OUT`), it executes the cases saved in IN through `ops.gemm_bf16` / `ops.gemm_bf16_cat` on cuda:0
and saves the outputs and the plan each case got (sv_op_gemm_plan_info) to OUT: the GPU tests use it to run a case list in a fresh
process, where the A/B switches SURGVID_GEMM_TMA_OUT / _EPI_BUFS / _EPI_LAG / _PREFETCH (read once per process) can be set.
"""
from __future__ import annotations

import math
import os
import sys

import torch

ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
BLOCK_M, BLOCK_K, K_STEP = 128, 64, 16

# Accumulation term of the gate, relative to |A| |W|^T + |bias|.  The worst this term had to cover over the case table and every A/B
# switch of tests/test_gemm_gpu.py was 7.0e-7 (one B200, 1000 W power limit); 2^-19 = 1.9e-6 leaves 2.7x.  The CPU emulation's fp32
# accumulation (16-deep k-steps) stays within half of the gate with it.
TAU_ACC = 2.0 ** -19
TAU_OUT = {False: 2.0 ** -8, True: 4 * 2.0 ** -24}   # keyed by out_fp32
GELU_POLY_ABS = 8e-5                                  # packed erf polynomial (bf16 GELU outputs): <= 6.1e-5, plus its fp32 evaluation
GELU_LIP = 1.13                                       # max |GELU'(x)|
BIAS_GATE = 0.08                                      # mean signed bf16 rounding error toward zero, in ulps
BIAS_MIN_ELEMS = 2000                                 # fewer eligible elements: the bias check is skipped
BIAS_ELIGIBLE = 0.02                                  # eligible: accumulation bound <= 2 % of the element's bf16 ulp

GELU_HUGE = (8.1e37, -8.1e37, 1e38, -1e38, 3e38, -3e38)   # pre-activations past 8.04e37 (gelu_sweep)
STRESS = ("randn", "bigres", "colbias", "gelu_sweep", "cancel", "rowid")


def _act64(y: torch.Tensor, act: int) -> torch.Tensor:
    if act == ACT_GELU:
        return 0.5 * y * (1.0 + torch.erf(y * (0.5 ** 0.5)))
    if act == ACT_RELU:
        return y.clamp_min(0.0)
    return y


def reference(a, w, bias, act, residual, a2=None):
    """-> (ref, mag) float64 [M, N] on the operands' device: ref = act([a | a2] w^T + bias) + residual, mag = |A| |W|^T + |bias|."""
    A = a.double() if a2 is None else torch.cat([a.double(), a2.double()], 1)
    W = w.double()
    y = A @ W.T
    mag = A.abs() @ W.abs().T
    if bias is not None:
        y = y + bias.double()
        mag = mag + bias.double().abs()
    y = _act64(y, act)
    if residual is not None:
        y = y + residual.double()
    return y, mag


def _bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 values (8 significant bits) at |x| (float64)."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def gate_bound(ref, mag, act: int, out_fp32: bool):
    lip = GELU_LIP if act == ACT_GELU else 1.0
    tau_abs = GELU_POLY_ABS if (act == ACT_GELU and not out_fp32) else 0.0
    acc = TAU_ACC * lip * mag + tau_abs
    return acc + TAU_OUT[bool(out_fp32)] * ref.abs(), acc


def gate_errors(out, ref, mag, act: int, out_fp32: bool, block_n: int | None = None, row0: int = 0, check_bias: bool = True) -> dict:
    """Worst elementwise |out - ref| / bound (with where it occurs) and, for bf16 outputs, the mean signed rounding error in ulps.
    `row0` is the row of out[0] in the whole output (for sampled rows).  `check_bias=False` for outputs whose values sit on a grid
    (rowid): the bias check assumes values spread evenly within an ulp."""
    o, r, m = out.double(), ref.double().to(out.device), mag.double().to(out.device)
    if not bool(torch.isfinite(o).all()):
        bad = (~torch.isfinite(o)).nonzero()[0].tolist()
        return {"ratio": math.inf, "bias_ulp": None, "bias_ratio": 0.0, "row": row0 + bad[0], "col": bad[1], "block_n": block_n,
                "err": math.inf, "bound": 0.0, "n_bias": 0, "tau_acc_seen": math.inf}
    bound, acc = gate_bound(r, m, act, out_fp32)
    err = (o - r).abs()
    q = err / bound.clamp_min(1e-300)
    i = int(q.argmax())
    row, col = divmod(i, q.shape[1])
    # the smallest TAU_ACC this output would pass with: what is left of the error after the output and polynomial terms, over L * mag
    lip_mag = (GELU_LIP if act == ACT_GELU else 1.0) * m
    tau_seen = float(((err - (bound - TAU_ACC * lip_mag)).clamp_min(0) / lip_mag.clamp_min(1e-300)).max())
    res = {"ratio": float(q.max()), "row": row0 + row, "col": col, "block_n": block_n, "err": float(err.view(-1)[i]),
           "bound": float(bound.view(-1)[i]), "bias_ulp": None, "bias_ratio": 0.0, "n_bias": 0, "tau_acc_seen": tau_seen}
    if not out_fp32 and check_bias:
        ulp = _bf16_ulp(r)
        ok = (acc <= BIAS_ELIGIBLE * ulp) & (r != 0)
        n = int(ok.sum())
        res["n_bias"] = n
        if n >= BIAS_MIN_ELEMS:
            b = float((((o - r) * torch.sign(r)) / ulp)[ok].mean())
            res["bias_ulp"], res["bias_ratio"] = b, abs(b) / BIAS_GATE
    return res


def gate_ratio(e: dict) -> float:
    """How far over the gate an error is (> 1: rejected)."""
    return max(e["ratio"], e["bias_ratio"])


def passes_gate(e: dict) -> bool:
    return gate_ratio(e) <= 1.0


def describe(e: dict) -> str:
    bn = e["block_n"]
    where = f"row {e['row']} col {e['col']} (M tile {e['row'] // BLOCK_M}" + (f", N tile {e['col'] // bn})" if bn else ")")
    s = f"worst |err|/bound {e['ratio']:.3g} at {where}: |err| {e['err']:.3e}, bound {e['bound']:.3e}"
    if e["bias_ulp"] is not None:
        s += f"; rounding bias {e['bias_ulp']:+.4f} ulp over {e['n_bias']} elements (gate {BIAS_GATE})"
    return s


def assert_gate(out, ref, mag, act: int, out_fp32: bool, what: str = "", block_n: int | None = None, row0: int = 0, check_bias: bool = True) -> dict:
    e = gate_errors(out, ref, mag, act, out_fp32, block_n, row0, check_bias)
    assert passes_gate(e), f"{what}: {describe(e)}"
    return e


# --------------------------------------------------------------------------------------------------------------- inputs
def make_inputs(kind: str, M: int, N: int, K: int, K2: int = 0, seed: int = 0, device="cpu", bias: bool = True, residual: bool = True) -> dict:
    """Seeded operands: a bf16 [M, K - K2], a2 bf16 [M, K2] (None when K2 == 0), w bf16 [N, K] (rows scaled 1/sqrt(K)), bias fp32 [N],
    residual fp32 [M, N] (None when not wanted; colbias and gelu_sweep always have a bias; bigres and rowid only act through the residual).
      randn       A ~ N(0, 1), bias ~ 0.5 N(0, 1), residual ~ N(0, 1).
      bigres      |residual| ~ 1e3: a residual that passes through bf16 loses ~2 in the sum.
      colbias     bias is a per-column ramp (-4 ... 4): a bias slice shifted by a tile or a 16 / 32-column chunk is off by >= 16 steps.
      gelu_sweep  small A W^T and a bias ramp over [-10, 10]: pre-activations cross the erf polynomial's clamp and the tails; the first
                  columns' biases are GELU_HUGE, where x * xc * Q overflowed when it was evaluated as (x * xc) * Q.
      cancel      rows of A share a large mean (~32) and the rows of W sum to ~0: |ref| << |A| |W|^T.
      rowid       residual[r, c] = r % 1024 + c / 1024: any mix-up of rows, lane quarters or M tiles moves the result by >= 1 (values on
                  a grid: the gate's rounding-bias check does not apply)."""
    assert kind in STRESS, kind
    g = torch.Generator(device=device).manual_seed(seed)

    def rn(*shape):
        return torch.randn(shape, generator=g, device=device)

    A = rn(M, K)
    W = rn(N, K) / math.sqrt(K)
    b = 0.5 * rn(N)
    R = rn(M, N)
    if kind == "bigres":
        R = (torch.rand((M, N), generator=g, device=device) * 2 - 1) * 1000.0
    elif kind == "colbias":
        b = torch.linspace(-4.0, 4.0, N, device=device)
    elif kind == "gelu_sweep":
        W = W * 0.3
        b = torch.linspace(-10.0, 10.0, N, device=device)[torch.randperm(N, generator=g, device=device)]
        b[:len(GELU_HUGE)] = torch.tensor(GELU_HUGE, device=device)
    elif kind == "cancel":
        A = 32.0 + A
        W = W - W.mean(1, keepdim=True)
    elif kind == "rowid":
        r = torch.arange(M, device=device, dtype=torch.float32)[:, None]
        c = torch.arange(N, device=device, dtype=torch.float32)[None, :]
        R = (r % 1024) + c / 1024
    A = A.to(torch.bfloat16)
    need_bias = bias or kind in ("colbias", "gelu_sweep")
    return {"a": A[:, :K - K2].contiguous(), "a2": A[:, K - K2:].contiguous() if K2 else None, "w": W.to(torch.bfloat16),
            "bias": b if need_bias else None, "residual": R if residual else None}


# --------------------------------------------------------------------------------------------------------------- emulator
GELU_POLY_LIM = 4.244771   # the polynomial's clamp: fp32 xc * Q(xc^2) is exactly 0.5 there (common.cuh)
GELU_POLY_COEF = (5.626770213e-11, -5.371870724e-09, 2.268296714e-07, -5.646215765e-06, 9.359063167e-05, -1.109400333e-03, 9.818119241e-03,
                  -6.634692395e-02, 3.989031282e-01)


def gelu_poly_f32(x: torch.Tensor) -> torch.Tensor:
    """f2_gelu_erf_poly (common.cuh) in fp32, FMA by FMA: 0.5 x + x (xc Q(xc^2)) with xc = clamp(x), the GELU of bf16 outputs."""
    def fma(a, b, c):   # the product of two fp32 values is exact in float64
        return (a.double() * b.double() + c.double()).float()

    x = x.float()
    lim = torch.tensor(GELU_POLY_LIM, dtype=torch.float32)
    xc = torch.minimum(torch.maximum(x, -lim), lim)
    w = xc * xc
    q = fma(torch.tensor(GELU_POLY_COEF[0]), w, torch.tensor(GELU_POLY_COEF[1]))
    for c in GELU_POLY_COEF[2:]:
        q = fma(q, w, torch.tensor(c))
    return fma(x, xc * q, x * 0.5)


def gelu_erf_f32(x: torch.Tensor) -> torch.Tensor:
    return 0.5 * x * (1.0 + torch.erf(x * 0.70710678118654752440))


def gelu_tanh_f32(x: torch.Tensor) -> torch.Tensor:
    return 0.5 * x * (1.0 + torch.tanh(0.7978845608028654 * (x + 0.044715 * x * x * x)))


PAD_VALUE = 1.0   # what a kernel that reads operand columns past K would find there (the GPU tests put NaN)

# Known ways the GEMM goes wrong: (stress kind, out_fp32, act, predicate (M, N, K, K2, block_n) -> can the bug change the output at all).
BUGS = {
    "drop_ragged_k_block": ("randn", True, ACT_NONE, lambda M, N, K, K2, bn: K % BLOCK_K != 0),
    "first_tile_bias_everywhere": ("colbias", True, ACT_NONE, lambda M, N, K, K2, bn: N > bn),
    "bias_shift_16": ("colbias", True, ACT_NONE, lambda M, N, K, K2, bn: N > 16),
    "residual_via_bf16": ("bigres", True, ACT_NONE, lambda M, N, K, K2, bn: True),
    "act_after_residual": ("bigres", True, ACT_GELU, lambda M, N, K, K2, bn: True),
    "tanh_gelu_f32": ("gelu_sweep", True, ACT_GELU, lambda M, N, K, K2, bn: True),
    "bf16_truncation": ("randn", False, ACT_NONE, lambda M, N, K, K2, bn: True),
    "last_m_tile_from_previous": ("rowid", True, ACT_NONE, lambda M, N, K, K2, bn: M > BLOCK_M and M % BLOCK_M != 0),
    "residual_lane_quarter_32": ("rowid", True, ACT_NONE, lambda M, N, K, K2, bn: True),
    "a2_wrong_k_offset": ("randn", True, ACT_NONE, lambda M, N, K, K2, bn: K2 > 0),
    "pad_columns_read": ("randn", True, ACT_NONE, lambda M, N, K, K2, bn: K % BLOCK_K != 0),
}


def emulate(a, w, bias, act: int, residual, out_fp32: bool, a2=None, block_n: int | None = None, bug: str | None = None) -> torch.Tensor:
    """The kernel's arithmetic on the CPU -> [M, N] float32 (bf16 values for a bf16 output)."""
    assert bug is None or bug in BUGS, bug
    M, N = a.shape[0], w.shape[0]
    if a2 is not None and bug == "a2_wrong_k_offset":
        a2 = torch.nn.functional.pad(a2[:, 8:], (0, 8))           # segment read 8 columns too far on (zero-filled past K2)
    A = (a if a2 is None else torch.cat([a, a2], 1)).double()
    W = w.double()
    K = A.shape[1]
    kb = -(-K // BLOCK_K)
    k_pad = kb * BLOCK_K
    fill = PAD_VALUE if bug == "pad_columns_read" else 0.0
    A = torch.nn.functional.pad(A, (0, k_pad - K), value=fill)
    W = torch.nn.functional.pad(W, (0, k_pad - K), value=fill)
    k_end = (kb - 1) * BLOCK_K if (bug == "drop_ragged_k_block" and K % BLOCK_K) else k_pad
    k_steps = -(-K // K_STEP) * K_STEP if bug != "pad_columns_read" else k_pad   # the kernel issues ceil(k_left / 16) k-steps
    acc = torch.zeros((M, N), dtype=torch.float32)
    for k0 in range(0, min(k_end, k_steps), K_STEP):
        acc = acc + (A[:, k0:k0 + K_STEP] @ W[:, k0:k0 + K_STEP].T).float()   # one tcgen05 k-step, added to the fp32 accumulator
    b = torch.zeros(N) if bias is None else bias.float().clone()
    if bug == "first_tile_bias_everywhere":
        b = b[:block_n].repeat(-(-N // block_n))[:N]
    elif bug == "bias_shift_16":
        b = b.roll(-16)
    y = acc + b
    res = None if residual is None else residual.float()
    if res is not None and bug == "residual_via_bf16":
        res = res.to(torch.bfloat16).float()
    if res is not None and bug == "residual_lane_quarter_32":
        rows = torch.arange(M)
        src = rows // BLOCK_M * BLOCK_M + (rows % BLOCK_M + 32) % BLOCK_M
        res = torch.where((src < M)[:, None], res[src.clamp_max(M - 1)], torch.zeros(()))
    if bug == "act_after_residual" and res is not None:
        y, res = y + res, None
    if act == ACT_GELU:
        y = gelu_tanh_f32(y) if bug == "tanh_gelu_f32" else (gelu_erf_f32(y) if out_fp32 else gelu_poly_f32(y))
    elif act == ACT_RELU:
        y = y.clamp_min(0.0)
    if res is not None:
        y = y + res
    if not out_fp32:
        if bug == "bf16_truncation":
            y = (y.view(torch.int32) & -65536).view(torch.float32)
        else:
            y = y.to(torch.bfloat16).float()
    if bug == "last_m_tile_from_previous" and M > BLOCK_M and M % BLOCK_M:
        r0 = M // BLOCK_M * BLOCK_M
        y[r0:] = y[r0 - BLOCK_M:M - BLOCK_M].clone()
    return y


# --------------------------------------------------------------------------------------------------------------- GPU runs
def plan_info(case: dict, num_sms: int | None = None) -> dict:
    """The plan sv_op_gemm_bf16(_cat) gives this case in this process (SURGVID_GEMM_PAIR is read per call, as the ops do)."""
    from surgvid_b200 import ops

    pair = int(os.environ["SURGVID_GEMM_PAIR"]) if "SURGVID_GEMM_PAIR" in os.environ else -1
    a2 = case.get("a2")
    K = case["w"].shape[1]
    return ops.gemm_plan_info(case["a"].shape[0], case["w"].shape[0], K, 0 if a2 is None else a2.shape[1], case["out_fp32"],
                              case.get("residual") is not None, pair, num_sms)


def call(case: dict):
    """ops.gemm_bf16 / ops.gemm_bf16_cat on one case: a dict with a, a2 (or None), w, bias, act, residual, out_fp32, and optionally
    in_place (the residual is updated in place) and out_margin = (rows, cols): the output is then a view inside a NaN-filled buffer with
    that many rows / columns on every side.  -> (output block, whole output buffer)."""
    from surgvid_b200 import ops

    dev = torch.device("cuda:0")
    t = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in case.items()}
    M, N = t["a"].shape[0], t["w"].shape[0]
    dtype = torch.float32 if t["out_fp32"] else torch.bfloat16
    res = t.get("residual")
    if t.get("in_place"):
        buf = res.clone() if res.is_contiguous() else res.as_strided((res.shape[0], res.stride(0)), (res.stride(0), 1)).clone()
        out = res = buf[:, :N]
    else:
        gr, gc = t.get("out_margin", (0, 0))
        ldc = N + 2 * gc
        buf = torch.full((M + 2 * gr, ldc), float("nan"), dtype=dtype, device=dev)
        out = buf[gr:gr + M, gc:gc + N]
    kw = dict(bias=t.get("bias"), act=t.get("act", ACT_NONE), residual=res, out=out)
    if t.get("a2") is None:
        ops.gemm_bf16(t["a"], t["w"], **kw)
    else:
        ops.gemm_bf16_cat(t["a"], t["a2"], t["w"], **kw)
    return out, buf


def run_cases(cases):
    """Runs each case through `call` -> ([output blocks on the CPU], [plan of each case], [margins of the output kept their bits])."""
    outs, plans, intact = [], [], []
    for c in cases:
        plans.append(plan_info(c))
        out, buf = call(c)
        keep = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
        gr, gc = (0, 0) if c.get("in_place") else c.get("out_margin", (0, 0))
        keep[gr:gr + out.shape[0], gc:gc + out.shape[1]] = False
        intact.append(bool(torch.isnan(buf[keep]).all()) if not c.get("in_place") else True)
        outs.append(out.cpu())
    return outs, plans, intact


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import surgvid_b200  # noqa: F401

    outs, plans, intact = run_cases(torch.load(sys.argv[1]))
    torch.save({"outs": outs, "plans": plans, "intact": intact}, sys.argv[2])
