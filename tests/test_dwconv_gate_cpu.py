"""The DWConv3x3 + GELU accuracy gate (tests/dw_ref.py) judged on the CPU: the GELU forms of common.cuh (coefficients parsed from the source)
meet the bounds the gate assumes; the gate accepts each kernel's honest arithmetic on every stress input and rejects each known bug,
injected into the same emulation, on the input it targets; where a bug cannot change a shape the emulation stays bit-identical.  Also
without a device: argument errors come back as SV_ERR_INVALID, and sv_op_dwconv_plan_info agrees with the plan formulas."""
import ctypes
import math

import pytest
import torch

import dw_ref as D
import gemm_ref as G

# (B, H, W, C, form, tw): ragged and exact row / column tiles, one and several channel blocks, each kernel form
SHAPES = [(2, 9, 20, 256, "tma4", 8), (3, 14, 14, 128, "tma4", 7), (2, 10, 16, 128, "tma2", 8), (2, 12, 27, 192, "simt", 8),
          (4, 15, 45, 12, "simt", 8), (3, 8, 9, 320, "simt", 8)]
MIN_REJECTION = 4.0
MODES = {"simt": (0,), "tma4": (0, 1, 2), "tma2": (0, 1, 2)}


def _sid(s):
    return f"{s[4]}-{s[0]}x{s[1]}x{s[2]}x{s[3]}"


def _run(kind, shape, mode, bug=None, seed=1):
    B, H, W, C, form, tw = shape
    d = D.make_inputs(kind, B, H, W, C, seed=seed, tw=tw)
    ref, a, m = D.reference(d["x"], d["w9c"], d["bias"])
    out = D.emulate(d["x"], d["w9c"], d["bias"], form, mode, tw, bug)
    return out, ref, a, m


# ------------------------------------------------------------------------------------------------------- GELU formulas
def test_gelu_constants_parse_and_match_the_emulators():
    k = D.gelu_constants()
    assert len(k["poly"]) == 9 and len(k["g"]) == 3
    assert tuple(k["poly"]) == G.GELU_POLY_COEF and k["lim"] == G.GELU_POLY_LIM
    assert all(abs(a - b) <= 1e-9 * abs(b) for a, b in zip(k["g"], D.GELU_G))


def _poly64(x, k):
    xc = x.clamp(-k["lim"], k["lim"])
    w = xc * xc
    q = torch.full_like(x, k["poly"][0])
    for c in k["poly"][1:]:
        q = q * w + c
    return 0.5 * x + x * (xc * q)


def _g64(x, k):
    u = (x * x).clamp_max(49.0)
    return x * (k["g"][0] + k["g"][1] * u + k["g"][2] * u * u)


def test_gelu_formulas_meet_their_stated_bounds():
    """In float64 on [-12, 12]: the polynomial (mode 0) within 6.1e-5 (common.cuh), the sigmoid and tanh forms (modes 1, 2) within 3.0e-5;
    all within the gate's tau_gelu."""
    k = D.gelu_constants()
    x = torch.linspace(-12, 12, 480001, dtype=torch.float64)
    exact = D.gelu64(x)
    e0 = float((_poly64(x, k) - exact).abs().max())
    e1 = float((x * torch.sigmoid(2 * _g64(x, k)) - exact).abs().max())
    e2 = float((0.5 * x * (1 + torch.tanh(_g64(x, k))) - exact).abs().max())
    print(f"\nGELU formula error in float64 on [-12, 12]: polynomial {e0:.3e}, sigmoid {e1:.3e}, tanh {e2:.3e}")
    assert e0 <= 6.1e-5 < D.GELU_TAU[0][0]
    assert e1 <= 3.0e-5 <= D.GELU_TAU[1][0] and e2 <= 3.0e-5 <= D.GELU_TAU[2][0]


def test_polynomial_gelu_in_fp32_is_finite_and_bounded_on_every_bf16_value():
    """The fp32 evaluation, FMA by FMA as the kernels run it, on every finite bf16 value: finite everywhere (x * (xc * Q) cannot overflow),
    within tau_gelu(0) + 2^-22 |x| of GELU (the clamp saturates exactly: beyond it y is x or 0), and GELU(-1e38) is 0."""
    v = D.finite_bf16_values().float()
    y = G.gelu_poly_f32(v)
    assert bool(torch.isfinite(y).all()), v[~torch.isfinite(y)][:8]
    err = (y.double() - D.gelu64(v.double())).abs()
    assert bool((err <= D.GELU_TAU[0][0] + 2.0 ** -22 * v.double().abs()).all()), float(err.max())
    big = torch.tensor([-1e38, -8.1e37, -3e38, 8.1e37, 3e38, -100.0, -12.0])
    assert G.gelu_poly_f32(big)[[0, 1, 2, 5]].abs().max() == 0 and torch.equal(G.gelu_poly_f32(big)[3:5], big[3:5])


# ------------------------------------------------------------------------------------------------------- gate vs the emulator
@pytest.mark.parametrize("shape", SHAPES, ids=_sid)
@pytest.mark.parametrize("kind", D.STRESS)
def test_gate_accepts_honest_emulation(kind, shape):
    for mode in MODES[shape[4]]:
        out, ref, a, m = _run(kind, shape, mode)
        e = D.gate_errors(out, ref, a, m, mode, check_bias=kind not in ("coord", "gelu_sweep"))
        assert D.passes_gate(e), (mode, D.describe(e))
        assert e["bias_ratio"] <= 0.5, (mode, D.describe(e))


REJECTIONS = {}


def _bug_mode(bug, form):
    """GELU mode 2 (the default) except where its tanh.approx term hides the bug: the erf-vs-tanh formula difference, and truncation, which
    the rounding-bias check sees only where the GELU term is below 2 % of an ulp."""
    if form == "simt" or bug == "tanh_approx_gelu":
        return 0
    return 1 if bug == "bf16_truncation" else 2


@pytest.mark.parametrize("shape", SHAPES, ids=_sid)
@pytest.mark.parametrize("bug", list(D.BUGS))
def test_gate_rejects_emulated_bug(bug, shape):
    kind, changes = D.BUGS[bug]
    mode = _bug_mode(bug, shape[4])
    out, ref, a, m = _run(kind, shape, mode, bug)
    if changes(*shape):
        e = D.gate_errors(out, ref, a, m, mode, check_bias=kind not in ("coord", "gelu_sweep"))
        factor = D.gate_ratio(e)
        REJECTIONS[bug] = min(REJECTIONS.get(bug, math.inf), factor)
        assert factor >= MIN_REJECTION, (bug, kind, D.describe(e))
    else:
        honest, _, _, _ = _run(kind, shape, mode)
        assert torch.equal(out, honest), f"{bug} changes the output at {shape}, where it was expected not to"


@pytest.mark.parametrize("bug", list(D.BUGS))
def test_every_bug_is_exercised(bug):
    assert sum(bool(D.BUGS[bug][1](*s)) for s in SHAPES) >= 2


def test_rejection_factors(capsys):
    """Smallest factor by which the gate rejects each bug over the shapes (printed; the per-shape tests assert >= MIN_REJECTION)."""
    for bug, (kind, changes) in D.BUGS.items():
        if bug not in REJECTIONS:
            for s in SHAPES:
                if changes(*s):
                    mode = _bug_mode(bug, s[4])
                    out, ref, a, m = _run(kind, s, mode, bug)
                    e = D.gate_errors(out, ref, a, m, mode, check_bias=kind not in ("coord", "gelu_sweep"))
                    REJECTIONS[bug] = min(REJECTIONS.get(bug, math.inf), D.gate_ratio(e))
    with capsys.disabled():
        print("\nDWConv gate rejection factor per emulated bug (smallest over the shapes):")
        for bug, f in sorted(REJECTIONS.items(), key=lambda t: t[1]):
            print(f"  {bug:30s} {f:12.1f}x  ({D.BUGS[bug][0]})")
    assert min(REJECTIONS.values()) >= MIN_REJECTION


def test_reference_layout_and_nan_planting():
    """The reference is GELU(sum_t w[t] x[h + kh - 1, w + kw - 1] + b) with zero padding per frame; a planted NaN poisons exactly its 3x3
    neighbourhood within its frame and channel."""
    d = D.make_inputs("coord", 2, 5, 6, 8, seed=3)
    ref, a, m = D.reference(d["x"], d["w9c"], d["bias"])
    x, w, b = d["x"].double(), d["w9c"].double(), d["bias"].double()
    for (f, h, ww, c) in ((0, 0, 0, 0), (1, 4, 5, 7), (1, 2, 3, 4), (0, 4, 0, 1)):
        s = float(b[c])
        for kh in range(3):
            for kw in range(3):
                hh, wx = h + kh - 1, ww + kw - 1
                if 0 <= hh < 5 and 0 <= wx < 6:
                    s += float(w[kh * 3 + kw, c] * x[f, hh, wx, c])
        assert abs(float(a[f, h, ww, c]) - s) < 1e-12
    d = D.make_inputs("nan_plant", 2, 9, 17, 8, seed=3, tw=8)
    ref, _, _ = D.reference(d["x"], d["w9c"], d["bias"])
    assert torch.equal(torch.isnan(ref), expected_nan_mask(torch.isnan(d["x"].float())))
    sites = D.nan_sites(2, 9, 17, 8, 8)
    assert {(h, w) for _, h, w, _ in sites} >= {(0, 0), (8, 16), (6, 7), (7, 8), (0, 8)}


def expected_nan_mask(nan_in: torch.Tensor) -> torch.Tensor:
    """Where a NaN input poisons the output: its 3x3 neighbourhood within the frame, same channel."""
    p = torch.nn.functional.pad(nan_in.float(), (0, 0, 1, 1, 1, 1))
    H, W = nan_in.shape[1], nan_in.shape[2]
    return sum(p[:, kh:kh + H, kw:kw + W] for kh in range(3) for kw in range(3)) > 0


# ------------------------------------------------------------------------------------------------------- argument errors, no device
BASE = 1 << 20   # dummy device addresses: the argument checks fail before anything is read through them


@pytest.mark.parametrize("B,H,W,C,msg", [(1, 8, 8, 6, "row stride"), (2, 8, 8, 130, "row stride"), (10000, 49, 8, 64, "grid limits"),
                                         (9363, 49, 8, 64, "grid limits"), (0, 8, 8, 64, "positive"), (1, 8, 0, 128, "positive")])
def test_dwconv_argument_errors(B, H, W, C, msg):
    """C % 4 != 0, the SIMT kernel's grid limit B * ceil(H / 7) <= 65535 (9363 * 7 = 65541) and empty shapes fail with SV_ERR_INVALID
    before the device is touched."""
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import _native

    lib = _native.lib()
    rc = lib.sv_op_dwconv3x3_gelu(BASE, BASE + 65536, BASE + 2 * 65536, B, H, W, C, BASE + 3 * 65536, None)
    assert rc == 1 and msg.encode() in lib.sv_last_error(), lib.sv_last_error()
    info = (ctypes.c_int32 * 14)()
    assert lib.sv_op_dwconv_plan_info(B, H, W, C, 148, info) == 1


# ------------------------------------------------------------------------------------------------------- plan query vs the formulas
def formula_plan(B, H, W, C, sms=148, cpl=4, stages=4, prefetch=2, gelu=2):
    """The plan dwconv_tma.cu / elementwise.cu document, computed here independently."""
    if C % 128:
        tx, ty, cb = -(-W // 8), -(-H // 7), -(-C // 128)
        n = tx * ty * cb * B
        return dict(kernel="simt", cpl=4, gelu=0, stages=0, prefetch=0, tw=8, tiles_x=tx, tiles_y=ty, cblks=cb, num_tiles=n, grid=n,
                    max_tiles_per_cta=1, crosses_frame=0, crosses_cblk=0)
    tw = 8 if W % 8 == 0 else (7 if W % 7 == 0 else 8)
    tx, ty, cb = -(-W // tw), -(-H // 7), C // (32 * cpl)
    n = cb * B * ty * tx
    grid = min(n, (2 if cpl == 4 else 4) * sms)
    per, extra = divmod(n, grid)
    ranges = []
    for i in range(grid):
        tb = i * per + min(i, extra)
        ranges.append(range(tb, tb + per + (i < extra)))
    frame = lambda t: t // (ty * tx)
    cblk = lambda t: t // (B * ty * tx)
    return dict(kernel="tma", cpl=cpl, gelu=gelu, stages=stages, prefetch=prefetch, tw=tw, tiles_x=tx, tiles_y=ty, cblks=cb, num_tiles=n,
                grid=grid, max_tiles_per_cta=max(len(r) for r in ranges),
                crosses_frame=int(any(frame(r[0]) != frame(r[-1]) for r in ranges)),
                crosses_cblk=int(any(cblk(r[0]) != cblk(r[-1]) for r in ranges)))


def test_plan_query_matches_formulas_on_the_gpu_case_table():
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import ops
    import test_dwconv_gpu as T

    for c in T.CASES:
        assert ops.dwconv_plan_info(*c, num_sms=148) == formula_plan(*c), c
    p = ops.dwconv_plan_info(45, 56, 56, 256, num_sms=148)
    assert (p["num_tiles"], p["grid"], p["max_tiles_per_cta"], p["crosses_frame"], p["crosses_cblk"]) == (5040, 296, 18, 1, 1), p
    assert ops.dwconv_plan_info(2, 56, 56, 256, num_sms=148)["max_tiles_per_cta"] == 1
