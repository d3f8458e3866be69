"""DWConv3x3 + bias + GELU on the GPU (`sv_op_dwconv3x3_gelu`: the TMA kernel of dwconv_tma.cu for C % 128 == 0, the SIMT kernel of
elementwise.cu otherwise) against the float64 reference of tests/dw_ref.py under its format-derived gate: a case table that reaches, by
the plan query, both kernels, every column-tile width, every H % 7, tiny frames, the model's stage shapes and CTA ranges long enough for
the shared-memory ring to wrap several times across frame and channel-block boundaries; every stress input; exact NaN isolation, frame
independence and repeatability; a sentinel guard behind the output; the A/B switches in a fresh process; the exhaustive GELU sweep of
each GELU form; and the fused mixffn_fc2 kernel under the GEMM gate plus its DWConv terms."""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch

import dw_ref as D
import gemm_ref as G
import surgvid_b200  # noqa: F401
from surgvid_b200 import _native, ops
from test_dwconv_gate_cpu import expected_nan_mask

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (B, H, W, C).  SIMT kernel: C in {4, 12, 64, 192, 320}.  TMA kernel: tw = 8 with W % 8 == 0, tw = 7 (W = 7, 14, 35), ragged tw = 8
# (W = 5, 27, 107, 214); H % 7 = 0 ... 6; H = W = 1; the stage shapes of mit_b3_evp at 224^2 and 480x854; 45 x 56 x 56 x 256: 5040 tiles,
# 18 per CTA at 148 SMs, CTA ranges that cross frames and the channel-block boundary.
CASES = [
    (2, 9, 5, 4), (1, 15, 27, 12), (2, 17, 56, 64), (3, 13, 14, 192), (2, 12, 35, 320), (3, 1, 1, 4),
    (1, 29, 16, 128), (2, 11, 7, 128), (1, 12, 35, 256), (2, 9, 5, 128), (1, 20, 27, 256), (1, 13, 107, 128), (1, 17, 214, 256),
    (1, 1, 1, 128), (2, 1, 1, 256),
    (2, 56, 56, 256), (2, 28, 28, 512), (2, 14, 14, 1280), (2, 7, 7, 2048),
    (1, 120, 214, 256), (1, 60, 107, 512), (1, 30, 54, 1280), (1, 15, 27, 2048),
    (45, 56, 56, 256),
]
LONG = (45, 56, 56, 256)
GATE_KINDS = ("randn", "asym_taps", "coord", "cancel", "bigbias")
SENTINEL = 0x7FA5            # a bf16 NaN the kernels never produce (their NaN is 0x7FFF)
GUARD = 4096                 # bf16 elements behind the output in the same allocation
SEEN = {}                    # worst gate terms over the run, printed by test_report_gate_terms


def _id(c):
    return "x".join(map(str, c))


def _mode(plan):
    return plan["gelu"] if plan["kernel"] == "tma" else 0


def call_guarded(d):
    """sv_op_dwconv3x3_gelu through the C ABI into the head of a sentinel-filled buffer -> (output, every element written, guard intact)."""
    x, w, b = d["x"].to(DEV), d["w9c"].to(DEV), d["bias"].to(DEV)
    B, H, W, C = x.shape
    n = x.numel()
    buf = torch.full((n + GUARD,), SENTINEL, dtype=torch.int16, device=DEV)
    lib = _native.lib()
    rc = lib.sv_op_dwconv3x3_gelu(x.data_ptr(), w.data_ptr(), b.data_ptr(), B, H, W, C, buf.data_ptr(),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _native.check(rc, "sv_op_dwconv3x3_gelu")
    torch.cuda.synchronize()
    out = buf[:n].view(torch.bfloat16).view(B, H, W, C)
    return out, bool((buf[:n] != SENTINEL).all()), bool((buf[n:] == SENTINEL).all())


def _note(key, e):
    s = SEEN.setdefault(key, {"ratio": 0.0, "tau_acc_seen": 0.0})
    s["ratio"] = max(s["ratio"], e["ratio"])
    s["tau_acc_seen"] = max(s["tau_acc_seen"], e["tau_acc_seen"])


# ------------------------------------------------------------------------------------------------------- case table
def test_case_table_reaches_every_form():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    plans = {c: ops.dwconv_plan_info(*c) for c in CASES}
    simt = {c[3] for c, p in plans.items() if p["kernel"] == "simt"}
    assert simt == {4, 12, 64, 192, 320}, simt
    tma = {c: p for c, p in plans.items() if p["kernel"] == "tma"}
    assert {c[2] for c, p in tma.items() if p["tw"] == 8 and c[2] % 8 == 0} and {c[2] for c, p in tma.items() if p["tw"] == 7} >= {7, 14, 35}
    assert {c[2] for c, p in tma.items() if p["tw"] == 8 and c[2] % 8} >= {5, 27, 107, 214}
    assert {c[1] % 7 for c in CASES} == set(range(7)) and {c[1] % 7 for c in tma} == set(range(7))
    assert any(c[1] == c[2] == 1 for c in tma) and any(c[1] == c[2] == 1 for c in CASES if c not in tma) and any(c[0] == 1 for c in tma)
    p = plans[LONG]
    print(f"\n{_id(LONG)} at {sms} SMs: {p}")
    assert p["max_tiles_per_cta"] > 2 * p["stages"] and p["crosses_frame"] and p["crosses_cblk"], p


# ------------------------------------------------------------------------------------------------------- gate, guard, repeatability
@pytest.mark.parametrize("kind", GATE_KINDS)
@pytest.mark.parametrize("c", CASES, ids=_id)
def test_dwconv_matches_fp64_reference(c, kind):
    """Gate against float64; every output element written and nothing past it; a second run bit-identical."""
    d = D.make_inputs(kind, *c, seed=10 * CASES.index(c) + GATE_KINDS.index(kind), device=DEV)
    plan = ops.dwconv_plan_info(*c)
    mode = _mode(plan)
    out, written, guard_ok = call_guarded(d)
    assert written, f"{_id(c)}: some output elements were never written"
    assert guard_ok, f"{_id(c)}: wrote past the end of its output"
    ref, a, m = D.reference(d["x"], d["w9c"], d["bias"])
    e = D.assert_gate(out, ref, a, m, mode, f"{_id(c)} {kind} {plan['kernel']} gelu {mode}", check_bias=kind != "coord")
    _note((plan["kernel"], mode), e)
    again, _, _ = call_guarded(d)
    assert torch.equal(out.view(torch.int16), again.view(torch.int16)), f"{_id(c)}: second run differs"


NAN_CASES = [c for c in CASES if c[0] * c[1] * c[2] * c[3] <= 4_000_000 and c[1] * c[2] > 1]


@pytest.mark.parametrize("c", NAN_CASES, ids=_id)
def test_planted_nan_poisons_exactly_its_neighbourhood(c):
    """NaN at frame corners, row- and column-tile seams and the first and last rows: NaN in exactly its 3x3 neighbourhood, clipped to its
    frame, in its own channel; everything else finite and within the gate."""
    plan = ops.dwconv_plan_info(*c)
    d = D.make_inputs("nan_plant", *c, seed=5, device=DEV, tw=plan["tw"])
    out, written, guard_ok = call_guarded(d)
    assert written and guard_ok
    want = expected_nan_mask(torch.isnan(d["x"].float()))
    got = torch.isnan(out.float())
    assert torch.equal(got, want), f"{_id(c)}: {int((got != want).sum())} elements differ, first at {tuple((got != want).nonzero()[0].tolist())}"
    ref, a, m = D.reference(d["x"], d["w9c"], d["bias"])
    D.assert_gate(out, ref, a, m, _mode(plan), f"{_id(c)} nan_plant")


@pytest.mark.parametrize("c", [c for c in CASES if c[0] > 1], ids=_id)
def test_frames_are_independent(c):
    """dwconv(x)[b] == dwconv(x[b:b+1]) bit for bit: no halo or tile crosses a frame."""
    d = D.make_inputs("coord", *c, seed=2, device=DEV)
    out = ops.dwconv3x3_gelu(d["x"], d["w9c"], d["bias"])
    for b in sorted({0, c[0] // 2, c[0] - 1}):
        one = ops.dwconv3x3_gelu(d["x"][b:b + 1].contiguous(), d["w9c"], d["bias"])
        assert torch.equal(out[b:b + 1].view(torch.int16), one.view(torch.int16)), f"{_id(c)}: frame {b} depends on its neighbours"


# ------------------------------------------------------------------------------------------------------- A/B switches (fresh process)
SWITCH_CASES = [(2, 56, 56, 256), (1, 20, 27, 256), (2, 11, 7, 128), (2, 7, 7, 2048), (1, 1, 1, 128), (1, 17, 214, 256), LONG, (2, 12, 35, 320)]
SWEEP_CASE = (2, 16, 16, 128)                 # 65 536 outputs: every finite bf16 value once through the TMA kernel
SWITCHES = {
    "CPL=2": {"SURGVID_DW_CPL": "2"},
    "STAGES=2,PREFETCH=1": {"SURGVID_DW_STAGES": "2", "SURGVID_DW_PREFETCH": "1"},
    "STAGES=8,PREFETCH=1": {"SURGVID_DW_STAGES": "8", "SURGVID_DW_PREFETCH": "1"},
    "STAGES=8,PREFETCH=7": {"SURGVID_DW_STAGES": "8", "SURGVID_DW_PREFETCH": "7"},
    "GELU=0": {"SURGVID_DW_GELU": "0"},
    "GELU=1": {"SURGVID_DW_GELU": "1"},
    "CPL=2,GELU=0": {"SURGVID_DW_CPL": "2", "SURGVID_DW_GELU": "0"},
    "CPL=2,GELU=1": {"SURGVID_DW_CPL": "2", "SURGVID_DW_GELU": "1"},
}
BIT_IDENTICAL = {"CPL=2": None, "STAGES=2,PREFETCH=1": None, "STAGES=8,PREFETCH=1": None, "STAGES=8,PREFETCH=7": None,
                 "CPL=2,GELU=0": "GELU=0", "CPL=2,GELU=1": "GELU=1"}   # switch -> the run it must equal (None: the default)


def _switch_inputs():
    ins = [D.make_inputs("randn", *c, seed=i) for i, c in enumerate(SWITCH_CASES)]
    return ins + [D.make_inputs("gelu_sweep", *SWEEP_CASE)]


def run_in_child(cases, env_overrides, tmp_path):
    """dw_ref.py as a script in a fresh process with the given switches -> (outputs, plans)."""
    torch.save(cases, tmp_path / "in.pt")
    env = {k: v for k, v in os.environ.items() if not k.startswith("SURGVID_DW_")}
    env.update(env_overrides)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [D.__file__, str(tmp_path / "in.pt"), str(tmp_path / "out.pt")]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    res = torch.load(tmp_path / "out.pt")
    return res["outs"], res["plans"]


@pytest.fixture(scope="module")
def switch_runs(tmp_path_factory):
    """The switch cases on the default path (this process; no SURGVID_DW_* switch may be set here) and under every switch."""
    assert not any(k.startswith("SURGVID_DW_") for k in os.environ), "run the DWConv tests without SURGVID_DW_* switches"
    ins = _switch_inputs()
    runs = {None: D.run_cases(ins)}
    for name, env in SWITCHES.items():
        runs[name] = run_in_child(ins, env, tmp_path_factory.mktemp(name.replace(",", "_").replace("=", "")))
    return ins, runs


@pytest.mark.parametrize("name", list(SWITCHES))
def test_switch_passes_gate_and_keeps_bits(name, switch_runs):
    """Each switch changes the plan as it says and passes its own GELU form's gate.  CPL, stages and prefetch only move tiles between CTAs and
    channels between lanes (every output's arithmetic is the same), so those runs are bit-identical to the run with the same GELU form."""
    ins, runs = switch_runs
    outs, plans = runs[name]
    env = SWITCHES[name]
    for c, d, o, p in zip(SWITCH_CASES + [SWEEP_CASE], ins, outs, plans):
        what = f"{_id(c)} {name}"
        if p["kernel"] == "tma":
            assert p["cpl"] == int(env.get("SURGVID_DW_CPL", 4)) and p["gelu"] == int(env.get("SURGVID_DW_GELU", 2)), (what, p)
            if "SURGVID_DW_STAGES" in env:
                assert (p["stages"], p["prefetch"]) == (int(env["SURGVID_DW_STAGES"]), int(env["SURGVID_DW_PREFETCH"])), (what, p)
            if c == LONG:
                assert p["max_tiles_per_cta"] > 2 * p["stages"] and p["crosses_frame"] and p["crosses_cblk"], (what, p)
        ref, a, m = D.reference(d["x"].to(DEV), d["w9c"], d["bias"])
        e = D.assert_gate(o, ref, a, m, _mode(p), what, check_bias=c != SWEEP_CASE)
        _note((p["kernel"], _mode(p)), e)
        if name in BIT_IDENTICAL:
            base = runs[BIT_IDENTICAL[name]][0][(SWITCH_CASES + [SWEEP_CASE]).index(c)]
            assert torch.equal(o.view(torch.int16), base.view(torch.int16)), f"{what}: differs from {BIT_IDENTICAL[name] or 'the default'}"


def test_every_kernel_form_reached(switch_runs):
    _, runs = switch_runs
    forms = {(p["kernel"], p["cpl"], _mode(p)) for outs, plans in runs.values() for p in plans}
    print(f"\nDWConv (kernel, cpl, gelu) forms run: {sorted(forms)}")
    assert forms >= {("simt", 4, 0)} | {("tma", cpl, g) for cpl in (2, 4) for g in (0, 1, 2)}, forms


def _ulps(out, ref):
    return ((out.double() - ref).abs() / G._bf16_ulp(ref)).nan_to_num(0.0)


def test_gelu_tail_per_mode(switch_runs, capsys):
    """Every finite bf16 value through GELU mode 0, 1 and 2 of the TMA kernel (gelu_sweep: a == x exactly).  Prints the worst error in bf16
    ulps of the output for x < 0 (bands of x) and x >= 0, and the smallest per-|a| term that covers mode 2 beside the 2.5e-4 common.cuh
    states; the gate itself was asserted by test_switch_passes_gate_and_keeps_bits and here for the default."""
    ins, runs = switch_runs
    d = ins[-1]
    x = d["x"].double().to(DEV)
    ref = D.gelu64(x)
    normal = ref.abs() >= 2.0 ** -126
    bands = [(-3.0, 0.0), (-4.0, -3.0), (-6.0, -4.0), (-math.inf, -6.0), (0.0, math.inf)]
    lines = []
    for name, mode in ((None, 2), ("GELU=0", 0), ("GELU=1", 1)):
        out = runs[name][0][-1].to(DEV)
        assert runs[name][1][-1]["gelu"] == mode
        u = _ulps(out, ref)
        err = (out.double() - ref).abs()
        row = []
        for lo, hi in bands:
            sel = (x >= lo) & (x < hi) & normal
            row.append(f"x in [{lo:g}, {hi:g}): {float(u[sel].max()):10.1f} ulp, |err| {float(err[(x >= lo) & (x < hi)].max()):.2e}")
        lines.append((mode, row))
        if mode == 2:
            tail = ((err - 3.0e-5 - D.TAU_OUT * ref.abs() - D.TAU_ACC * D.GELU_LIP * x.abs()).clamp_min(0) / x.abs().clamp_min(1e-300)).max()
            lines.append((2, [f"smallest per-|a| term covering mode 2: {float(tail):.3e} (common.cuh: 2.5e-4)"]))
        D.assert_gate(out, ref, x, x.abs(), mode, f"gelu_sweep mode {mode}", check_bias=False)
    with capsys.disabled():
        print(f"\nGELU error over every finite bf16 value ({torch.cuda.get_device_name(0)}):")
        for mode, row in lines:
            for r in row:
                print(f"  mode {mode}  {r}")


# ------------------------------------------------------------------------------------------------------- mixffn_fc2
MIXFFN = [
    # (frames, H, W, hidden, N, tail_cols): the three fusable stages of mit_b3_evp at 224^2, a no-tail case, ragged row tiles, enough
    # frames that every CTA of the persistent grid walks several tiles, 480x854 stage 3; then ragged shapes
    (3, 14, 14, 1280, 320, 80), (2, 56, 56, 256, 64, 16), (2, 28, 28, 512, 128, 32), (2, 14, 14, 1280, 320, 0),
    (2, 11, 12, 128, 64, 0), (1, 9, 14, 64, 32, 8), (200, 14, 14, 1280, 320, 80), (3, 30, 54, 1280, 320, 80),
    (3, 13, 6, 192, 48, 8), (1, 5, 2, 64, 16, 0), (2, 9, 26, 320, 96, 24),
]


@pytest.mark.parametrize("cfg", MIXFFN, ids=_id)
def test_mixffn_fc2_gate(cfg):
    """x += bias + GELU(dwconv3x3(h1) + b_dw) @ W[:, :hidden].T + tail @ W[:, hidden:].T in float64, under the GEMM gate on h2 = GELU(...)
    plus the bf16 rounding of h2 (2^-8 |h2| |W|^T) and the DWConv terms (accumulation and the polynomial's tau) through |W|^T."""
    B, H, W, hid, N, tc = cfg
    g = torch.Generator().manual_seed(MIXFFN.index(cfg))
    rn = lambda *s: torch.randn(s, generator=g).to(DEV)
    h1 = rn(B, H, W, hid).to(torch.bfloat16)
    w9c = (rn(9, hid) / 3).contiguous()
    bdw = 0.2 * rn(hid)
    wcat = (rn(N, hid + tc) / math.sqrt(hid)).to(torch.bfloat16)
    bias = 0.3 * rn(N)
    tail = rn(B * H * W, tc).to(torch.bfloat16) if tc else None
    x0 = rn(B * H * W, N)
    x = ops.mixffn_fc2(h1, w9c, bdw, wcat, bias, x0.clone(), tail)
    torch.cuda.synchronize()
    h, _, m_dw = D.reference(h1, w9c, bdw)
    M = B * H * W
    h, m_dw = h.reshape(M, hid), m_dw.reshape(M, hid)
    Wh = wcat[:, :hid].double()
    ref = x0.double() + bias.double() + h @ Wh.T
    mag_h = h.abs() @ Wh.abs().T
    mag = mag_h + bias.double().abs()
    if tc:
        Wt = wcat[:, hid:].double()
        ref += tail.double() @ Wt.T
        mag += tail.double().abs() @ Wt.abs().T
    dw_err = (D.TAU_ACC * D.GELU_LIP * m_dw + D.GELU_TAU[0][0]) @ Wh.abs().T
    bound = G.TAU_ACC * mag + D.TAU_OUT * mag_h + dw_err + G.TAU_OUT[True] * ref.abs()
    assert bool(torch.isfinite(x).all())
    q = (x.double() - ref).abs() / bound
    i = int(q.argmax())
    SEEN[("mixffn", 0)] = {"ratio": max(SEEN.get(("mixffn", 0), {"ratio": 0.0})["ratio"], float(q.max())), "tau_acc_seen": float("nan")}
    assert float(q.max()) <= 1.0, f"{cfg}: worst |err|/bound {float(q.max()):.3g} at row {i // N} col {i % N}"
    del h, m_dw, ref, mag, mag_h, dw_err, bound, q
    torch.cuda.empty_cache()


def test_report_gate_terms(capsys):
    """The worst gate ratio and the smallest TAU_ACC each (kernel, GELU form) would have passed with, over this run (printed)."""
    with capsys.disabled():
        print(f"\nDWConv gate over this run ({torch.cuda.get_device_name(0)}), TAU_ACC = {D.TAU_ACC:.3g}:")
        for k, v in sorted(SEEN.items()):
            print(f"  {k[0]:6s} gelu {k[1]}: worst |err|/bound {v['ratio']:.3f}, accumulation term needed {v['tau_acc_seen']:.3g}")
