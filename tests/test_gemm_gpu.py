"""The tcgen05 GEMM on the GPU (`sv_op_gemm_bf16`, `sv_op_gemm_bf16_cat`) against the float64 reference of tests/gemm_ref.py under its
format-derived gate: a case table annotated with the plan each case must get (every UMMA width, every ring depth, each epilogue form single
and as a CTA pair, ragged K / M / N edges, several tiles per CTA), every act x bias x output form, the A/B switches in a fresh process, and
isolation: NaN-filled operand padding that must never be read, a NaN-filled output buffer whose margins must keep their bits, bit-identical
repeats, and outputs past 2^31 elements.

Epilogue forms (SV_GEMM_EPI_*): bf16_tma (bf16 result, no residual), f32_tma (fp32 result), f32_tma_resid (fp32 result + fp32 residual
through a ring of TMA loads), transpose (bf16 result + residual, and everything under SURGVID_GEMM_TMA_OUT=0)."""
import os
import subprocess
import sys

import pytest
import torch

import gemm_ref as G
import surgvid_b200  # noqa: F401
from surgvid_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PLAN_SMS = 148   # the annotations below are the plans at this SM count (B200)

FORMS = {"bf16_tma": (False, False), "f32_tma": (True, False), "f32_tma_resid": (True, True), "transpose": (False, True)}   # out_fp32, residual

# (epilogue form, M, N, K, K2, pair request (-1 auto), annotated plan at 148 SMs: block_n, pair, num_stages)
CASES = [
    # fp32 result: every UMMA width 16 ... 256
    ("f32_tma", 1, 8, 8, 0, -1, 16, 0, 8),
    ("f32_tma", 300, 792, 72, 0, -1, 32, 0, 7),
    ("f32_tma", 300, 1576, 136, 0, -1, 48, 0, 6),
    ("f32_tma", 12000, 56, 200, 0, -1, 64, 0, 6),
    ("f32_tma", 12000, 72, 56, 0, -1, 80, 0, 5),
    ("f32_tma", 7000, 136, 64, 0, -1, 96, 0, 5),
    ("f32_tma", 12000, 104, 80, 0, -1, 112, 0, 5),
    ("f32_tma", 12000, 120, 120, 0, -1, 128, 0, 4),
    ("f32_tma", 12000, 136, 16, 0, -1, 144, 0, 4),
    ("f32_tma", 12000, 152, 264, 0, -1, 160, 0, 4),
    ("f32_tma", 12000, 168, 328, 0, -1, 176, 0, 4),
    ("f32_tma", 12000, 184, 392, 0, -1, 192, 0, 3),
    ("f32_tma", 12000, 200, 24, 0, -1, 208, 0, 3),
    ("f32_tma", 12000, 216, 48, 0, -1, 224, 0, 3),
    ("f32_tma", 12000, 232, 144, 0, -1, 240, 0, 3),
    ("f32_tma", 12000, 248, 208, 0, -1, 256, 0, 3),
    # bf16 result through TMA stores: every multiple of 32
    ("bf16_tma", 1, 8, 64, 0, -1, 32, 0, 7),
    ("bf16_tma", 300, 1576, 80, 0, -1, 64, 0, 6),
    ("bf16_tma", 12000, 72, 120, 0, -1, 96, 0, 5),
    ("bf16_tma", 12000, 104, 16, 0, -1, 128, 0, 4),
    ("bf16_tma", 12000, 136, 264, 0, -1, 160, 0, 4),
    ("bf16_tma", 12000, 168, 328, 0, -1, 192, 0, 3),
    ("bf16_tma", 12000, 200, 392, 0, -1, 224, 0, 3),
    ("bf16_tma", 12000, 232, 24, 0, -1, 256, 0, 3),
    # fp32 result + residual ring; (300 | 1000) x 272: the last N tile has 16 columns, so warps of the odd half own no chunk of it
    ("f32_tma_resid", 777, 64, 256, 0, -1, 16, 0, 8),
    ("f32_tma_resid", 5000, 176, 200, 0, -1, 64, 0, 6),
    ("f32_tma_resid", 3000, 48, 72, 0, -1, 16, 0, 8),
    ("f32_tma_resid", 1000, 320, 1280, 0, -1, 32, 0, 7),
    ("f32_tma_resid", 300, 272, 64, 0, 0, 32, 0, 7),
    ("f32_tma_resid", 1000, 272, 120, 0, 1, 32, 1, 8),
    ("f32_tma_resid", 39200, 320, 1360, 80, -1, 160, 1, 5),     # the model's fc2 + adapter: pair, two segments, 4+ tiles per CTA
    # transposing epilogue (bf16 result + fp32 residual)
    ("transpose", 1000, 320, 200, 0, -1, 32, 0, 8),
    ("transpose", 129, 24, 72, 0, -1, 16, 0, 8),
    ("transpose", 4000, 256, 136, 0, -1, 64, 0, 7),
    ("transpose", 300, 520, 1024, 0, -1, 16, 0, 8),
    ("transpose", 1000, 320, 200, 0, 1, 32, 1, 8),
    ("transpose", 1100, 96, 56, 0, 1, 32, 1, 8),                # pair, M % 256 = 76: the second CTA of the last pair gets no rows
    ("transpose", 1000, 128, 576, 64, 1, 32, 1, 8),
    # pair mode elsewhere, second A segments, several tiles per CTA
    ("bf16_tma", 300, 1280, 320, 0, 1, 32, 1, 8),
    ("bf16_tma", 3000, 2048, 512, 0, -1, 192, 1, 5),
    ("bf16_tma", 1000, 128, 576, 64, -1, 32, 0, 7),
    ("f32_tma", 5000, 1280, 520, 0, -1, 192, 1, 5),
    ("f32_tma", 1100, 200, 16, 0, 1, 32, 1, 8),
    ("f32_tma", 98, 2048, 8192, 0, -1, 32, 1, 8),
    ("f32_tma", 5000, 320, 72, 8, -1, 112, 0, 5),
    ("f32_tma", 148 * 128 * 3 + 77, 256, 192, 0, -1, 256, 0, 3),   # 3 tiles per CTA: ring and accumulator phases wrap
]


def _id(c):
    return f"{c[0]}-{c[1]}x{c[2]}x{c[3]}" + (f"+{c[4]}" if c[4] else "") + ({0: "-single", 1: "-pair"}.get(c[5], ""))


def _kinds(i, c):
    pool = G.STRESS[1:] if FORMS[c[0]][1] else ("colbias", "gelu_sweep", "cancel")
    return ["randn", pool[i % len(pool)]]


def _act(i, kind):
    return G.ACT_GELU if kind == "gelu_sweep" else i % 3


def _nan_padded(x, left=0, right=8):
    """The values of x as a view into a wider NaN-filled buffer (left / right pad columns), so any read past the view shows."""
    buf = torch.full((x.shape[0], left + x.shape[1] + right), float("nan"), dtype=x.dtype, device=x.device)
    buf[:, left:left + x.shape[1]] = x
    return buf[:, left:left + x.shape[1]]


def make_case(form, M, N, K, K2=0, kind="randn", act=G.ACT_NONE, seed=0, bias=True, in_place=False):
    out_fp32, res = FORMS[form]
    d = G.make_inputs(kind, M, N, K, K2, seed=seed, device=DEV, bias=bias, residual=res)
    d["a"], d["w"] = _nan_padded(d["a"]), _nan_padded(d["w"])
    if K2:
        d["a2"] = _nan_padded(d["a2"], left=8)     # a column slice of a wider tensor, as the model's adapter tokens
    if res:
        d["residual"] = _nan_padded(d["residual"])  # ldr = N + 8 != ldc
    d.update(act=act, out_fp32=out_fp32, in_place=in_place, out_margin=(2, 8))
    return d


def check_plan(c, plan, sms):
    form, _, _, _, _, pair_req, block_n, pair, stages = c
    assert plan["epilogue"] == form, (_id(c), plan)
    if pair_req >= 0:
        assert plan["pair"] == pair_req, (_id(c), plan)
    if sms == PLAN_SMS:
        assert (plan["block_n"], plan["pair"], plan["num_stages"]) == (block_n, pair, stages), (_id(c), plan)


def _margins_keep_nan(out, buf, margin=(2, 8)):
    keep = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    gr, gc = margin
    keep[gr:gr + out.shape[0], gc:gc + out.shape[1]] = False
    ibits = torch.int32 if buf.dtype == torch.float32 else torch.int16
    nan_bits = torch.full((1,), float("nan"), dtype=buf.dtype, device=buf.device).view(ibits)
    return bool((buf.view(ibits)[keep] == nan_bits).all())


def _ref(d):
    return G.reference(d["a"], d["w"], d["bias"], d["act"], d["residual"], d.get("a2"))


def _set_pair(monkeypatch, pair_req):
    if pair_req >= 0:
        monkeypatch.setenv("SURGVID_GEMM_PAIR", str(pair_req))
    else:
        monkeypatch.delenv("SURGVID_GEMM_PAIR", raising=False)


PARAMS = [pytest.param(c, kind, _act(i, kind), id=f"{_id(c)}-{kind}-act{_act(i, kind)}") for i, c in enumerate(CASES) for kind in _kinds(i, c)]


@pytest.mark.parametrize("c,kind,act", PARAMS)
def test_gemm_matches_fp64_reference(c, kind, act, monkeypatch):
    """Gate against float64, the annotated plan, NaN operand padding never read, output margins untouched, repeat bit for bit."""
    form, M, N, K, K2, pair_req = c[:6]
    _set_pair(monkeypatch, pair_req)
    d = make_case(form, M, N, K, K2, kind, act, seed=7)
    plan = G.plan_info(d)
    check_plan(c, plan, torch.cuda.get_device_properties(0).multi_processor_count)
    out, buf = G.call(d)
    ref, mag = _ref(d)
    G.assert_gate(out, ref, mag, act, FORMS[form][0], f"{_id(c)} {kind} act {act}", plan["block_n"], check_bias=kind != "rowid")
    assert _margins_keep_nan(out, buf), f"{_id(c)}: wrote outside its output block"
    again, _ = G.call(d)
    assert torch.equal(out, again), f"{_id(c)}: second run differs"


# ------------------------------------------------------------------------------------------------------- act x bias x output form
RESID_MODES = [(False, "none"), (False, "separate"), (True, "none"), (True, "separate"), (True, "in_place")]   # (out_fp32, residual)


@pytest.mark.parametrize("shape", [(1000, 320, 200), (300, 272, 64)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("out_fp32,resid", RESID_MODES, ids=[f"{'f32' if f else 'bf16'}-{r}" for f, r in RESID_MODES])
@pytest.mark.parametrize("bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("act", [G.ACT_NONE, G.ACT_GELU, G.ACT_RELU], ids=["none", "gelu", "relu"])
def test_gemm_act_bias_output_forms(shape, out_fp32, resid, bias, act):
    M, N, K = shape
    form = ("f32_tma_resid" if resid != "none" else "f32_tma") if out_fp32 else ("transpose" if resid != "none" else "bf16_tma")
    d = make_case(form, M, N, K, kind="randn", act=act, seed=11, bias=bias, in_place=resid == "in_place")
    ref, mag = _ref(d)                                        # before an in-place call overwrites the residual's copy
    out, buf = G.call(d)
    G.assert_gate(out, ref, mag, act, out_fp32, f"{shape} {form} {resid} bias={bias} act={act}")
    if resid != "in_place":
        assert _margins_keep_nan(out, buf)


# ------------------------------------------------------------------------------------------------------- A/B switches (fresh process)
SWITCH_CASES = [c for c in CASES if c[5] < 0 and c[1] * c[2] <= 4_000_000][::3] + [c for c in CASES if c[1] == 39200]   # + the fc2 form
SWITCHES = [{"SURGVID_GEMM_TMA_OUT": "0"}] + [
    {"SURGVID_GEMM_EPI_BUFS": str(b), "SURGVID_GEMM_EPI_LAG": str(lag)} for b in (2, 3, 4) for lag in range(1, b)] + [
    {"SURGVID_GEMM_PREFETCH": "2"}, {"SURGVID_GEMM_PREFETCH": "8"}, {"SURGVID_GEMM_PAIR": "0"}, {"SURGVID_GEMM_PAIR": "1"}]


def _switch_inputs():
    out = []
    for i, c in enumerate(SWITCH_CASES):
        act = (G.ACT_GELU, G.ACT_NONE, G.ACT_RELU)[i % 3]
        out.append(make_case(c[0], c[1], c[2], c[3], c[4], "randn", act, seed=i))
    return out


def run_in_child(cases, env_overrides, tmp_path):
    """gemm_ref.py as a script in a fresh process with the given switches -> (outputs, plans, margins intact)."""
    torch.save([{k: (v.cpu() if torch.is_tensor(v) else v) for k, v in d.items()} for d in cases], tmp_path / "in.pt")
    env = {k: v for k, v in os.environ.items() if not k.startswith("SURGVID_GEMM_")}
    env.update(env_overrides)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [G.__file__, str(tmp_path / "in.pt"), str(tmp_path / "out.pt")]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    res = torch.load(tmp_path / "out.pt")
    return res["outs"], res["plans"], res["intact"]


@pytest.fixture(scope="module")
def switch_default():
    """The switch cases on the default path, in this process (no SURGVID_GEMM_* switch may be set here)."""
    assert not any(k.startswith("SURGVID_GEMM_") for k in os.environ), "run the GEMM tests without SURGVID_GEMM_* switches"
    ins = _switch_inputs()
    outs, plans, intact = G.run_cases(ins)
    assert all(intact)
    return ins, outs, plans


@pytest.mark.parametrize("sw", SWITCHES, ids=lambda s: ",".join(f"{k[13:]}={v}" for k, v in s.items()))
def test_switch_matches_reference_and_default_bit_for_bit(sw, switch_default, tmp_path):
    """Each switch changes the plan as it says and passes the gate.  It also changes nothing in the arithmetic: every epilogue adds the
    bias, applies the activation of its output type (the erf polynomial for bf16, erff for fp32) and adds the residual in the same fp32
    order (FADD2 rounds as FADD does), and pair mode or another ring depth only moves tiles between CTAs.  So the output must be
    bit-identical to the default path, with one exception.  With GELU, an fp32 result and a residual, SURGVID_GEMM_TMA_OUT=0 moves the
    case from the TMA epilogue to epi_store (gemm_epi.cuh).  There `v = gelu_erf(v); v += res` is plain C++, and the compiler contracts
    GELU's final multiply 0.5x * (1 + erf) with the residual add into one FFMA.  The TMA epilogue adds the residual with add.rn.f32x2,
    which cannot be contracted.  The two results differ by at most one fp32 rounding of the product; that case is held to the gate."""
    ins, default, dplans = switch_default
    outs, plans, intact = run_in_child(ins, sw, tmp_path)
    for c, d, o, od, p, pd, ok in zip(SWITCH_CASES, ins, outs, default, plans, dplans, intact):
        what = f"{_id(c)} {sw}"
        if "SURGVID_GEMM_TMA_OUT" in sw:
            assert p["epilogue"] == "transpose" and p["tma_out"] == 0, (what, p)
        if "SURGVID_GEMM_EPI_BUFS" in sw:
            assert (p["epi_bufs"], p["epi_lag"]) == (int(sw["SURGVID_GEMM_EPI_BUFS"]), int(sw["SURGVID_GEMM_EPI_LAG"])), (what, p)
        if "SURGVID_GEMM_PREFETCH" in sw:
            assert p["prefetch"] == int(sw["SURGVID_GEMM_PREFETCH"]), (what, p)
        if "SURGVID_GEMM_PAIR" in sw:
            assert p["pair"] == int(sw["SURGVID_GEMM_PAIR"]), (what, p)
        assert ok, f"{what}: wrote outside its output block"
        ref, mag = _ref(d)
        G.assert_gate(o, ref.cpu(), mag.cpu(), d["act"], d["out_fp32"], what, p["block_n"])
        if "SURGVID_GEMM_TMA_OUT" in sw and d["out_fp32"] and d["residual"] is not None and d["act"] == G.ACT_GELU:
            continue   # the transposing epilogue fuses GELU's last multiply with the residual add (one FFMA, one rounding)
        assert torch.equal(o, od), f"{what}: differs from the default path ({pd})"


def test_switch_cases_reach_every_form():
    forms = {c[0] for c in SWITCH_CASES}
    assert forms == set(FORMS), forms


# ------------------------------------------------------------------------------------------------------- more than 2^31 output elements
@pytest.mark.parametrize("form", ["transpose", "f32_tma"])
def test_gemm_output_past_2_31_elements(form):
    """M = 2^23 + 1000, N = 256: the output has 2^31 + 256 000 elements; the transposing epilogue computes row * ldc in 64 bits, the TMA
    store takes 64-bit coordinates from the tensor map.  Checked in float64 on the first tile, the rows around element 2^31 and the last
    256 rows; the output starts NaN-filled, so rows that were never written fail."""
    M, N, K = 2 ** 23 + 1000, 256, 64
    out_fp32, res = FORMS[form]
    g = torch.Generator(device=DEV).manual_seed(5)
    a = torch.randn((M, K), generator=g, device=DEV).to(torch.bfloat16)
    w = (torch.randn((N, K), generator=g, device=DEV) / 8).to(torch.bfloat16)
    bias = torch.randn((N,), generator=g, device=DEV)
    r = torch.randn((M, N), generator=g, device=DEV) if res else None
    out = torch.full((M, N), float("nan"), dtype=torch.float32 if out_fp32 else torch.bfloat16, device=DEV)
    plan = ops.gemm_plan_info(M, N, K, 0, out_fp32, res)
    assert plan["epilogue"] == form, plan
    ops.gemm_bf16(a, w, bias=bias, residual=r, out=out)
    mid = 2 ** 31 // N
    for r0, r1 in ((0, 128), (mid - 256, mid + 256), (M - 256, M)):
        ref, mag = G.reference(a[r0:r1], w, bias, G.ACT_NONE, None if r is None else r[r0:r1])
        G.assert_gate(out[r0:r1], ref, mag, G.ACT_NONE, out_fp32, f"{form} rows {r0}:{r1}", plan["block_n"], row0=r0)
    del a, r, out
    torch.cuda.empty_cache()
