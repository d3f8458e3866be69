"""LayerNorm on the GPU (`sv_op_layernorm`, `sv_op_layernorm_nchw`) against the float64 reference of tests/layernorm_ref.py under its gate:
every row of ln_dispatch (exact and predicated lane mappings), both eps values, 1 row, a warp's rows minus one, a ragged last block and
a large count; fp32 only, bf16 only and both outputs; bf16 == the fp32 result rounded to nearest even; the channel-major form bit-identical
to the token-major one; stress rows (constant, |mean| / std = 1e3, variance near eps, |x| of 1e4 and 1e-20); more than 2^31 elements."""
import pytest
import torch

import layernorm_ref as L
import surgvid_b200  # noqa: F401
from surgvid_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# C -> rows per warp (32 / lanes per row) of ln_dispatch's mapping for it
WIDTHS = {4: 8, 8: 8, 12: 8, 16: 16, 20: 4, 24: 4, 36: 2, 40: 16, 60: 2, 68: 1, 80: 8, 100: 1, 124: 1, 128: 8, 132: 1, 160: 4, 252: 1,
          256: 4, 260: 1, 320: 2, 384: 1, 388: 1, 500: 1, 508: 1, 512: 1}
SEEN = {}


def _rows_list(C):
    rpw = WIDTHS[C]
    return sorted({1, max(1, rpw - 1), 8 * rpw * 3 + 5, 40_000})


def _run(kind, rows, C, eps, seed=0):
    d = L.make_inputs(kind, rows, C, seed=seed, device=DEV)
    of, ob = ops.layernorm(d["x"], d["gamma"], d["beta"], eps, want_f32=True, want_bf16=True)
    torch.cuda.synchronize()
    return d, of, ob


@pytest.mark.parametrize("eps", [1e-5, 1e-6])
@pytest.mark.parametrize("C", list(WIDTHS))
def test_layernorm_every_lane_mapping(C, eps):
    """Gate on fp32 and bf16 outputs; bf16 bit-identical to the fp32 result rounded to nearest even."""
    for rows in _rows_list(C):
        d, of, ob = _run("randn", rows, C, eps, seed=C + rows)
        r = L.reference(d["x"], d["gamma"], d["beta"], eps)
        e = L.assert_gate(of, r, True, f"C {C} rows {rows} eps {eps} fp32")
        SEEN["fp32"] = max(SEEN.get("fp32", 0.0), e["ratio"])
        L.assert_gate(ob, r, False, f"C {C} rows {rows} eps {eps} bf16", check_bias=rows * C >= 20_000)
        assert torch.equal(ob.view(torch.int16), of.to(torch.bfloat16).view(torch.int16)), f"C {C} rows {rows}: bf16 is not RNE(fp32)"


@pytest.mark.parametrize("C", [12, 64, 100, 320, 512])
def test_layernorm_output_combinations(C):
    """fp32 only and bf16 only give the same bits as both together."""
    d, of, ob = _run("randn", 1237, C, 1e-6, seed=1)
    f_only, none = ops.layernorm(d["x"], d["gamma"], d["beta"], 1e-6, want_f32=True, want_bf16=False)
    none2, b_only = ops.layernorm(d["x"], d["gamma"], d["beta"], 1e-6, want_f32=False, want_bf16=True)
    assert none is None and none2 is None
    assert torch.equal(f_only, of) and torch.equal(b_only.view(torch.int16), ob.view(torch.int16))


@pytest.mark.parametrize("kind", L.STRESS[1:])
@pytest.mark.parametrize("C", [12, 64, 100, 320, 512])
def test_layernorm_stress(kind, C):
    for eps in (1e-5, 1e-6):
        d, of, ob = _run(kind, 3000, C, eps, seed=C)
        r = L.reference(d["x"], d["gamma"], d["beta"], eps)
        e = L.assert_gate(of, r, True, f"{kind} C {C} eps {eps} fp32")
        SEEN[kind] = max(SEEN.get(kind, 0.0), e["ratio"])
        L.assert_gate(ob, r, False, f"{kind} C {C} eps {eps} bf16", check_bias=kind not in ("const", "tiny"))
        assert torch.equal(ob.view(torch.int16), of.to(torch.bfloat16).view(torch.int16))


@pytest.mark.parametrize("tokens,frames", [(1, 37), (49, 5), (3136, 2), (333, 7)])
def test_layernorm_nchw_bit_identical_to_token_major(tokens, frames):
    """The channel-major form writes exactly the token-major fp32 values, permuted, at every width; its bf16 copy is the same too.
    333 tokens per frame: CTA row blocks straddle frames."""
    for C in WIDTHS:
        d = L.make_inputs("randn", tokens * frames, C, seed=C, device=DEV)
        of, ob = ops.layernorm(d["x"], d["gamma"], d["beta"], 1e-6, want_f32=True, want_bf16=True)
        nchw, ob2 = ops.layernorm_nchw(d["x"], d["gamma"], d["beta"], 1e-6, tokens, want_bf16=True)
        want = of.view(frames, tokens, C).permute(0, 2, 1)
        assert torch.equal(nchw.view(frames, C, tokens), want), f"C {C} tokens {tokens}"
        assert torch.equal(ob2.view(torch.int16), ob.view(torch.int16)), f"C {C} tokens {tokens}: bf16"


def test_layernorm_past_2_31_elements():
    """rows * C > 2^31 token-major (C = 512): checked in float64 on the first rows, the rows around element 2^31 and the last rows."""
    C = 512
    rows = (1 << 31) // C + 3000
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn((rows, C), generator=g, device=DEV)
    gamma = 1 + 0.2 * torch.randn((C,), generator=g, device=DEV)
    beta = 0.3 * torch.randn((C,), generator=g, device=DEV)
    of = ops.layernorm(x, gamma, beta, 1e-6, want_f32=True, want_bf16=False)[0]
    mid = (1 << 31) // C
    for r0, r1 in ((0, 64), (mid - 64, mid + 64), (rows - 64, rows)):
        r = L.reference(x[r0:r1], gamma, beta, 1e-6)
        L.assert_gate(of[r0:r1], r, True, f"rows {r0}:{r1}")
    del x, of
    torch.cuda.empty_cache()


def test_report_gate_terms(capsys):
    with capsys.disabled():
        print(f"\nLayerNorm worst |err|/bound over this run ({torch.cuda.get_device_name(0)}): " + ", ".join(f"{k} {v:.3f}" for k, v in SEEN.items()))
