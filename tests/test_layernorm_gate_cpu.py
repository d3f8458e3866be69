"""The LayerNorm accuracy gate (tests/layernorm_ref.py) judged on the CPU: it accepts an fp32 emulation of the kernel's folded form on every
stress input and both output types, and rejects each known LayerNorm bug, injected into the same emulation, on the input it targets."""
import math

import pytest

import layernorm_ref as L

WIDTHS = [12, 64, 100, 320, 512]
MIN_REJECTION = 4.0


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("kind", L.STRESS)
@pytest.mark.parametrize("eps", [1e-5, 1e-6])
def test_gate_accepts_honest_emulation(kind, C, eps):
    d = L.make_inputs(kind, 300, C, seed=C)
    r = L.reference(d["x"], d["gamma"], d["beta"], eps)
    for fp32 in (True, False):
        e = L.gate_errors(L.emulate(d["x"], d["gamma"], d["beta"], eps, fp32), r, fp32, check_bias=kind not in ("const", "tiny"))
        assert e["ratio"] <= (0.5 if fp32 else 1.0), (fp32, e)


REJECTIONS = {}


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("bug", list(L.BUGS))
def test_gate_rejects_emulated_bug(bug, C):
    kind, fp32 = L.BUGS[bug]
    eps = 1e-5
    d = L.make_inputs(kind, 600, C, seed=C)
    r = L.reference(d["x"], d["gamma"], d["beta"], eps)
    e = L.gate_errors(L.emulate(d["x"], d["gamma"], d["beta"], eps, fp32, bug), r, fp32)
    REJECTIONS[bug] = min(REJECTIONS.get(bug, math.inf), e["ratio"])
    assert e["ratio"] >= MIN_REJECTION, (bug, C, e)


def test_rejection_factors(capsys):
    with capsys.disabled():
        print("\nLayerNorm gate rejection factor per emulated bug (smallest over the widths):")
        for bug, f in sorted(REJECTIONS.items(), key=lambda t: t[1]):
            print(f"  {bug:20s} {f:12.1f}x  ({L.BUGS[bug][0]})")
    assert REJECTIONS and min(REJECTIONS.values()) >= MIN_REJECTION
