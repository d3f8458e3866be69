"""The GEMM accuracy gate (tests/gemm_ref.py) judged on the CPU: it accepts the kernel's honest arithmetic on every stress input and rejects
each known GEMM bug, injected into the same emulation, by at least 5x on the input it targets.  Where a bug cannot change the output for a
shape, the emulation must come out bit-identical to the honest one, so the shape list hides no blind spot.  Also without a device: the
GPU case table reaches the whole plan space by `sv_op_gemm_plan_info` at 148 SMs, and argument errors come back as SV_ERR_INVALID."""
import ctypes

import pytest
import torch

import gemm_ref as G

# (M, N, K, K2): K in {8, 72, 200, 1360, 8192}; second A segments; ragged and exact M tiles; one and several N tiles
SHAPES = [(300, 200, 8, 0), (300, 520, 72, 8), (256, 200, 200, 0), (300, 136, 200, 8), (200, 520, 1360, 80), (384, 200, 1360, 0),
          (130, 96, 8192, 0)]
MIN_REJECTION = 5.0


def _block_n(shape, out_fp32):
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import ops

    M, N, K, K2 = shape
    return ops.gemm_plan_info(M, N, K, K2, out_fp32, True, -1, num_sms=148)["block_n"]


def _run(kind, shape, act, out_fp32, bug=None, seed=1):
    M, N, K, K2 = shape
    d = G.make_inputs(kind, M, N, K, K2, seed=seed)
    ref, mag = G.reference(d["a"], d["w"], d["bias"], act, d["residual"], d["a2"])
    out = G.emulate(d["a"], d["w"], d["bias"], act, d["residual"], out_fp32, d["a2"], _block_n(shape, out_fp32), bug)
    return out, ref, mag


def _sid(s):
    return "x".join(map(str, s[:3])) + (f"+{s[3]}" if s[3] else "")


@pytest.mark.parametrize("shape", SHAPES, ids=_sid)
@pytest.mark.parametrize("kind", G.STRESS)
@pytest.mark.parametrize("out_fp32", [True, False], ids=["f32", "bf16"])
def test_gate_accepts_honest_emulation(kind, shape, out_fp32):
    """fp32 outputs stay within 1/2 of the gate.  A bf16 output's elementwise error is dominated by its final rounding, which reaches its
    own bound (2^-8 |y|) by construction, so there it must stay within the gate, and its rounding bias within 1/2 of the bias gate."""
    for act in (G.ACT_NONE, G.ACT_GELU, G.ACT_RELU):
        out, ref, mag = _run(kind, shape, act, out_fp32)
        e = G.gate_errors(out, ref, mag, act, out_fp32, check_bias=kind != "rowid")
        assert e["ratio"] <= (0.5 if out_fp32 else 1.0), (act, G.describe(e))
        assert e["bias_ratio"] <= 0.5, (act, G.describe(e))
        if not out_fp32 and shape[0] * shape[1] >= 4 * G.BIAS_MIN_ELEMS and shape[2] <= 1360 and kind not in ("cancel", "rowid"):
            assert e["bias_ulp"] is not None, "the rounding-bias check found too few eligible elements"


REJECTIONS = {}


@pytest.mark.parametrize("shape", SHAPES, ids=_sid)
@pytest.mark.parametrize("bug", list(G.BUGS))
def test_gate_rejects_emulated_bug(bug, shape):
    kind, out_fp32, act, changes = G.BUGS[bug]
    out, ref, mag = _run(kind, shape, act, out_fp32, bug)
    if changes(*shape, _block_n(shape, out_fp32)):
        e = G.gate_errors(out, ref, mag, act, out_fp32, _block_n(shape, out_fp32))
        factor = G.gate_ratio(e)
        REJECTIONS[bug] = min(REJECTIONS.get(bug, float("inf")), factor)
        assert factor >= MIN_REJECTION, (bug, kind, G.describe(e))
    else:
        honest, _, _ = _run(kind, shape, act, out_fp32)
        assert torch.equal(out, honest), f"{bug} changes the output at {shape}, where it was expected not to"


@pytest.mark.parametrize("bug", list(G.BUGS))
def test_every_bug_is_exercised(bug):
    kind, out_fp32, _, changes = G.BUGS[bug]
    assert sum(bool(changes(*s, _block_n(s, out_fp32))) for s in SHAPES) >= 2


def test_rejection_factors(capsys):
    """Smallest factor by which the gate rejects each bug over the shapes (printed; the per-shape tests assert >= 5)."""
    for bug, (kind, out_fp32, act, changes) in G.BUGS.items():
        if bug not in REJECTIONS:
            for s in SHAPES:
                if changes(*s, _block_n(s, out_fp32)):
                    out, ref, mag = _run(kind, s, act, out_fp32, bug)
                    REJECTIONS[bug] = min(REJECTIONS.get(bug, float("inf")), G.gate_ratio(G.gate_errors(out, ref, mag, act, out_fp32)))
    with capsys.disabled():
        print("\nGEMM gate rejection factor per emulated bug (smallest over the shapes):")
        for bug, f in sorted(REJECTIONS.items(), key=lambda t: t[1]):
            print(f"  {bug:28s} {f:10.1f}x  ({G.BUGS[bug][0]}, {'fp32' if G.BUGS[bug][1] else 'bf16'} output)")
    assert min(REJECTIONS.values()) >= MIN_REJECTION


def test_reference_and_emulation_layout():
    """The reference is act(A W^T + b) + r element by element; the two-segment A is [a | a2]; the honest emulation equals it to fp32."""
    d = G.make_inputs("randn", 5, 16, 72, 8, seed=3)
    ref, mag = G.reference(d["a"], d["w"], d["bias"], G.ACT_GELU, d["residual"], d["a2"])
    A = torch.cat([d["a"], d["a2"]], 1).double()
    for i, j in ((0, 0), (4, 15), (2, 7)):
        y = float(A[i] @ d["w"][j].double()) + float(d["bias"][j])
        want = 0.5 * y * (1 + torch.erf(torch.tensor(y, dtype=torch.float64) / 2 ** 0.5)) + float(d["residual"][i, j])
        assert abs(float(ref[i, j]) - float(want)) < 1e-12
        assert abs(float(mag[i, j]) - float(A[i].abs() @ d["w"][j].double().abs() + abs(float(d["bias"][j])))) < 1e-12
    out = G.emulate(d["a"], d["w"], d["bias"], G.ACT_GELU, d["residual"], True, d["a2"])
    torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5)


def test_gate_reports_worst_element_and_rejects_non_finite():
    d = G.make_inputs("randn", 300, 96, 64, seed=4)
    ref, mag = G.reference(d["a"], d["w"], d["bias"], G.ACT_NONE, d["residual"])
    out = ref.clone()
    out[200, 70] += 1e-3
    e = G.gate_errors(out, ref, mag, G.ACT_NONE, True, block_n=32)
    assert (e["row"], e["col"]) == (200, 70) and not G.passes_gate(e)
    assert "M tile 1, N tile 2" in G.describe(e)
    out = ref.clone()
    out[7, 5] = float("nan")
    assert not G.passes_gate(G.gate_errors(out, ref, mag, G.ACT_NONE, True))


def test_gelu_polynomial_matches_stated_error():
    """The emulated erf polynomial of bf16 GELU outputs is within the 6.1e-5 that common.cuh states (and so within GELU_POLY_ABS)."""
    x = torch.linspace(-12, 12, 200001)
    exact = G._act64(x.double(), G.ACT_GELU)
    assert float((G.gelu_poly_f32(x).double() - exact).abs().max()) <= 6.2e-5 < G.GELU_POLY_ABS


# ------------------------------------------------------------------------------------------------------- plan space of the GPU table
def _table_plans():
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import ops
    import test_gemm_gpu as T

    out = []
    for c in T.CASES:
        f32, res = T.FORMS[c[0]]
        out.append((c, ops.gemm_plan_info(c[1], c[2], c[3], c[4], f32, res, c[5], num_sms=148)))
    return out


def test_case_table_annotations_match_plan_query():
    import test_gemm_gpu as T

    for c, p in _table_plans():
        T.check_plan(c, p, 148)


def test_case_table_reaches_plan_space():
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import ops
    import test_gemm_gpu as T

    plans = _table_plans()
    f32_widths = {p["block_n"] for c, p in plans if T.FORMS[c[0]][0]}
    assert f32_widths == set(range(16, 257, 16)), sorted(f32_widths)
    bf16_tma_widths = {p["block_n"] for c, p in plans if c[0] == "bf16_tma"}
    assert bf16_tma_widths == set(range(32, 257, 32)), sorted(bf16_tma_widths)
    # every ring depth the planner can produce (default switches): all block_n x pair x epilogue form
    possible = set()
    for form, (f32, res) in T.FORMS.items():
        for N in range(16, 257, 16):
            for pair in (0, 1):
                possible.add(ops.gemm_plan_info(20000, N, 8, 0, f32, res, pair, num_sms=148)["num_stages"])
    assert {p["num_stages"] for _, p in plans} == possible, (sorted(possible), sorted({p["num_stages"] for _, p in plans}))
    for form in T.FORMS:
        assert {p["pair"] for c, p in plans if c[0] == form} == {0, 1}, form
    assert {c[3] % 64 for c, _ in plans} >= {0, 8, 16, 56} and any(c[3] < 64 for c, _ in plans)
    assert any(c[1] % 128 for c, _ in plans)
    assert any(p["pair"] and 0 < c[1] % 256 <= 128 for c, p in plans)                              # the pair's second CTA gets no rows
    assert any(c[0] == "f32_tma_resid" and c[2] % p["block_n"] == 16 for c, p in plans)             # zero-chunk tile of the residual ring
    assert any(c[0] == "f32_tma_resid" and p["pair"] and c[2] % p["block_n"] == 16 for c, p in plans)
    assert any(p["num_tiles"] >= 3 * (p["grid"] // (2 if p["pair"] else 1)) for _, p in plans)   # several tiles per CTA
    assert any(c[4] for c, _ in plans)


def test_plan_query_is_host_only_and_checks_shapes():
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import _native

    lib = _native.lib()
    info = (ctypes.c_int32 * 13)()
    assert lib.sv_op_gemm_plan_info(1000, 320, 200, 0, 0, 1, -1, 148, info) == _native.SV_OK
    assert info[9] == 3 and info[10] == 2     # transposing epilogue, gemm_bf16_tcgen05_kernel<act, false, true, false>
    for args in ((1000, 12, 64, 0), (1000, 16, 60, 0), (1000, 16, 200, 16), (0, 16, 64, 0), (10, 16, 64, 64)):
        assert lib.sv_op_gemm_plan_info(*args, 0, 0, -1, 148, info) == 1, args
    assert lib.sv_op_gemm_plan_info(10, 16, 64, 0, 0, 0, -1, 0, info) == 1


# ------------------------------------------------------------------------------------------------------- argument errors, no device
BASE = 1 << 20   # dummy device addresses: the argument checks fail before anything is read through them


def _gemm_args(**kw):
    a = dict(A=BASE, lda=64, W=BASE + 65536, ldw=64, M=100, N=32, K=64, bias=0, act=0, residual=0, ldr=0, out=BASE + 2 * 65536, ldc=32,
             out_fp32=0, stream=None)
    a.update(kw)
    return a


ARG_ERRORS = [
    ("K % 8", dict(K=60, lda=64, ldw=64), "K%8==0"),
    ("N % 8", dict(N=20, ldc=24), "N%8==0"),
    ("lda < K", dict(lda=56), "leading dimensions"),
    ("ldc < N", dict(ldc=24), "leading dimensions"),
    ("out misaligned", dict(out=BASE + 2 * 65536 + 8), "16B-aligned"),
    ("ldc % 8 (bf16)", dict(ldc=36), "16B-aligned"),
    ("residual misaligned", dict(residual=BASE + 3 * 65536 + 4, ldr=32), "residual alignment"),
    ("ldr < N", dict(residual=BASE + 3 * 65536, ldr=28), "residual alignment"),
    ("bias misaligned", dict(bias=BASE + 4 * 65536 + 4), "bias alignment"),
]


@pytest.mark.parametrize("what,kw,msg", ARG_ERRORS, ids=[e[0] for e in ARG_ERRORS])
def test_gemm_argument_errors(what, kw, msg):
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import _native

    lib = _native.lib()
    a = _gemm_args(**kw)
    rc = lib.sv_op_gemm_bf16(a["A"], a["lda"], a["W"], a["ldw"], a["M"], a["N"], a["K"], a["bias"] or None, a["act"], a["residual"] or None,
                             a["ldr"], a["out"], a["ldc"], a["out_fp32"], None)
    assert rc == 1, what
    assert msg.encode() in lib.sv_last_error(), lib.sv_last_error()


@pytest.mark.parametrize("K,K2,lda2", [(200, 16, 16), (200, 12, 16), (136, 16, 16), (136, 136, 136), (136, 8, 0)])
def test_gemm_cat_segment_rules(K, K2, lda2):
    """K - K2 must be a multiple of 64, K2 % 8 == 0, K2 < K and lda2 >= K2."""
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import _native

    lib = _native.lib()
    rc = lib.sv_op_gemm_bf16_cat(BASE, 128, BASE + 65536, lda2, K2, BASE + 2 * 65536, 256, 100, 32, K, None, 0, None, 0, BASE + 3 * 65536, 32,
                                 0, None)
    assert rc == 1 and b"second A segment" in lib.sv_last_error(), lib.sv_last_error()
