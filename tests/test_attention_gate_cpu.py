"""The attention accuracy gate (tests/attn_ref.py) judged on the CPU: it accepts the kernels' honest arithmetic (tiled online softmax,
bf16 probabilities and output) on every stress input, and rejects each known kernel bug, injected into the same emulation, on every
shape where the bug changes the output at all.  Where a bug cannot change the output (e.g. unmasked padding keys when N_kv is a
multiple of the key tile) the emulation must come out bit-identical to the honest one, so the shape list cannot hide a blind spot."""
import pytest
import torch

import attn_ref as A

# (B, heads, Nq, Nkv, hd, query rows per tile): the tcgen05 kernels take 128 query rows per tile, the mma.sync kernels 64.  One key
# tile / several, exact and ragged tile edges, one frame / one head, the head dims of the model.
SHAPES = [
    (2, 2, 129, 1, 64, 128), (2, 5, 127, 49, 64, 128), (1, 1, 128, 64, 64, 128), (2, 2, 129, 65, 64, 128), (1, 2, 200, 405, 64, 128),
    (2, 1, 130, 448, 64, 128), (2, 3, 100, 196, 40, 64), (2, 1, 70, 449, 20, 64), (3, 2, 65, 1000, 32, 64), (2, 8, 64, 256, 40, 64),
]


def _run(kind, shape, bug=None, seed=1):
    B, H, Nq, Nkv, hd, qt = shape
    q, k, v = A.make_inputs(kind, B, H, Nq, Nkv, hd, seed=seed)
    ref = A.reference(q, k, v, B, H, hd, hd ** -0.5)
    return A.emulate(q, k, v, B, H, hd, hd ** -0.5, qt, bug), ref


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("kind", A.STRESS)
def test_gate_accepts_honest_emulation(kind, shape):
    out, ref = _run(kind, shape)
    e = A.gate_errors(out, ref, shape[1], shape[4])
    # the limits leave at least 1.5x room over the honest arithmetic
    assert A.gate_ratio(e) <= 1 / 1.5, e


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("bug", list(A.BUGS))
def test_gate_rejects_emulated_bug(bug, shape):
    kind, changes = A.BUGS[bug]
    out, ref = _run(kind, shape, bug)
    if changes(*shape[:4], shape[5]):
        e = A.gate_errors(out, ref, shape[1], shape[4])
        assert not A.passes_gate(e), (bug, kind, e)
    else:
        honest, _ = _run(kind, shape)
        assert torch.equal(out, honest), f"{bug} changes the output at {shape}, where it was expected not to"


@pytest.mark.parametrize("bug", list(A.BUGS))
def test_every_bug_is_exercised(bug):
    _, changes = A.BUGS[bug]
    assert sum(bool(changes(*s[:4], s[5])) for s in SHAPES) >= 3


def test_reference_layout_matches_a_per_frame_per_head_loop():
    B, H, Nq, Nkv, hd = 2, 3, 5, 7, 8
    q, k, v = A.make_inputs("randn", B, H, Nq, Nkv, hd, seed=3)
    ref = A.reference(q, k, v, B, H, hd, 0.3)
    for b in range(B):
        for h in range(H):
            cols = slice(h * hd, (h + 1) * hd)
            qs, ks, vs = (t[b * n:(b + 1) * n, cols].double() for t, n in ((q, Nq), (k, Nkv), (v, Nkv)))
            want = torch.softmax(qs @ ks.T * 0.3, -1) @ vs
            torch.testing.assert_close(ref[b * Nq:(b + 1) * Nq, cols], want, rtol=1e-12, atol=1e-12)


def test_gate_checks_each_head_and_non_finite_values():
    B, H, Nq, Nkv, hd = 1, 8, 64, 49, 32
    q, k, v = A.make_inputs("randn", B, H, Nq, Nkv, hd, seed=4)
    ref = A.reference(q, k, v, B, H, hd, hd ** -0.5)
    out = ref.clone()
    out[:, 2 * hd:3 * hd] *= 1.006          # one head 0.6 % off: within the gate over all 8 heads, not within head 2's block
    e = A.gate_errors(out, ref, H, hd)
    assert e["rel_l2_block"] == "head 2" and not A.passes_gate(e)
    assert A.passes_gate(A.gate_errors(out[:, :2 * hd], ref[:, :2 * hd], 2, hd))
    out = ref.clone()
    out[7, 5] = float("nan")
    assert not A.passes_gate(A.gate_errors(out, ref, H, hd))


def test_sv_op_attention_rejects_misaligned_output():
    """The kernels store the output as bf16 pairs: an output pointer that is not 4-byte aligned is refused before any launch."""
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import _native

    lib = _native.lib()
    base = 1 << 20   # never dereferenced: the argument checks fail first
    rc = lib.sv_op_attention(base, 64, base + 4096, 64, base + 8192, 64, base + 16384 + 2, 64, 1, 1, 64, 64, 64, 0.125, None)
    assert rc != _native.SV_OK
    assert b"4-byte aligned" in lib.sv_last_error()


@pytest.mark.parametrize("hd,Nkv,ldo,o_off,want", [
    (64, 1, 320, 0, "attention_tc_single_kernel"), (64, 64, 320, 0, "attention_tc_single_kernel"), (64, 65, 320, 0, "attention_tc_kernel"),
    (64, 448, 64, 0, "attention_tc_kernel"), (64, 449, 64, 0, "attention_kernel"), (64, 49, 128, 4, "attention_kernel"),
    (64, 49, 132, 0, "attention_kernel"), (32, 64, 64, 0, "attention_resident_kv_kernel"), (40, 65, 200, 0, "attention_resident_multi_kernel"),
    (20, 256, 160, 0, "attention_resident_multi_kernel"), (20, 257, 160, 0, "attention_kernel"), (20, 49, 20, 0, "attention_kernel"),
    (40, 196, 200, 8, "attention_kernel"),
])
def test_dispatch_query(hd, Nkv, ldo, o_off, want):
    """sv_op_attention_kernel (the decision sv_op_attention launches by) on the host: no device memory is touched."""
    import surgvid_b200  # noqa: F401
    from surgvid_b200 import _native

    base = 1 << 20
    ld = 8 * 64
    i = _native.lib().sv_op_attention_kernel(base, ld, base + 4096, ld, base + 8192, ld, base + 16384 + o_off, ldo, Nkv, hd)
    assert A.KERNELS[i] == want
