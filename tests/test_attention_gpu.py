"""sv_op_attention on the GPU: every kernel behind the entry point against the float64 reference of tests/attn_ref.py, under the shared
gate, with stress inputs at the ragged key-tile edges; the A/B switches SURGVID_ATTN_TC=0 and SURGVID_ATTN_ORDER=1 in a fresh process;
and isolation: frames and heads do not bleed into each other, nothing outside the output block is written, runs repeat bit for bit.

Dispatch (launch_attention, attention.cu): the tcgen05 kernels take head_dim 64 with N_kv <= 448, leading dims % 8 == 0 and 16-byte
aligned pointers (one key tile: attention_tc_single_kernel, more: attention_tc_kernel<true>); otherwise the mma.sync kernels take
N_kv <= 64 (attention_resident_kv_kernel) or N_kv <= 256 (attention_resident_multi_kernel) when ldo % 8 == 0 and o is 16-byte aligned,
and attention_kernel takes everything else."""
import os
import subprocess
import sys

import pytest
import torch

import attn_ref as A
import surgvid_b200  # noqa: F401

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

TC1, TCM = "attention_tc_single_kernel", "attention_tc_kernel"
RES, RESM, GEN = "attention_resident_kv_kernel", "attention_resident_multi_kernel", "attention_kernel"

# (kernel, B, heads, Nq, Nkv, hd, o_offset): o_offset moves the output 2 elements off 16-byte alignment, which the tcgen05 and the
# resident kernels decline.  The first case of each kernel also runs the wide / uniform / large-V inputs.
CASES = [
    (TC1, 40, 1, 3136, 49, 64, 0), (TC1, 2, 5, 1, 1, 64, 0), (TC1, 3, 5, 127, 63, 64, 0), (TC1, 2, 1, 128, 64, 64, 0),
    (TC1, 2, 5, 129, 49, 64, 0), (TC1, 1, 5, 3136, 64, 64, 0),
    (TCM, 3, 2, 129, 65, 64, 0), (TCM, 2, 1, 127, 127, 64, 0), (TCM, 2, 5, 128, 128, 64, 0), (TCM, 1, 2, 1, 129, 64, 0),
    (TCM, 1, 1, 1000, 390, 64, 0), (TCM, 2, 8, 405, 405, 64, 0), (TCM, 2, 2, 257, 447, 64, 0), (TCM, 2, 2, 257, 448, 64, 0),
    (RES, 3, 8, 49, 1, 20, 0), (RES, 2, 5, 196, 64, 40, 0), (RES, 2, 2, 127, 63, 32, 0),
    (RESM, 2, 8, 196, 196, 40, 0), (RESM, 2, 2, 129, 65, 32, 0), (RESM, 1, 8, 300, 255, 20, 0), (RESM, 2, 5, 64, 256, 40, 0),
    (GEN, 1, 8, 300, 330, 20, 0), (GEN, 2, 2, 129, 257, 32, 0), (GEN, 1, 5, 65, 449, 40, 0), (GEN, 1, 2, 64, 449, 64, 0),
    (GEN, 1, 1, 100, 1000, 64, 0),
    (GEN, 2, 1, 130, 49, 20, 0), (GEN, 1, 1, 77, 196, 20, 0),          # hd 20, one head: ldo 20
    (GEN, 2, 2, 129, 49, 64, 2), (GEN, 1, 3, 200, 405, 64, 2),        # hd 64, o 4 bytes past 16-byte alignment
]
FIRST_OF_KERNEL = {c[0]: c for c in reversed(CASES)}


def _id(c):
    return f"{c[0].replace('attention_', '')}-{'x'.join(map(str, c[1:6]))}" + (f"-o+{c[6]}" if c[6] else "")


def _stress(c):
    kinds = ["randn"]
    if c[4] % A.KEY_TILE:
        kinds += ["neg", "plant_first"] + (["plant_last"] if c[4] > 1 else [])
    if FIRST_OF_KERNEL[c[0]] is c:
        kinds += ["wide", "uniform", "bigv"]
    return kinds


PARAMS = [pytest.param(c, kind, id=f"{_id(c)}-{kind}") for c in CASES for kind in _stress(c)]


def _case(c, kind="randn", seed=7):
    _, B, heads, Nq, Nkv, hd, off = c
    q, k, v = A.make_inputs(kind, B, heads, Nq, Nkv, hd, seed=seed, device=DEV)
    return {"q": q, "k": k, "v": v, "B": B, "heads": heads, "hd": hd, "scale": hd ** -0.5, "o_offset": off}


def _ref(d):
    return A.reference(d["q"], d["k"], d["v"], d["B"], d["heads"], d["hd"], d["scale"])


@pytest.mark.parametrize("c,kind", PARAMS)
def test_attention_matches_fp64_reference(c, kind):
    d = _case(c, kind)
    A.assert_gate(A.call(d), _ref(d), d["heads"], d["hd"], c[3], f"{_id(c)} {kind}")


def test_dispatch_table():
    """Every case of the table reaches the kernel it is annotated with."""
    _, kernels = A.run_cases([_case(c) for c in CASES])
    assert kernels == [c[0] for c in CASES]


# ----------------------------------------------------------------------------------------------- forced A/B paths (fresh process)
def _mma_kernel(Nkv):
    return RES if Nkv <= 64 else (RESM if Nkv <= 256 else GEN)


def _run_in_child(cases, env_overrides, tmp_path):
    torch.save([{k: (v.cpu() if torch.is_tensor(v) else v) for k, v in d.items()} for d in cases], tmp_path / "in.pt")
    env = dict(os.environ, **env_overrides)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [A.__file__, str(tmp_path / "in.pt"), str(tmp_path / "out.pt")]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-4000:]
    res = torch.load(tmp_path / "out.pt")
    return res["outs"], res["kernels"]


def test_tc_disabled_runs_mma_kernels_for_head_dim_64(tmp_path):
    """SURGVID_ATTN_TC=0 (the A/B switch of the tcgen05 kernels): the hd-64 shapes run on the mma.sync kernels, which must pass the gate
    against the fp64 reference and agree with the default (tcgen05) output within the gate."""
    runs = [(c, kind) for c in CASES if c[0] in (TC1, TCM) for kind in ["randn", "plant_last"] + (["neg"] if c[4] % A.KEY_TILE else [])]
    ins = [_case(c, kind) for c, kind in runs]
    forced, kernels = _run_in_child(ins, {"SURGVID_ATTN_TC": "0"}, tmp_path)
    assert kernels == [_mma_kernel(c[4]) for c, _ in runs]
    default, kernels = A.run_cases(ins)
    assert kernels == [c[0] for c, _ in runs]
    for (c, kind), d, f, o in zip(runs, ins, forced, default):
        A.assert_gate(f, _ref(d).cpu(), c[2], c[5], c[3], f"{_id(c)} {kind} SURGVID_ATTN_TC=0")
        A.assert_gate(f, o, c[2], c[5], c[3], f"{_id(c)} {kind} SURGVID_ATTN_TC=0 vs default")


def test_round_robin_order_of_single_tile_tc_kernel(tmp_path):
    """SURGVID_ATTN_ORDER=1: the persistent single-key-tile kernel deals (frame, head, query tile) items round-robin with the head
    fastest.  Only which CTA computes a tile changes, so the output is bit-identical to the default order (and passes the gate)."""
    cases = [c for c in CASES if c[0] == TC1 and c[2] > 1] + [(TC1, 7, 8, 196, 49, 64, 0)]
    ins = [_case(c, "plant_last" if c[4] > 1 else "randn") for c in cases]
    forced, kernels = _run_in_child(ins, {"SURGVID_ATTN_ORDER": "1"}, tmp_path)
    assert kernels == [TC1] * len(cases)
    default, _ = A.run_cases(ins)
    for c, d, f, o in zip(cases, ins, forced, default):
        A.assert_gate(f, _ref(d).cpu(), c[2], c[5], c[3], f"{_id(c)} SURGVID_ATTN_ORDER=1")
        assert torch.equal(f, o), _id(c)


# ----------------------------------------------------------------------------------------------- isolation
ISO = [(TC1, 3, 5, 127, 63, 64, 0), (TCM, 2, 8, 405, 405, 64, 0), (RES, 2, 2, 127, 63, 32, 0), (RESM, 2, 8, 196, 196, 40, 0),
       (GEN, 2, 2, 129, 257, 32, 0), (GEN, 2, 1, 130, 49, 20, 0), (GEN, 2, 2, 129, 49, 64, 2)]


@pytest.mark.parametrize("c", ISO, ids=_id)
def test_frames_and_heads_do_not_bleed(c):
    """New Q, K or V values in one frame (one head) leave every other frame (head) bit-identical, and do change their own."""
    d = _case(c)
    _, B, heads, Nq, Nkv, hd, _ = c
    base = A.call(d).clone()
    g = torch.Generator(device=DEV).manual_seed(99)
    b, h = B - 1, heads // 2
    for name in ("q", "k", "v"):
        n = Nq if name == "q" else Nkv
        for what, rows, cols, o_rows, o_cols in (("frame", slice(b * n, (b + 1) * n), slice(None), slice(b * Nq, (b + 1) * Nq), slice(None)),
                                                 ("head", slice(None), slice(h * hd, (h + 1) * hd), slice(None), slice(h * hd, (h + 1) * hd))):
            if what == "head" and heads == 1:
                continue
            e = dict(d)
            e[name] = d[name].clone()
            e[name][rows, cols] = torch.randn(e[name][rows, cols].shape, generator=g, device=DEV).to(torch.bfloat16)
            out = A.call(e)
            keep = torch.ones_like(out, dtype=torch.bool)
            keep[o_rows, o_cols] = False
            assert torch.equal(out[keep], base[keep]), f"{_id(c)}: new {name} in {what} {b if what == 'frame' else h} changed other outputs"
            assert not torch.equal(out[~keep], base[~keep]), f"{_id(c)}: new {name} in {what} left its own output unchanged"


@pytest.mark.parametrize("c", ISO, ids=_id)
def test_strided_output_writes_only_its_block_and_repeats_bit_for_bit(c):
    """Output into a NaN-filled buffer with ldo = heads*hd + 24 and guard rows before and after: every element outside the
    [B*Nq, heads*hd] block keeps its bits, the block equals the contiguous output, and a second run gives the same bits."""
    d = _case(c, "neg" if c[4] % A.KEY_TILE else "randn")
    _, B, heads, Nq, Nkv, hd, off = c
    C, rows, guard = heads * hd, B * Nq, 3
    ldo = C + 24
    buf = torch.full(((rows + 2 * guard) * ldo,), float("nan"), dtype=torch.bfloat16, device=DEV)
    fill = buf.view(torch.int16).clone()
    o = buf[guard * ldo + off:].as_strided((rows, C), (ldo, 1))
    contiguous = A.call(d)
    kernels = []
    A.call(d, out=o, kernels=kernels)
    assert kernels == [c[0]]
    inside = torch.zeros_like(buf, dtype=torch.bool)
    inside[guard * ldo + off:].as_strided((rows, C), (ldo, 1)).fill_(True)
    bits = buf.view(torch.int16)
    assert torch.equal(bits[~inside], fill[~inside]), f"{_id(c)}: wrote outside its output block"
    assert torch.equal(o, contiguous), _id(c)
    A.assert_gate(o, _ref(d), heads, hd, Nq, _id(c))
    again = o.clone()
    A.call(d, out=o)
    assert torch.equal(o, again), f"{_id(c)}: second run differs"
