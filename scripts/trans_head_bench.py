"""Trans-SVNet head at d_k 32 and 64 over the 80 Cholec80-shaped sequences (`synthetic.cholec80_video_lengths()`, 184 578 frames).

    python scripts/trans_head_bench.py [--reps 20] [--rounds 5] [--steps 500] [--out results/trans_head_bench.json]

The head's width follows mstcn_f_maps (d_k = d_v = min(64, f_maps), d_ff = f_maps), so each d_k is paired with its MS-TCN width: d_k 32
with f_maps 32, d_k 64 with f_maps 64.  Per width, with CUDA events around `reps` back-to-back warmed calls, the arms alternating over
`rounds` rounds (the median round is reported, with the min and max):
  * MS-TCN alone (`forward_videos`), MS-TCN + head (`Transformer.forward_videos`), and the head kernel alone (`forward_fused` on the
    MS-TCN logits and query, one `trans_head_kernel` launch);
  * FLOP per frame of the head, counted from the shapes below (a multiply-add is 2 FLOP), and the head kernel's FLOP/s from it.
Stream steps (`Transformer.open_stream` + `step`, MS-TCN and head) at 80 streams x 1 frame and 8 streams x 25 frames, from 100 frames
of history.  The device name, power limit and max SM clock are read in the same run.  Needs a CUDA device; there is no CPU path."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import surgvid_b200  # noqa: E402,F401
from surgvid_b200 import synthetic as S  # noqa: E402
from surgvid_b200.mstcn import MultiStageModel_S  # noqa: E402
from surgvid_b200.trans_head import Transformer  # noqa: E402

D, L, H = 14, 30, 4   # d_model (phases), len_q, heads


def head_flop_per_frame(d_k, d_ff, d_model=D, len_q=L, n_heads=H):
    """FLOP of one frame of Transformer2_3_1 (one encoder layer over the len_q window, one decoder step), multiply-add = 2."""
    hd = n_heads * d_k
    enc = (3 * len_q * d_model * hd            # Q, K, V projections of the window
           + 2 * n_heads * len_q * len_q * d_k  # scores and context
           + len_q * hd * d_model              # output projection
           + len_q * 2 * d_model * d_ff)       # FFN
    dec = (2 * len_q * d_model * hd            # K, V projections of the encoder output
           + d_model * hd                      # Q projection of the query
           + 2 * n_heads * len_q * d_k          # scores and context of the single query
           + hd * d_model                      # output projection
           + 2 * d_model * d_ff)               # FFN
    return 2 * (enc + dec)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "not available"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q}


def timed(fn, reps, e0, e1):
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def models(f_maps, dev):
    m = MultiStageModel_S(2, 8, f_maps, 2048, D, True)
    m.load_state_dict(S.synth_mstcn_state_dict(2, 8, f_maps, 2048, D, seed=1, mode="phase"))
    head = Transformer(f_maps, 2048, D, L)
    g = torch.Generator().manual_seed(21)
    with torch.no_grad():
        for p in head.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.05 if p.dim() == 2 and p.shape[1] == 2048 else 0.2))
    return m.to(dev).eval(), head.to(dev).eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("trans_head_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    print(json.dumps(info))
    lengths = [int(x) for x in S.cholec80_video_lengths()]
    T = sum(lengths)
    feats = torch.rand(T, 2048, device=dev, generator=torch.Generator(dev).manual_seed(80)) * 0.57
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    widths = {}
    for f_maps in (32, 64):
        m, head = models(f_maps, dev)
        head.attach(m)
        logits, query = m.forward_videos_query(feats, lengths)
        widths[f_maps] = {
            "mstcn_ms": lambda m=m: m.forward_videos(feats, lengths),
            "mstcn_plus_head_ms": lambda m=m, head=head: head.forward_videos(m, feats, lengths),
            "head_kernel_ms": lambda head=head, lg=logits[-1], q=query: head.transformer.forward_fused(lg, q, lengths),
        }
    arms = [(f, k) for f in widths for k in widths[f]]
    for f, k in arms:   # warm every shape
        for _ in range(3):
            widths[f][k]()
    torch.cuda.synchronize()
    samples = {arm: [] for arm in arms}
    for _ in range(a.rounds):
        for f, k in arms:
            samples[(f, k)].append(timed(widths[f][k], a.reps, e0, e1))

    rows = []
    for f_maps in (32, 64):
        d_k = min(64, f_maps)
        flop = head_flop_per_frame(d_k, f_maps)
        r = {"d_k": d_k, "d_ff": f_maps, "mstcn_f_maps": f_maps, "frames": T, "videos": len(lengths), "head_flop_per_frame": flop}
        for k in widths[f_maps]:
            s = samples[(f_maps, k)]
            r[k] = round(statistics.median(s), 4)
            r[k + "_min_max"] = [round(min(s), 4), round(max(s), 4)]
        r["head_kernel_tflops"] = round(flop * T / (r["head_kernel_ms"] * 1e-3) / 1e12, 3)
        rows.append(r)
        print(json.dumps(r))
    rows.append({"head_kernel_ratio_dk64_over_dk32": round(rows[1]["head_kernel_ms"] / rows[0]["head_kernel_ms"], 3)})
    print(json.dumps(rows[-1]))

    for f_maps in (32, 64):
        m, head = models(f_maps, dev)
        for n, chunk in ((80, 1), (8, 25)):
            st = head.open_stream(m, n)
            ids = list(range(n))
            fill = torch.rand(n * 100, 2048, device=dev) * 0.57
            st.step(fill, ids, [100] * n)   # 100 frames of history per stream
            x = feats[: n * chunk]
            for _ in range(20):
                st.step(x, ids, [chunk] * n)
            torch.cuda.synchronize()
            ms = timed(lambda: st.step(x, ids, [chunk] * n), a.steps, e0, e1)
            r = {"stream": True, "d_k": min(64, f_maps), "mstcn_f_maps": f_maps, "n_streams": n, "frames_per_step": chunk,
                 "device_ms_per_step": round(ms, 4), "launches_per_step": m.last_launch_count() + 2}
            rows.append(r)
            print(json.dumps(r))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump({"box": info, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
