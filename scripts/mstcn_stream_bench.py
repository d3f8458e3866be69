"""Online MS-TCN (+ Trans-SVNet head) step latency: n_streams in {1, 8, 80} x chunk in {1, 25}, with and without the head, timed from
seen = 100 and from seen = 5000, beside the offline forward over a stream's whole history (what the recompute alternative costs per tick).

    python scripts/mstcn_stream_bench.py [--steps 1000] [--out results/mstcn_stream_bench.json]

Per configuration: device ms per step (CUDA events around `steps` back-to-back warmed steps), host wall ms per step including a
device synchronise after every step, and kernels launched per step.  Needs a CUDA device; there is no CPU path."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import surgvid_b200  # noqa: E402,F401
from surgvid_b200 import synthetic as S  # noqa: E402
from surgvid_b200.mstcn import MultiStageModel_S  # noqa: E402
from surgvid_b200.trans_head import Transformer  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "not available"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mstcn_stream_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    m = MultiStageModel_S(2, 8, 32, 2048, 14, True)
    m.load_state_dict(S.synth_mstcn_state_dict(mode="phase"))
    m = m.to(dev).eval()
    head = Transformer(32, 2048, 14, 30).to(dev).eval()
    head.attach(m)
    feats = torch.rand(80 * 25, 2048, device=dev, generator=torch.Generator(dev).manual_seed(1)) * 0.57
    rows = []
    info = gpu_info()
    print(json.dumps(info))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for with_head in (False, True):
        for n in (1, 8, 80):
            for chunk in (1, 25):
                st = head.open_stream(m, n) if with_head else m.open_stream(n)
                ids, counts = list(range(n)), [chunk] * n
                x = feats[: n * chunk]
                fill = torch.rand(n * 100, 2048, device=dev) * 0.57
                for start in (100, 5000):
                    st.reset()
                    while int(st.seen[0]) < start:   # bring every stream to `start` frames of history
                        c = min(100, start - int(st.seen[0]))
                        st.step(fill[: n * c], ids, [c] * n)
                    for _ in range(20):
                        st.step(x, ids, counts)
                    torch.cuda.synchronize()
                    seen0 = int(st.seen[0])
                    e0.record()
                    for _ in range(a.steps):
                        st.step(x, ids, counts)
                    e1.record()
                    torch.cuda.synchronize()
                    dev_ms = e0.elapsed_time(e1) / a.steps
                    t0 = time.perf_counter()
                    k = max(100, a.steps // 5)
                    for _ in range(k):
                        st.step(x, ids, counts)
                        torch.cuda.synchronize()
                    host_ms = (time.perf_counter() - t0) * 1e3 / k
                    launches = m.last_launch_count() + (2 if with_head else 0)
                    r = {"head": with_head, "n_streams": n, "chunk": chunk, "seen_at_start": seen0, "device_ms_per_step": round(dev_ms, 4),
                         "host_ms_per_step_synced": round(host_ms, 4), "launches_per_step": launches}
                    rows.append(r)
                    print(json.dumps(r))
    # the recompute alternative: the offline forward over each stream's whole history (100 and 5000 frames), every tick
    for n in (1, 8, 80):
        for T in (100, 5000):
            hist = torch.rand(n * T, 2048, device=dev) * 0.57
            for with_head in (False, True):
                f = (lambda: head.forward_videos(m, hist, [T] * n)) if with_head else (lambda: m.forward_videos(hist, [T] * n))
                for _ in range(3):
                    f()
                torch.cuda.synchronize()
                reps = 50
                e0.record()
                for _ in range(reps):
                    f()
                e1.record()
                torch.cuda.synchronize()
                r = {"offline_recompute": True, "head": with_head, "n_streams": n, "history": T, "device_ms_per_call": round(e0.elapsed_time(e1) / reps, 4)}
                rows.append(r)
                print(json.dumps(r))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump({"box": info, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
