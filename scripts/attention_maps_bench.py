"""Cost of attention-map capture on one GPU, in one process:
  * `forward` vs `attention_maps` (sv_evp_forward vs sv_evp_forward_attention) for mit_b3_evp at 224x224 with 64 and 256 frames and at
    480x854 with 2 frames (device events, warm-up first);
  * attention_probs_kernel alone through `ops.attention_probs` at the four stage shapes of mit_b3_evp at 224x224 (64 and 256 frames),
    with its achieved rate from algorithmic bytes (fp32 maps written + bf16 q and k read once);
  * beside it, a device-to-device copy (torch's copy_, one cudaMemcpyAsync) of 2 GB, counted as bytes read + written;
  * the device name, power limit and max SM clock (nvidia-smi --query-gpu).
Writes attention_maps_bench.json to --out.

    python scripts/attention_maps_bench.py --out <directory>
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import surgvid_b200  # noqa: E402,F401
from surgvid_b200 import ops  # noqa: E402
from surgvid_b200 import synthetic as S  # noqa: E402
from surgvid_b200.models.mix_transformer_evp import mit_b3_evp  # noqa: E402


def device_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return {"nvidia_smi": r.stdout.strip(), "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for attention_maps_bench.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_maps_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": device_info()}

    # copy rate: 2 GB, read + written
    n = 1 << 29
    src, dst = torch.empty(n, device=dev), torch.empty(n, device=dev)
    ms = timed(lambda: dst.copy_(src), 20, 3)
    res["d2d_copy"] = {"bytes": 4 * n, "ms": ms, "GBps_read_plus_write": 2 * 4 * n / ms / 1e6}
    del src, dst

    m = mit_b3_evp()
    m.load_state_dict(S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=0, mode="stress"), strict=True)
    m = m.to(dev).eval()
    res["model"] = []
    for B, H, W in ((64, 224, 224), (256, 224, 224), (2, 480, 854)):
        x, seg, flow = (t.to(dev) for t in S.synth_frames(B, seed=1, H=H, W=W))
        with torch.no_grad():
            t_fwd = timed(lambda: m(x, seg, flow, return_features=True), args.reps, args.warmup)
            t_cap = timed(lambda: m.attention_maps(x, seg, flow), args.reps, args.warmup)
        off, _ = m.attention_maps_layout(B, H, W)
        res["model"].append({"frames": B, "H": H, "W": W, "forward_ms": t_fwd, "attention_maps_ms": t_cap,
                             "capture_extra_us_per_frame": 1e3 * (t_cap - t_fwd) / B, "maps_MB_per_frame": 4 * off[-1] / B / 1e6})
        print(json.dumps(res["model"][-1]), flush=True)
        del x, seg, flow
        torch.cuda.empty_cache()

    res["probs_kernel"] = []
    C = [64, 128, 320, 512]
    for B in (64, 256):
        for s, (heads, Nq, Nkv) in enumerate(((1, 3136, 49), (2, 784, 49), (5, 196, 49), (8, 49, 49))):
            hd = C[s] // heads
            q = torch.randn(B * Nq, C[s], device=dev).to(torch.bfloat16)
            kv = torch.randn(B * Nkv, 2 * C[s], device=dev).to(torch.bfloat16)
            out = torch.empty((B, heads, Nq, Nkv), device=dev)
            ms = timed(lambda: ops.attention_probs(q, kv[:, :C[s]], B, heads, Nq, Nkv, hd, hd ** -0.5, out=out), 50, 5)
            nbytes = 4.0 * B * heads * Nq * Nkv + 2.0 * B * (Nq + Nkv) * C[s]
            r = {"frames": B, "stage": s + 1, "heads": heads, "Nq": Nq, "Nkv": Nkv, "hd": hd, "ms": ms, "alg_bytes": nbytes,
                 "GBps": nbytes / ms / 1e6}
            r["of_copy_rate"] = r["GBps"] / res["d2d_copy"]["GBps_read_plus_write"]
            res["probs_kernel"].append(r)
            print(json.dumps(r), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "attention_maps_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["device"]))
    print(json.dumps(res["d2d_copy"]))


if __name__ == "__main__":
    main()
