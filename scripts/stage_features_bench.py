"""Cost of forward_features on one GPU, in one process:
  * mit_b3_evp `forward_features(x, y)` (encoder-only plans, fp32 NCHW stage maps) vs `extract_features(x, y, None)` and
    `extract_features(x, y, flow)` (LFB features), at 224x224 with 256 frames and 480x854 with 2 frames: device events after warm-up,
    the three calls alternated over several rounds (median per call), and the kernels each plan launches;
  * the stage LayerNorm alone at the four stage shapes of mit_b3_evp at 224x224 with 256 frames: the token-major form the full forward
    runs there (bf16 result only: 4 B read + 2 B written per element) vs the channel-major form of forward_features (4 B read, 2 B bf16
    and 4 B fp32 written), with the achieved rate from those algorithmic bytes;
  * beside it, a device-to-device copy (torch's copy_, one cudaMemcpyAsync) of 2 GB, counted as bytes read + written;
  * the device name, power limit and max SM clock (nvidia-smi --query-gpu).
Writes stage_features_bench.json to --out.

    python scripts/stage_features_bench.py --out <directory>
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import surgvid_b200  # noqa: E402,F401
from surgvid_b200 import _native  # noqa: E402
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
    ap.add_argument("--out", required=True, help="directory for stage_features_bench.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage_features_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": device_info()}

    n = 1 << 29  # 2 GB, read + written
    src, dst = torch.empty(n, device=dev), torch.empty(n, device=dev)
    ms = timed(lambda: dst.copy_(src), 20, 3)
    res["d2d_copy"] = {"bytes": 4 * n, "ms": ms, "GBps_read_plus_write": 2 * 4 * n / ms / 1e6}
    del src, dst

    m = mit_b3_evp()
    m.load_state_dict(S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=0, mode="stress"), strict=True)
    m = m.to(dev).eval()
    res["model"] = []
    for B, H, W in ((256, 224, 224), (2, 480, 854)):
        x, seg, flow = (t.to(dev) for t in S.synth_frames(B, seed=1, H=H, W=W))
        calls = {"forward_features": lambda: m.forward_features(x, seg), "extract_features_noflow": lambda: m.extract_features(x, seg, None),
                 "extract_features_flow": lambda: m.extract_features(x, seg, flow)}
        times, launches = {k: [] for k in calls}, {}
        with torch.no_grad():
            for k, fn in calls.items():   # warm-up: plans, workspace, modules
                fn()
                launches[k] = m.last_launch_count()
            for _ in range(args.rounds):
                for k, fn in calls.items():
                    times[k].append(timed(fn, args.reps, 1))
        r = {"frames": B, "H": H, "W": W, "launches": launches, "ms_median": {k: statistics.median(v) for k, v in times.items()},
             "ms_rounds": times}
        shapes = m.stage_shapes(H, W)
        r["nchw_store_MB_per_frame"] = sum(4 * c * h * w for c, h, w in shapes) / 1e6
        r["forward_features_of_noflow"] = r["ms_median"]["forward_features"] / r["ms_median"]["extract_features_noflow"]
        res["model"].append(r)
        print(json.dumps(r), flush=True)
        del x, seg, flow
        torch.cuda.empty_cache()

    lib = _native.lib()
    st = torch.cuda.current_stream(dev).cuda_stream
    res["stage_norm"] = []
    B = 256
    for s, (C, h, w) in enumerate(m.stage_shapes(224, 224)):
        rows, tokens = B * h * w, h * w
        x = torch.randn(rows, C, device=dev)
        g, b = torch.randn(C, device=dev), torch.randn(C, device=dev)
        ob = torch.empty(rows, C, dtype=torch.bfloat16, device=dev)
        onchw = torch.empty(B, C, tokens, device=dev)
        p = [ctypes.c_void_p(t.data_ptr()) for t in (x, g, b, ob, onchw)]

        def plain():
            _native.check(lib.sv_op_layernorm(p[0], p[1], p[2], 1e-6, rows, C, None, p[3], ctypes.c_void_p(st)), "sv_op_layernorm")

        def nchw():
            _native.check(lib.sv_op_layernorm_nchw(p[0], p[1], p[2], 1e-6, rows, C, tokens, p[4], p[3], ctypes.c_void_p(st)),
                          "sv_op_layernorm_nchw")

        t = {"plain": [], "nchw": []}
        for _ in range(args.rounds):
            t["plain"].append(timed(plain, 50, 5))
            t["nchw"].append(timed(nchw, 50, 5))
        r = {"stage": s + 1, "rows": rows, "C": C, "tokens_per_frame": tokens}
        for k, nb in (("plain", 6.0), ("nchw", 10.0)):
            ms = statistics.median(t[k])
            r[k] = {"ms": ms, "alg_bytes": nb * rows * C, "GBps": nb * rows * C / ms / 1e6,
                    "of_copy_rate": nb * rows * C / ms / 1e6 / res["d2d_copy"]["GBps_read_plus_write"]}
        r["nchw_GBps_of_plain"] = r["nchw"]["GBps"] / r["plain"]["GBps"]
        res["stage_norm"].append(r)
        print(json.dumps(r), flush=True)
        del x, ob, onchw
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "stage_features_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["device"]))
    print(json.dumps(res["d2d_copy"]))


if __name__ == "__main__":
    main()
